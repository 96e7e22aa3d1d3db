// tc_common.cuh -- inline-PTX wrappers shared by the tcgen05 kernels (mbarrier, TMA bulk copy,
// tcgen05.mma / ld / commit, UMMA shared-memory descriptors for the 128-byte swizzle).
#pragma once
#include <cuda_bf16.h>
#include "common.cuh"

namespace bmp {
namespace tc {

constexpr int NEPI = 256;
constexpr int NTHR = 320;
constexpr int PANEL_BYTES = 128 * 128;     // activation panel: 128 rows x 64 bf16, SW128 K-major
constexpr int ADJ_TILE_BYTES = 64 * 128;   // one (mol, e) adjacency tile: 64 rows x 64 bf16

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// A waiting thread is SUSPENDED (it wakes when the phase completes, or after this many nanoseconds to re-test) instead of
// re-issuing try_wait back to back: a spinning elected lane would otherwise take most of its scheduler's issue slots from
// the epilogue warps that share the scheduler.
constexpr uint32_t MBAR_SUSPEND_NS = 20000;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(MBAR_SUSPEND_NS) : "memory");
}
// wait with a sleep between polls (not latency-critical waits of an elected lane: the polling leaves the issue slots to the warps
// that share its scheduler)
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity, uint32_t ns) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "nanosleep.u32 %2;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(ns) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// smem -> global bulk store (async proxy; completion tracked by the issuing thread's bulk group)
__device__ __forceinline__ void tma_bulk_s2g(void *dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all committed bulk stores of this thread have finished READING shared memory
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }
// BF16-mode gate math: tanh.approx based (as in the encoder epilogues)
__device__ __forceinline__ float act_fast(int act, float x) {
    switch (act) {
        case BMP_ACT_TANH: return tanh_fast(x);
        case BMP_ACT_RELU: return x > 0.f ? x : 0.f;
        case BMP_ACT_SIGMOID: return sigmoid_fast(x);
        default: return x;
    }
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&t);
}

// smem matrix descriptors (SWIZZLE_128B, version 1).  K-major: SBO = 1024 B (8 rows x 128 B).
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// MN-major: LBO = stride between 64-element MN blocks (one panel = 16 KB), SBO = 8 k-rows = 1024 B.
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(PANEL_BYTES >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// Epilogue -> MMA hand-off, one mbarrier arrival per WARP: every thread orders its own shared-memory writes
// (generic proxy) and TMEM reads before the warp converges, then lane 0 arrives for all 32.
__device__ __forceinline__ void warp_arrive(uint32_t bar, int lane) {
    fence_proxy_async();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}

// instruction descriptor: D fp32, A/B bf16, M = 128, N = n
__host__ __device__ constexpr uint32_t idesc(int n, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}

// byte offset of element (row, k) inside a [rows][64] bf16 SW128 K-major block
__device__ __forceinline__ uint32_t sw128(uint32_t row, uint32_t k) {
    return row * 128u + ((((k >> 3) ^ (row & 7u)) << 4) | ((k & 7u) << 1));
}


// A operand read MN-major from adjacency tiles (two bond types = two 64-row blocks, 8 KB apart)
__device__ __forceinline__ uint64_t desc_mnmajor_adj(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(ADJ_TILE_BYTES >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__host__ __device__ constexpr uint32_t idesc2(int n, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}

// stage the adjacency of a tile (2 molecules x 4 bond types) as bf16 SW128 tiles [mol][e][i][j].  The source is the reference's
// fp32 array (mb,E,N,N) or, with `u8` = 1, the same array stored as bytes (exact for 0/1 bonds, a quarter of the traffic), or,
// with `u8` = 2, bit-packed rows (mb,E,N,ceil(N/8)): bit j&7 of byte j>>3 = adj[i][j] (numpy.packbits(..., bitorder='little');
// 2 KB per molecule at N = 64, 1/32 of the fp32 bytes).
// Loads are issued in batches of 8 vectors per thread so the DRAM latency is paid a few times per tile, not per element.
template <int NE>
__device__ __forceinline__ void stage_adjacency(uint8_t *s_adj, const void *__restrict__ adj_any, int u8, int tile, int mb, int N, int tid,
                                                const int32_t *__restrict__ midx = nullptr) {
    // midx: molecule b of this call is row midx[b] of a drug TABLE (atoms / adjacency read through the index, no gather copy)
    auto srcmol = [&](int mg) -> long { return midx ? (long)__ldg(midx + mg) : (long)mg; };
    if (u8 == 2) {
        const uint8_t *adj = reinterpret_cast<const uint8_t *>(adj_any);
        const int W = (N + 7) >> 3;
        constexpr int ROWS = 8 * 64, PER = (ROWS + NE - 1) / NE;      // items: (mol,e) x i ; one packed row each
        uint64_t bits[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int idx = u * NE + tid;
            const int i = idx & 63, me = idx >> 6;
            const int mg = tile * 2 + (me >> 2);
            bits[u] = 0;
            if (idx < ROWS && mg < mb && i < N) {
                const uint8_t *src = adj + ((srcmol(mg) * 4 + (me & 3)) * N + i) * W;
                if (W == 8) {
                    bits[u] = __ldg(reinterpret_cast<const unsigned long long *>(src));
                } else {
                    for (int x = 0; x < W; ++x) bits[u] |= (uint64_t)src[x] << (8 * x);
                }
                if (N < 64) bits[u] &= (1ull << N) - 1ull;
            }
        }
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int idx = u * NE + tid;
            if (idx >= ROWS) continue;
            const int i = idx & 63, me = idx >> 6;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint32_t b = (uint32_t)(bits[u] >> (8 * c)) & 0xFFu;
                uint32_t o[4];
#pragma unroll
                for (int x = 0; x < 4; ++x)
                    o[x] = ((b >> (2 * x)) & 1u ? 0x3F80u : 0u) | ((b >> (2 * x + 1)) & 1u ? 0x3F800000u : 0u);
                *reinterpret_cast<uint4 *>(s_adj + me * ADJ_TILE_BYTES + sw128(i, 8 * c)) = make_uint4(o[0], o[1], o[2], o[3]);
            }
        }
        return;
    }
    if (u8) {
        const uint8_t *adj = reinterpret_cast<const uint8_t *>(adj_any);
        constexpr int ITEMS = 8 * 64 * 4, PER = (ITEMS + NE - 1) / NE;     // items: (mol,e) x i x (j/16)
        uint4 v[PER];
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int idx = u * NE + tid;
            const int j16 = (idx & 3) * 16, i = (idx >> 2) & 63, me = idx >> 8;
            const int mg = tile * 2 + (me >> 2);
            v[u] = make_uint4(0, 0, 0, 0);
            if (idx < ITEMS && mg < mb && i < N && j16 < N) {
                const uint8_t *src = adj + ((srcmol(mg) * 4 + (me & 3)) * N + i) * N + j16;
                if ((N & 15) == 0) {
                    v[u] = __ldg(reinterpret_cast<const uint4 *>(src));
                } else {
                    uint32_t w[4] = {0, 0, 0, 0};
                    for (int x = 0; x < 16 && j16 + x < N; ++x) w[x >> 2] |= (uint32_t)src[x] << (8 * (x & 3));
                    v[u] = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < PER; ++u) {
            const int idx = u * NE + tid;
            if (idx >= ITEMS) continue;
            const int j16 = (idx & 3) * 16, i = (idx >> 2) & 63, me = idx >> 8;
            const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            uint32_t o[8];
#pragma unroll
            for (int x = 0; x < 8; ++x) {
                const uint32_t b0 = (w[x >> 1] >> (16 * (x & 1))) & 0xFFu, b1 = (w[x >> 1] >> (16 * (x & 1) + 8)) & 0xFFu;
                o[x] = pack_bf16((float)b0, (float)b1);
            }
            *reinterpret_cast<uint4 *>(s_adj + me * ADJ_TILE_BYTES + sw128(i, j16)) = make_uint4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<uint4 *>(s_adj + me * ADJ_TILE_BYTES + sw128(i, j16 + 8)) = make_uint4(o[4], o[5], o[6], o[7]);
        }
        return;
    }
    const float *adj = reinterpret_cast<const float *>(adj_any);
    constexpr int BATCH = 8;
    for (int base = 0; base < 8 * 64 * 16; base += NE * BATCH) {      // items: (mol,e) x i x (j/4)
        float4 v[BATCH];
#pragma unroll
        for (int u = 0; u < BATCH; ++u) {
            const int idx = base + u * NE + tid;
            const int j4 = (idx & 15) * 4, i = (idx >> 4) & 63, me = idx >> 10;
            const int mg = tile * 2 + (me >> 2);
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (mg < mb && i < N) {
                const float *src = adj + ((srcmol(mg) * 4 + (me & 3)) * N + i) * N + j4;
                if ((N & 3) == 0) {
                    if (j4 < N) v[u] = __ldg(reinterpret_cast<const float4 *>(src));
                } else {
                    if (j4 + 0 < N) v[u].x = src[0];
                    if (j4 + 1 < N) v[u].y = src[1];
                    if (j4 + 2 < N) v[u].z = src[2];
                    if (j4 + 3 < N) v[u].w = src[3];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < BATCH; ++u) {
            const int idx = base + u * NE + tid;
            const int j4 = (idx & 15) * 4, i = (idx >> 4) & 63, me = idx >> 10;
            uint2 pk = make_uint2(pack_bf16(v[u].x, v[u].y), pack_bf16(v[u].z, v[u].w));
            *reinterpret_cast<uint2 *>(s_adj + me * ADJ_TILE_BYTES + sw128(i, j4)) = pk;
        }
    }
}

// rescale_adj (models/relgcn.py:20-28) on the STAGED tiles: adj[mol][e][i][j] /= sum_{e',i'} adj[mol][e'][i'][j] (1 where that
// sum is 0).  `inv` is 128 floats of scratch shared memory; all NE epilogue threads call this (named barrier 1).
template <int NE>
__device__ __forceinline__ void rescale_staged_adjacency(uint8_t *s_adj, float *inv, int tid) {
    asm volatile("bar.sync 1, %0;" ::"n"(NE));           // staging complete
    if (tid < 128) {
        const int mol = tid >> 6, j = tid & 63;
        float s = 0.f;
        for (int e = 0; e < 4; ++e) {
            const uint8_t *t = s_adj + (mol * 4 + e) * ADJ_TILE_BYTES;
#pragma unroll 8
            for (int i = 0; i < 64; ++i) s += __bfloat162float(*reinterpret_cast<const __nv_bfloat16 *>(t + sw128(i, j)));
        }
        inv[tid] = s != 0.f ? 1.f / s : 1.f;
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NE));
    for (int idx = tid; idx < 8 * 64 * 16; idx += NE) {   // items: (mol,e) x i x (j/4)
        const int j4 = (idx & 15) * 4, i = (idx >> 4) & 63, me = idx >> 10;
        uint2 *p = reinterpret_cast<uint2 *>(s_adj + me * ADJ_TILE_BYTES + sw128(i, j4));
        const uint2 u = *p;
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&u.y));
        const float *w = inv + (me >> 2) * 64 + j4;
        *p = make_uint2(pack_bf16(a.x * w[0], a.y * w[1]), pack_bf16(b.x * w[2], b.y * w[3]));
    }
    asm volatile("bar.sync 1, %0;" ::"n"(NE));           // inv may be reused, tiles are final
}

// pull the next tile's adjacency (2 molecules x 4 bond types x N x N fp32, contiguous) towards L2
template <int NE>
__device__ __forceinline__ void prefetch_adjacency_l2(const void *__restrict__ adj, int u8, int tile, int mb, int N, int tid,
                                                      const int32_t *__restrict__ midx = nullptr) {
    const long first = (long)tile * 2, nmol = first + 2 <= mb ? 2 : (first < mb ? 1 : 0);
    const long per_mol = u8 == 2 ? 4L * N * ((N + 7) >> 3) : 4L * N * N * (u8 ? 1 : 4);
    if (midx) {      // table rows: the two molecules of the tile are not adjacent in memory
        for (long m = 0; m < nmol; ++m) {
            const char *base = reinterpret_cast<const char *>(adj) + (long)__ldg(midx + first + m) * per_mol;
            for (long off = (long)tid * 128; off < per_mol; off += (long)NE * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
        }
        return;
    }
    const char *base = reinterpret_cast<const char *>(adj) + first * per_mol;
    const long bytes = nmol * per_mol;
    for (long off = (long)tid * 128; off < bytes; off += (long)NE * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + off));
}

// ---- coalesced global I/O for the lane == row register layout -----------------------------------
// An epilogue warp owns 32 tile rows; each lane holds W consecutive fp32 columns of ITS row (the
// tcgen05.ld 32x32b layout).  Going to global memory lane-per-row touches 32 different lines per
// instruction; these helpers transpose through a warp-private, XOR-swizzled staging block so that W/4
// lanes cover one row segment and every instruction moves full sectors of 32/(W/4) rows.
// rowptr(r) -> pointer to the first of the W columns of warp row r (0..31), or nullptr (row not live).
template <int CH>
__device__ __forceinline__ int swz_key(int r) { return (r * CH / 8) & (CH - 1); }
template <int W, class RowPtr>
__device__ __forceinline__ void warp_store_rows(float *stg, const float *v, int lane, RowPtr rowptr) {
    constexpr int CH = W / 4, RPI = 32 / CH;         // 16-byte chunks per row, rows per instruction
#pragma unroll
    for (int j = 0; j < CH; ++j)
        *reinterpret_cast<float4 *>(stg + lane * W + ((j ^ swz_key<CH>(lane)) << 2)) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    __syncwarp();
    const int ch = lane & (CH - 1);
#pragma unroll
    for (int it = 0; it < 32 / RPI; ++it) {
        const int r = it * RPI + lane / CH;
        const float4 x = *reinterpret_cast<const float4 *>(stg + r * W + ((ch ^ swz_key<CH>(r)) << 2));
        float *dst = rowptr(r);
        if (dst) *reinterpret_cast<float4 *>(dst + ch * 4) = x;
    }
    __syncwarp();
}
template <int W, class RowPtr>
__device__ __forceinline__ void warp_load_rows(float *stg, float *v, int lane, RowPtr rowptr) {
    constexpr int CH = W / 4, RPI = 32 / CH;
    const int ch = lane & (CH - 1);
#pragma unroll
    for (int it = 0; it < 32 / RPI; ++it) {
        const int r = it * RPI + lane / CH;
        const float *src = rowptr(r);
        const float4 x = src ? *reinterpret_cast<const float4 *>(src + ch * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4 *>(stg + r * W + ((ch ^ swz_key<CH>(r)) << 2)) = x;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < CH; ++j) {
        const float4 x = *reinterpret_cast<const float4 *>(stg + lane * W + ((j ^ swz_key<CH>(lane)) << 2));
        v[4 * j] = x.x; v[4 * j + 1] = x.y; v[4 * j + 2] = x.z; v[4 * j + 3] = x.w;
    }
    __syncwarp();
}

// Split form of warp_load_rows: issue the coalesced global loads of several arrays first (so their
// latencies overlap), then transpose each through the staging block.
template <int W, class RowPtr>
__device__ __forceinline__ void warp_ldg_rows(float4 (&x)[W / 4], int lane, RowPtr rowptr) {
    constexpr int CH = W / 4, RPI = 32 / CH;
    const int ch = lane & (CH - 1);
#pragma unroll
    for (int it = 0; it < CH; ++it) {
        const int r = it * RPI + lane / CH;
        const float *src = rowptr(r);
        x[it] = src ? __ldg(reinterpret_cast<const float4 *>(src + ch * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int W>
__device__ __forceinline__ void warp_transpose_in(float *stg, const float4 (&x)[W / 4], float *v, int lane) {
    constexpr int CH = W / 4, RPI = 32 / CH;
    const int ch = lane & (CH - 1);
#pragma unroll
    for (int it = 0; it < CH; ++it) {
        const int r = it * RPI + lane / CH;
        *reinterpret_cast<float4 *>(stg + r * W + ((ch ^ swz_key<CH>(r)) << 2)) = x[it];
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < CH; ++j) {
        const float4 t = *reinterpret_cast<const float4 *>(stg + lane * W + ((j ^ swz_key<CH>(lane)) << 2));
        v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
    }
    __syncwarp();
}

// ---- bf16 panel stash (stash v2) -----------------------------------------------------------------
// Per (step t, tile): forward dumps the operand panels h_t, m_t, r*h_t (KP panels each) verbatim and the
// gate values z | hbar | r | state as bf16 in the epilogue threads' native order ([16-byte chunk][thread]);
// backward dumps the delta panels (3KP) and the P panels (4KP).  A 64-row half of a panel is an MN-major
// UMMA operand block for the parameter-gradient contraction (wgrad_tc2.cu).
struct Stash2 {
    uint8_t *Xp, *Mp, *RSp, *Zn, *Dp, *Pp;
    long n_tiles;
    int KP, T;
    __host__ __device__ static size_t bytes(long n_tiles, int H, int T) {
        const size_t KP = H / 64, per = (size_t)n_tiles * T;
        return per * (3 * KP + 3 * KP + 4 * KP) * PANEL_BYTES + per * 4 * ((size_t)128 * H * 2) + 4096;
    }
    __host__ __device__ void carve(void *base, long nt, int H, int T_) {
        n_tiles = nt; KP = H / 64; T = T_;
        const size_t per = (size_t)nt * T_;
        uint8_t *p = (uint8_t *)(((uintptr_t)base + 1023) & ~(uintptr_t)1023);
        Xp = p; p += per * KP * PANEL_BYTES;
        Mp = p; p += per * KP * PANEL_BYTES;
        RSp = p; p += per * KP * PANEL_BYTES;
        Dp = p; p += per * 3 * KP * PANEL_BYTES;
        Pp = p; p += per * 4 * KP * PANEL_BYTES;
        Zn = p;
    }
    // native gate block of (t, tile, array a in 0..3 = z, hbar, r, state): 128 rows x H bf16 = [16-byte chunk][epilogue thread]
    __host__ __device__ uint8_t *zn(int t, long tile, int a, int H) const {
        return Zn + (((size_t)t * n_tiles + tile) * 4 + a) * ((size_t)128 * H * 2);
    }

};

}  // namespace tc

// ---- grouped parameter-gradient contraction over the panel stash (wgrad_tc2.cu) -------------------
namespace w2 {
struct Args {
    const uint8_t *A;                  // panel array of the A operand: [t][tile][a_ppt panels][16 KB]
    int a_ppt;
    int a_panel[2][2];                 // per M tile: the two 64-column blocks of A (= 64-row blocks of C); -1: absent
    int n_mt;                          // M tiles (1 or 2; two only with nb <= 3)
    const uint8_t *B[6];               // per B block: panel array, panels per tile, panel index
    int b_ppt[6], b_panel[6];
    int nb;
    float *C[2][2][6];                 // target of (M tile, A block, B block): element (row 0, col 0), row-major; NULL: skip
    int ldc[6];
    float *C2[2][2][6];                // optional second target of the same sum
    int ldc2[6];
    float *bias[2][2], *bias2[2][2];   // column sums of the A block (stride bias_stride) or NULL
    int bias_stride;
    int t0, t1, n_tiles;               // steps [t0, t1], tiles per step
    long chunks_per_cta;               // unused (kept for layout stability)
};
// Several contractions over the SAME (step, tile) range in ONE launch: the CTAs are split into classes (one Args each) in
// proportion to the bytes a class reads per unit, and every class walks the units in the same strided order, so all classes
// are on the same few units at the same time -- a panel that several classes need (h, m) comes from HBM once and from L2 for
// the others.
constexpr int MAX_CLASSES = 6;
struct Multi {
    Args cls[MAX_CLASSES];
    int n;
    int cta0[MAX_CLASSES + 1];         // class c owns CTAs [cta0[c], cta0[c+1])
    float *part[MAX_CLASSES];          // deterministic mode: class c's [CTAs][plen] partials (det.cuh), else nullptr
    long plen[MAX_CLASSES];
};
}  // namespace w2
}  // namespace bmp
