// relgcn_tc.cu -- RelGCN encoder (embed -> L x act(RelGCNUpdate)) on tcgen05 (BMP_MODE_BF16), forward and backward.
//
// Replaces models/relgcn.py:61-73 and models/update/relgcn_update.py:24-44 like relgcn.cu, with the machinery of the
// GGNN encoder (ggnn_tc.cu / ggnn_tc_bwd.cu): persistent CTA per SM, a tile = two padded molecules = 128 rows,
// adjacency (bf16) and the layer input resident in shared memory, accumulators in TMEM, weights streamed as packed
// bf16 tiles.  A layer is re-associated exactly like the GGNN message:
//   out = h W_s^T + b_s + sum_e A_e (h W_e^T + b_e) = [h | A_0 h | .. | A_3 h] [W_s | W_0 | .. | W_3]^T + b_s + sum_e deg_e b_e
//   MMA-1  AH[(e,i), c] = sum_j A_e[i,j] h[j,c]            per (molecule, bond-type pair), B = the h panels read MN-major
//   MMA-2  out = h W_s^T (+)= AHcat Wcat^T                 K = (1 + 4) C, one accumulator
//   epilogue: bias, activation, next layer's bf16 operand panels (and the bf16 panel stash for the backward)
// Backward per layer (delta = dL/dout * act'(out)):
//   MMA-s  dh  = delta W_s ;  MMA-P  P_e = A_e^T delta (both operands MN-major) ;  MMA-dh  dh += Pcat Wcat
// Parameter gradients are grouped contractions over the dumped panels (wgrad_tc2.cu): dW_s = delta^T h, dW_e = P_e^T h,
// db_s = colsum(delta), db_e = colsum(P_e).  All layers must share one channel count C in {64, 128}; `rescale_adj` is
// applied to the staged bf16 tiles (forward and backward alike); bmp_rescale_adj is the same normalisation as a stand-alone op.
#include "tc_common.cuh"

namespace bmp {
namespace rgt {
using namespace tc;

template <int H>
struct Cfg {
    static constexpr int KP = H / 64;
    static constexpr int EPW = H / 8;                       // epilogue warps: 4 TMEM lane quarters x (H / 32) column groups
    static constexpr int NE = 32 * EPW, NT = NE + 64;
    static constexpr int TILE_BYTES = H * 128;              // weight tile: H rows (n) x 64 bf16 (k)
    static constexpr int STAGES = 4;
    static constexpr int TILES = 5 * KP;                    // per layer, forward and backward alike
    static constexpr int TMEM_COLS = 4 * H;
    // forward
    static constexpr int OFF_H = 0;
    static constexpr int OFF_ADJ = OFF_H + KP * PANEL_BYTES;
    static constexpr int OFF_AH = OFF_ADJ + 8 * ADJ_TILE_BYTES;          // one K half of AHcat; store staging at the tile ends
    static constexpr int OFF_W = OFF_AH + 2 * KP * PANEL_BYTES;
    static constexpr int OFF_BAR = OFF_W + STAGES * TILE_BYTES;
    static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
    // backward: [Pcat half: 2KP panels][delta: KP panels] | adjacency | weight ring
    static constexpr int B_OFF_D = 0;
    static constexpr int B_OFF_ADJ = B_OFF_D + 3 * KP * PANEL_BYTES;
    static constexpr int B_OFF_W = B_OFF_ADJ + 8 * ADJ_TILE_BYTES;
    static constexpr int B_OFF_BAR = B_OFF_W + STAGES * TILE_BYTES;
    static constexpr int B_SMEM_BYTES = B_OFF_BAR + 256 + 1024;
};

struct Args {
    int mb, N, L, n_types, act, scale_adj;
    const int32_t *atoms;
    const float *embed_W, *h_in;
    const void *adj;                         // fp32 (mb,E,N,N), or bytes when adj_u8
    int adj_u8;
    const uint8_t *img[BMP_MAX_STEPS];       // forward: [self KP][msg 4KP] tiles ; backward: [self^T KP][dh 4KP]
    const float *self_b[BMP_MAX_STEPS], *edge_b[BMP_MAX_STEPS];
    float *h_out;                            // forward: (mb, N, H)
    const float *d_h_out;                    // backward in
    float *d_h0;                             // backward out (mb, N, H)
    Stash2 st;                               // forward writes (use2), backward reads + writes
    int use2;
};

__device__ __forceinline__ float act_grad_from_out(int act, float y) {
    switch (act) {
        case BMP_ACT_TANH: return 1.f - y * y;
        case BMP_ACT_RELU: return y > 0.f ? 1.f : 0.f;
        case BMP_ACT_SIGMOID: return y * (1.f - y);
        default: return 1.f;
    }
}

// native block holding act(out) of layer l (input of layer l+1): slot 3 of step l+1, or slot 0 of the last step
__device__ __forceinline__ uint8_t *out_block(const Stash2 &st, int l, int L, long tile, int H) {
    return l + 1 < L ? st.zn(l + 1, tile, 3, H) : st.zn(L - 1, tile, 0, H);
}

// ------------------------------------------------------------------------------------------------ forward
template <int H, bool V2>
__global__ void __launch_bounds__(Cfg<H>::NT, 1) relgcn_tc_kernel(const Args a) {
    using C = Cfg<H>;
    constexpr int KP = C::KP, EPW = C::EPW, NE = C::NE, NC = 32;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_h = sbase + C::OFF_H, s_adj = sbase + C::OFF_ADJ, s_ah = sbase + C::OFF_AH, s_w = sbase + C::OFF_W;
    const uint32_t s_bar = sbase + C::OFF_BAR;
    auto BAR = [&](int i) { return s_bar + 8u * i; };
    constexpr int B_FULL = 0, B_EMPTY = 4, B_HREADY = 8, B_D1 = 9, B_AHREADY = 13, B_AHFREE = 15, B_M = 16, NBAR = 17;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::OFF_BAR + 8 * NBAR + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (a.mb + 1) / 2;

    if (tid == 0) {
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(BAR(B_FULL + s), 1); mbar_init(BAR(B_EMPTY + s), 1); }
        mbar_init(BAR(B_HREADY), EPW);
        for (int i = 0; i < 4; ++i) mbar_init(BAR(B_D1 + i), 1);
        mbar_init(BAR(B_AHREADY), EPW);
        mbar_init(BAR(B_AHREADY + 1), EPW);
        mbar_init(BAR(B_AHFREE), 1);
        mbar_init(BAR(B_M), 1);
        fence_mbar_init();
    }
    if (warp == EPW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"(C::TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == EPW) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int l = 0; l < a.L; ++l)
                    for (int s = 0; s < C::TILES; ++s) {
                        mbar_wait(BAR(B_EMPTY + stage), phase ^ 1);
                        mbar_expect_tx(BAR(B_FULL + stage), C::TILE_BYTES);
                        tma_bulk_g2s(s_w + stage * C::TILE_BYTES, a.img[l] + (size_t)s * C::TILE_BYTES, C::TILE_BYTES, BAR(B_FULL + stage));
                        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    }
        }
    } else if (warp == EPW + 1) {
        if (lane == 0) {
            constexpr uint32_t ID_KK = idesc(H, 0), ID_KMN = idesc(H, 1);
            uint32_t stage = 0, phase = 0, it = 0;
            auto mma_wtile = [&](uint32_t a_addr, bool first) {
                mbar_wait(BAR(B_FULL + stage), phase);
                tc_fence_after();
                const uint32_t b_addr = s_w + stage * C::TILE_BYTES;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem, desc_kmajor(a_addr + k * 32), desc_kmajor(b_addr + k * 32), ID_KK, (first && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_EMPTY + stage));
                if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            };
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int l = 0; l < a.L; ++l, ++it) {
                    const uint32_t par = it & 1;
                    mbar_wait(BAR(B_HREADY), par);
                    tc_fence_after();
                    if (V2) {       // dump the layer input h_l (operand panels) for the parameter-gradient contractions
                        tma_bulk_s2g(a.st.Xp + ((size_t)l * n_tiles + tile) * KP * PANEL_BYTES, s_h, KP * PANEL_BYTES);
                        bulk_commit();
                    }
                    for (int p = 0; p < 2; ++p)
                        for (int mol = 0; mol < 2; ++mol) {
                            const uint32_t a_addr = s_adj + (mol * 4 + 2 * p) * ADJ_TILE_BYTES;
                            const uint32_t b_addr = s_h + mol * 64 * 128;
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc_mma(tmem + (2 * p + mol) * H, desc_kmajor(a_addr + k * 32), desc_mnmajor(b_addr + k * 16 * 128), ID_KMN, k ? 1u : 0u);
                            tc_commit(BAR(B_D1 + 2 * p + mol));
                        }
                    mbar_wait(BAR(B_AHREADY), par);        // D1 regions 0, 1 consumed: region 0 becomes the layer's accumulator
                    tc_fence_after();
                    for (int kp = 0; kp < KP; ++kp) mma_wtile(s_h + kp * PANEL_BYTES, kp == 0);          // self term
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_ah + kp * PANEL_BYTES, false);       // bond types 0, 1
                    tc_commit(BAR(B_AHFREE));
                    mbar_wait(BAR(B_AHREADY + 1), par);
                    tc_fence_after();
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_ah + kp * PANEL_BYTES, false);       // bond types 2, 3
                    if (V2) bulk_wait_read();              // the h_l dump has left shared memory: the epilogue may rewrite the panels
                    tc_commit(BAR(B_M));
                }
        }
    } else {
        const int q = warp & 3, hf = warp >> 2;
        const int row = 32 * q + lane, colbase = hf * NC;
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
        const int molslot = row >> 6, atom = row & 63;
        float *stg = reinterpret_cast<float *>(smem + C::OFF_AH + warp * 2048);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int molg = tile * 2 + molslot;
            const bool live = molg < a.mb && atom < a.N;
            const long grow = (long)molg * a.N + atom;
            float hreg[NC];
            {
                const float *src = nullptr;
                if (live) {
                    if (a.atoms) {
                        int id = __ldg(a.atoms + grow);
                        id = id < 0 ? 0 : (id >= a.n_types ? a.n_types - 1 : id);
                        src = a.embed_W + (long)id * H + colbase;
                    } else {
                        src = a.h_in + grow * H + colbase;
                    }
                }
#pragma unroll
                for (int c = 0; c < NC; c += 4) {
                    float4 v = src ? __ldg(reinterpret_cast<const float4 *>(src + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    hreg[c] = v.x; hreg[c + 1] = v.y; hreg[c + 2] = v.z; hreg[c + 3] = v.w;
                }
            }
            stage_adjacency<NE>(smem + C::OFF_ADJ, a.adj, a.adj_u8, tile, a.mb, a.N, tid);
            if (a.scale_adj) rescale_staged_adjacency<NE>(smem + C::OFF_ADJ, reinterpret_cast<float *>(smem + C::OFF_AH), tid);
            auto store_h_operand = [&]() {
#pragma unroll
                for (int g = 0; g < NC / 8; ++g) {
                    const int kk = colbase + 8 * g;
                    uint4 pk = make_uint4(pack_bf16(hreg[8 * g], hreg[8 * g + 1]), pack_bf16(hreg[8 * g + 2], hreg[8 * g + 3]),
                                          pack_bf16(hreg[8 * g + 4], hreg[8 * g + 5]), pack_bf16(hreg[8 * g + 6], hreg[8 * g + 7]));
                    *reinterpret_cast<uint4 *>(smem + C::OFF_H + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pk;
                }
            };
            store_h_operand();
            asm volatile("bar.sync 1, %0;" ::"n"(NE));
            // degrees (row sums of the staged tiles): one bond type per column group, exchanged through the idle AH buffer
            float deg[4];
            {
                float *dsh = reinterpret_cast<float *>(smem + C::OFF_AH);
                for (int e = hf; e < 4; e += EPW / 4) {
                    float s0 = 0.f, s1 = 0.f;
                    const uint8_t *rowp = smem + C::OFF_ADJ + (molslot * 4 + e) * ADJ_TILE_BYTES + atom * 128;
#pragma unroll
                    for (int ch = 0; ch < 8; ++ch) {
                        uint4 u = *reinterpret_cast<const uint4 *>(rowp + ((ch ^ (atom & 7)) << 4));
                        const __nv_bfloat162 *b2 = reinterpret_cast<const __nv_bfloat162 *>(&u);
#pragma unroll
                        for (int x = 0; x < 4; ++x) { float2 f = __bfloat1622float2(b2[x]); s0 += f.x; s1 += f.y; }
                    }
                    dsh[e * 128 + row] = s0 + s1;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(NE));
#pragma unroll
                for (int e = 0; e < 4; ++e) deg[e] = dsh[e * 128 + row];
                asm volatile("bar.sync 1, %0;" ::"n"(NE));
            }
            warp_arrive(BAR(B_HREADY), lane);

            for (int l = 0; l < a.L; ++l, ++it) {
                const uint32_t par = it & 1;
                uint32_t v[32];
                // ---- E1: AH accumulators -> bf16 A-operand panels (two K halves)
                for (int p = 0; p < 2; ++p) {
                    if (p == 1) mbar_wait(BAR(B_AHFREE), par);
                    for (int mol = 0; mol < 2; ++mol) {
                        mbar_wait(BAR(B_D1 + 2 * p + mol), par);
                        tc_fence_after();
                        const int orow = mol * 64 + atom, kbase = molslot * H + colbase;
                        tc_ld32(t_lane + (2 * p + mol) * H + colbase, v);
                        tc_wait_ld();
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const int kk = kbase + 8 * g;
                            uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
                            *reinterpret_cast<uint4 *>(smem + C::OFF_AH + (kk >> 6) * PANEL_BYTES + sw128(orow, kk & 63)) = pk;
                        }
                    }
                    warp_arrive(BAR(B_AHREADY + p), lane);
                }
                // ---- E2: bias, activation -> the next layer's input
                mbar_wait(BAR(B_M), par);
                tc_fence_after();
                tc_ld32(t_lane + colbase, v);
                tc_wait_ld();
                {
                    const float *bs = a.self_b[l], *be = a.edge_b[l];
#pragma unroll
                    for (int x = 0; x < 32; x += 4) {
                        const float4 s4 = bs ? __ldg(reinterpret_cast<const float4 *>(bs + colbase + x)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        const float sb[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
                        for (int y = 0; y < 4; ++y) {
                            float val = __uint_as_float(v[x + y]) + sb[y];
                            if (be) {
                                const float4 b4 = __ldg(reinterpret_cast<const float4 *>(be) + colbase + x + y);
                                val += deg[0] * b4.x + deg[1] * b4.y + deg[2] * b4.z + deg[3] * b4.w;
                            }
                            hreg[x + y] = act_fast(a.act, val);
                        }
                    }
                }
                if (V2) {       // act(out) in the thread-native bf16 order: the backward needs it for act'
                    uint8_t *base = out_block(a.st, l, a.L, tile, H);
#pragma unroll
                    for (int g = 0; g < NC / 8; ++g) {
                        uint4 pk = make_uint4(pack_bf16(hreg[8 * g], hreg[8 * g + 1]), pack_bf16(hreg[8 * g + 2], hreg[8 * g + 3]),
                                              pack_bf16(hreg[8 * g + 4], hreg[8 * g + 5]), pack_bf16(hreg[8 * g + 6], hreg[8 * g + 7]));
                        *reinterpret_cast<uint4 *>(base + ((size_t)g * NE + tid) * 16) = pk;
                    }
                }
                if (l + 1 < a.L) {
                    store_h_operand();
                    warp_arrive(BAR(B_HREADY), lane);
                } else {
                    if (a.h_out) {
#pragma unroll
                        for (int h2 = 0; h2 < 2; ++h2)
                            warp_store_rows<16>(stg, hreg + 16 * h2, lane, [&](int r) -> float * {
                                const int tr = 32 * q + r, mg = tile * 2 + (tr >> 6), at = tr & 63;
                                return (mg < a.mb && at < a.N) ? a.h_out + ((long)mg * a.N + at) * H + colbase + 16 * h2 : nullptr;
                            });
                    }
                    tc_fence_before();
                    asm volatile("bar.sync 1, %0;" ::"n"(NE));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPW + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(C::TMEM_COLS));
    }
}

// ------------------------------------------------------------------------------------------------ backward
template <int H>
__global__ void __launch_bounds__(Cfg<H>::NT, 1) relgcn_tc_bwd_kernel(const Args a) {
    using C = Cfg<H>;
    constexpr int KP = C::KP, EPW = C::EPW, NE = C::NE, NC = 32;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_d = sbase + C::B_OFF_D, s_adj = sbase + C::B_OFF_ADJ, s_w = sbase + C::B_OFF_W, s_bar = sbase + C::B_OFF_BAR;
    const uint32_t s_dm = s_d + 2 * KP * PANEL_BYTES;        // delta panels: A of MMA-s (K-major), B of MMA-P (MN-major)
    auto BAR = [&](int i) { return s_bar + 8u * i; };
    constexpr int B_FULL = 0, B_EMPTY = 4, B_DRDY = 8, B_P = 9, B_PRDY = 13, B_PFREE = 15, B_DH = 16, NBAR = 17;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::B_OFF_BAR + 8 * NBAR + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (a.mb + 1) / 2;
    constexpr uint32_t COL_DHX = H;

    if (tid == 0) {
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(BAR(B_FULL + s), 1); mbar_init(BAR(B_EMPTY + s), 1); }
        mbar_init(BAR(B_DRDY), EPW);
        for (int i = 0; i < 4; ++i) mbar_init(BAR(B_P + i), 1);
        mbar_init(BAR(B_PRDY), EPW);
        mbar_init(BAR(B_PRDY + 1), EPW);
        mbar_init(BAR(B_PFREE), 1);
        mbar_init(BAR(B_DH), 1);
        fence_mbar_init();
    }
    if (warp == EPW + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"(C::TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == EPW) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int l = a.L - 1; l >= 0; --l)
                    for (int s = 0; s < C::TILES; ++s) {
                        mbar_wait(BAR(B_EMPTY + stage), phase ^ 1);
                        mbar_expect_tx(BAR(B_FULL + stage), C::TILE_BYTES);
                        tma_bulk_g2s(s_w + stage * C::TILE_BYTES, a.img[l] + (size_t)s * C::TILE_BYTES, C::TILE_BYTES, BAR(B_FULL + stage));
                        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    }
        }
    } else if (warp == EPW + 1) {
        if (lane == 0) {
            constexpr uint32_t ID_KK = idesc2(H, 0, 0), ID_MNMN = idesc2(H, 1, 1);
            uint32_t stage = 0, phase = 0, it = 0;
            auto mma_wtile = [&](uint32_t a_addr, bool first) {
                mbar_wait(BAR(B_FULL + stage), phase);
                tc_fence_after();
                const uint32_t b_addr = s_w + stage * C::TILE_BYTES;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem + COL_DHX, desc_kmajor(a_addr + k * 32), desc_kmajor(b_addr + k * 32), ID_KK, (first && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_EMPTY + stage));
                if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            };
            auto mma_p = [&](int mol, int p, uint32_t dcol, int bar) {
                const uint32_t a_addr = s_adj + (mol * 4 + 2 * p) * ADJ_TILE_BYTES;
                const uint32_t b_addr = s_dm + mol * 64 * 128;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem + dcol, desc_mnmajor_adj(a_addr + k * 16 * 128), desc_mnmajor(b_addr + k * 16 * 128), ID_MNMN, k ? 1u : 0u);
                tc_commit(BAR(bar));
            };
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int l = a.L - 1; l >= 0; --l, ++it) {
                    const uint32_t par = it & 1;
                    mbar_wait(BAR(B_DRDY), par);
                    tc_fence_after();
                    uint8_t *Dt = a.st.Dp + ((size_t)l * n_tiles + tile) * 3 * KP * PANEL_BYTES;
                    uint8_t *Pt = a.st.Pp + ((size_t)l * n_tiles + tile) * 4 * KP * PANEL_BYTES;
                    tma_bulk_s2g(Dt + (size_t)2 * KP * PANEL_BYTES, s_dm, KP * PANEL_BYTES);      // delta panels (slot of delta_h)
                    bulk_commit();
                    for (int kp = 0; kp < KP; ++kp) mma_wtile(s_dm + kp * PANEL_BYTES, kp == 0);   // dh = delta W_s
                    mma_p(0, 0, 0 * H, B_P + 0);
                    mma_p(1, 0, 2 * H, B_P + 1);
                    mma_p(0, 1, 3 * H, B_P + 2);
                    mbar_wait(BAR(B_PRDY + 0), par);
                    tc_fence_after();
                    tma_bulk_s2g(Pt, s_d, 2 * KP * PANEL_BYTES);
                    bulk_commit();
                    mma_p(1, 1, 0 * H, B_P + 3);
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_d + kp * PANEL_BYTES, false);
                    bulk_wait_read();
                    tc_commit(BAR(B_PFREE));
                    mbar_wait(BAR(B_PRDY + 1), par);
                    tc_fence_after();
                    tma_bulk_s2g(Pt + (size_t)2 * KP * PANEL_BYTES, s_d, 2 * KP * PANEL_BYTES);
                    bulk_commit();
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_d + kp * PANEL_BYTES, false);
                    bulk_wait_read();          // delta and P dumps are out: the next layer may rewrite the panels
                    tc_commit(BAR(B_DH));
                }
        }
    } else {
        const int q = warp & 3, hf = warp >> 2;
        const int row = 32 * q + lane, colbase = hf * NC;
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
        const int molslot = row >> 6, atom = row & 63;
        float acc[NC];
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int molg = tile * 2 + molslot;
            const bool live = molg < a.mb && atom < a.N;
            const long grow = (long)molg * a.N + atom;
            stage_adjacency<NE>(smem + C::B_OFF_ADJ, a.adj, a.adj_u8, tile, a.mb, a.N, tid);
            if (a.scale_adj) rescale_staged_adjacency<NE>(smem + C::B_OFF_ADJ, reinterpret_cast<float *>(smem + C::B_OFF_D), tid);
            {
                const float *src = live ? a.d_h_out + grow * H + colbase : nullptr;
#pragma unroll
                for (int c = 0; c < NC; c += 4) {
                    float4 v = src ? __ldg(reinterpret_cast<const float4 *>(src + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    acc[c] = v.x; acc[c + 1] = v.y; acc[c + 2] = v.z; acc[c + 3] = v.w;
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(NE));      // adjacency staged (MMA-P reads it after the first hand-off)
            for (int l = a.L - 1; l >= 0; --l, ++it) {
                const uint32_t par = it & 1;
                uint32_t v[32];
                // ---- delta = dL/dout * act'(out) -> bf16 operand panels
                {
                    const uint8_t *bo = out_block(a.st, l, a.L, tile, H);
                    uint4 op[NC / 8];
#pragma unroll
                    for (int g = 0; g < NC / 8; ++g) op[g] = __ldg(reinterpret_cast<const uint4 *>(bo + ((size_t)g * NE + tid) * 16));
#pragma unroll
                    for (int g = 0; g < NC / 8; ++g) {
                        const __nv_bfloat162 *o2 = reinterpret_cast<const __nv_bfloat162 *>(&op[g]);
                        float d[8];
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            const float2 oo = __bfloat1622float2(o2[x]);
                            d[2 * x] = live ? acc[8 * g + 2 * x] * act_grad_from_out(a.act, oo.x) : 0.f;
                            d[2 * x + 1] = live ? acc[8 * g + 2 * x + 1] * act_grad_from_out(a.act, oo.y) : 0.f;
                        }
                        const int kk = colbase + 8 * g;
                        *reinterpret_cast<uint4 *>(smem + C::B_OFF_D + (2 * KP + (kk >> 6)) * PANEL_BYTES + sw128(row, kk & 63)) =
                            make_uint4(pack_bf16(d[0], d[1]), pack_bf16(d[2], d[3]), pack_bf16(d[4], d[5]), pack_bf16(d[6], d[7]));
                    }
                }
                warp_arrive(BAR(B_DRDY), lane);
                // ---- P accumulators -> bf16 A-operand panels (two K halves)
                for (int p = 0; p < 2; ++p) {
                    if (p == 1) mbar_wait(BAR(B_PFREE), par);
                    for (int mol = 0; mol < 2; ++mol) {
                        const int pi = 2 * p + mol;
                        const uint32_t pcol = (pi == 0 || pi == 3) ? 0u : (pi == 1 ? 2u * H : 3u * H);
                        mbar_wait(BAR(B_P + pi), par);
                        tc_fence_after();
                        const int orow = mol * 64 + atom, kbase = molslot * H + colbase;
                        tc_ld32(t_lane + pcol + colbase, v);
                        tc_wait_ld();
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const int kk = kbase + 8 * g;
                            uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5])),
                                                  pack_bf16(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
                            *reinterpret_cast<uint4 *>(smem + C::B_OFF_D + (kk >> 6) * PANEL_BYTES + sw128(orow, kk & 63)) = pk;
                        }
                    }
                    warp_arrive(BAR(B_PRDY + p), lane);
                }
                // ---- dL/dh_l = delta W_s + sum_e P_e W_e
                mbar_wait(BAR(B_DH), par);
                tc_fence_after();
                tc_ld32(t_lane + COL_DHX + colbase, v);
                tc_wait_ld();
#pragma unroll
                for (int x = 0; x < 32; ++x) acc[x] = __uint_as_float(v[x]);
                if (l == 0) {
                    if (a.d_h0) {
                        float *stg = reinterpret_cast<float *>(smem + C::B_OFF_D + warp * 2048);
#pragma unroll
                        for (int h2 = 0; h2 < 2; ++h2)
                            warp_store_rows<16>(stg, acc + 16 * h2, lane, [&](int r) -> float * {
                                const int tr = 32 * q + r, mg = tile * 2 + (tr >> 6), at = tr & 63;
                                return (mg < a.mb && at < a.N) ? a.d_h0 + ((long)mg * a.N + at) * H + colbase + 16 * h2 : nullptr;
                            });
                    }
                    tc_fence_before();
                    asm volatile("bar.sync 1, %0;" ::"n"(NE));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPW + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(C::TMEM_COLS));
    }
}

// ---- weight images of one layer: bf16, SW128 K-major tiles [H n][64 k]
//   forward : [self KP: B[n][k] = W_s[n][k]] [msg 4KP: K = e*H + c': B[n][K] = W_e[n*4+e][c']]
//   backward: [self KP: B[n][k] = W_s[k][n]] [dh  4KP: K = e*H + c : B[n][K] = W_e[c*4+e][n]]
struct PackArgs {
    int H, bwd;
    const float *self_W, *edge_W;
    uint8_t *img;
};
__global__ void pack_relgcn_kernel(const PackArgs p) {
    const int H = p.H, KP = H / 64;
    const long total = (long)5 * KP * H * 64;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int k = idx & 63, n = (idx >> 6) % H, tile = (int)(idx / (64L * H));
        float w;
        if (tile < KP) {
            const int K = tile * 64 + k;
            w = p.bwd ? p.self_W[(long)K * H + n] : p.self_W[(long)n * H + K];
        } else {
            const int K = (tile - KP) * 64 + k, e = K / H, c = K % H;
            w = p.bwd ? p.edge_W[((long)c * 4 + e) * H + n] : p.edge_W[((long)n * 4 + e) * H + c];
        }
        const uint32_t off = (uint32_t)n * 128u + ((((uint32_t)(k >> 3) ^ ((uint32_t)n & 7u)) << 4) | (((uint32_t)k & 7u) << 1));
        *reinterpret_cast<__nv_bfloat16 *>(p.img + (size_t)tile * H * 128 + off) = __float2bfloat16_rn(w);
    }
}

static size_t image_bytes(int H) { return (size_t)(5 * (H / 64)) * H * 128 + 256; }

// adj_out[b,e,i,j] = adj[b,e,i,j] / max-safe(sum_{e',i'} adj[b,e',i',j])   (models/relgcn.py:20-28)
__global__ void __launch_bounds__(256) rescale_adj_kernel(const float *__restrict__ adj, float *__restrict__ out, int E, int N) {
    __shared__ float part[4][64], inv[BMP_X3_MAX_ATOMS];
    const long base = (long)blockIdx.x * E * N * N;
    column_inverse_degree(adj + base, E, N, part, inv);
    for (int i = threadIdx.x; i < E * N * N; i += blockDim.x) out[base + i] = __ldg(adj + base + i) * inv[i % N];
}

}  // namespace rgt
}  // namespace bmp

using namespace bmp;

int bmp_wgrad_panels(bmp::w2::Args &k, void *stream);   // wgrad_tc2.cu

extern "C" int bmp_rescale_adj(const float *adj, float *adj_out, int mb, int n_edge, int n_atoms, void *stream) {
    if (!adj || !adj_out || mb <= 0 || n_edge <= 0 || n_atoms <= 0) { set_error("bmp_rescale_adj: bad arguments"); return BMP_EINVAL; }
    if (n_atoms > BMP_X3_MAX_ATOMS) { set_error("bmp_rescale_adj: n_atoms=%d outside 1..%d", n_atoms, BMP_X3_MAX_ATOMS); return BMP_ESHAPE; }
    rgt::rescale_adj_kernel<<<mb, 256, 0, (cudaStream_t)stream>>>(adj, adj_out, n_edge, n_atoms);
    count_launch();
    return check_launch("rescale_adj_kernel");
}

extern "C" size_t bmp_relgcn_tc_workspace_bytes(int channels, int n_layers) {
    if (channels != 64 && channels != 128) return 0;
    return rgt::image_bytes(channels) * (size_t)n_layers + 2048;
}

// whether the tcgen05 kernels cover this stack: one channel count in {64, 128} for every layer, 4 bond types
bool bmp_relgcn_tc_supported(const int *ch, int n_layers, int n_edge) {
    if (n_edge != 4 || n_layers < 1 || n_layers > BMP_MAX_STEPS || (ch[0] != 64 && ch[0] != 128)) return false;
    for (int l = 1; l <= n_layers; ++l)
        if (ch[l] != ch[0]) return false;
    return true;
}

static int rgt_pack(rgt::Args &k, int H, int L, const float *const *self_W, const float *const *edge_W, void *ws, size_t ws_bytes,
                    bool ready, bool bwd, cudaStream_t st) {
    if (!ws || ws_bytes < bmp_relgcn_tc_workspace_bytes(H, L)) {
        set_error("BMP_MODE_BF16 RelGCN: tc_workspace of >= %zu bytes required", bmp_relgcn_tc_workspace_bytes(H, L));
        return BMP_EINVAL;
    }
    uint8_t *base = (uint8_t *)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    const size_t ib = rgt::image_bytes(H);
    for (int l = 0; l < L; ++l) {
        if (!self_W[l] || !edge_W[l]) { set_error("BMP_MODE_BF16 RelGCN: null parameter at layer %d", l); return BMP_EINVAL; }
        rgt::PackArgs p;
        p.H = H; p.bwd = bwd; p.self_W = self_W[l]; p.edge_W = edge_W[l]; p.img = base + (size_t)l * ib;
        if (!ready) {
            rgt::pack_relgcn_kernel<<<64, 256, 0, st>>>(p);
            count_launch();
        }
        k.img[l] = p.img;
    }
    return check_launch("pack_relgcn_kernel");
}

int bmp_relgcn_forward_tc(const bmp_relgcn_fwd_t *a, void *stream) {
    const int H = a->ch[0], L = a->n_layers;
    cudaStream_t st = (cudaStream_t)stream;
    if (!aligned16({a->h_in, a->embed_W, a->adj, a->h_out, a->tc_workspace, a->stash2})) { set_error("BMP_MODE_BF16 RelGCN: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    rgt::Args k = {};
    k.mb = a->mb; k.N = a->n_atoms; k.L = L; k.n_types = a->n_atom_types; k.act = a->act; k.scale_adj = a->scale_adj;
    k.atoms = a->atoms; k.embed_W = a->embed_W; k.h_in = a->h_in; k.adj = a->adj; k.adj_u8 = a->adj_u8; k.h_out = a->h_out;
    for (int l = 0; l < L; ++l) {
        k.self_b[l] = a->self_b[l]; k.edge_b[l] = a->edge_b[l];
        if (!aligned16({a->self_b[l], a->edge_b[l]})) { set_error("BMP_MODE_BF16 RelGCN: biases must be 16-byte aligned"); return BMP_EINVAL; }
    }
    int rc = rgt_pack(k, H, L, a->self_W, a->edge_W, a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, false, st);
    if (rc) return rc;
    const int n_tiles = (a->mb + 1) / 2;
    k.use2 = a->stash2 != nullptr;
    if (k.use2) k.st.carve(a->stash2, n_tiles, H, L);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = n_tiles < sms ? n_tiles : sms;
#define LAUNCH_RG(HH, VV)                                                                                                     \
    do {                                                                                                                       \
        cudaFuncSetAttribute(rgt::relgcn_tc_kernel<HH, VV>, cudaFuncAttributeMaxDynamicSharedMemorySize, rgt::Cfg<HH>::SMEM_BYTES); \
        rgt::relgcn_tc_kernel<HH, VV><<<grid, rgt::Cfg<HH>::NT, rgt::Cfg<HH>::SMEM_BYTES, st>>>(k);                              \
    } while (0)
    if (H == 64) { if (k.use2) LAUNCH_RG(64, true); else LAUNCH_RG(64, false); }
    else { if (k.use2) LAUNCH_RG(128, true); else LAUNCH_RG(128, false); }
#undef LAUNCH_RG
    count_launch();
    return check_launch("relgcn_tc_kernel");
}

int bmp_relgcn_backward_tc(const bmp_relgcn_bwd_t *a, void *stream) {
    const int H = a->ch[0], L = a->n_layers, KP = H / 64;
    cudaStream_t st = (cudaStream_t)stream;
    if (!a->stash2 || !a->d_h_out || !a->d_h0) { set_error("BMP_MODE_BF16 RelGCN backward: stash2, d_h_out and d_h0 are required"); return BMP_EINVAL; }
    if (!aligned16({a->adj, a->d_h_out, a->d_h0, a->tc_workspace, a->stash2})) { set_error("BMP_MODE_BF16 RelGCN backward: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    rgt::Args k = {};
    k.mb = a->mb; k.N = a->n_atoms; k.L = L; k.act = a->act; k.scale_adj = a->scale_adj; k.adj = a->adj; k.adj_u8 = a->adj_u8; k.d_h_out = a->d_h_out; k.d_h0 = a->d_h0;
    int rc = rgt_pack(k, H, L, a->self_W, a->edge_W, a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, true, st);
    if (rc) return rc;
    const int n_tiles = (a->mb + 1) / 2;
    k.use2 = 1;
    k.st.carve(a->stash2, n_tiles, H, L);
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = n_tiles < sms ? n_tiles : sms;
    if (H == 64) {
        cudaFuncSetAttribute(rgt::relgcn_tc_bwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, rgt::Cfg<64>::B_SMEM_BYTES);
        rgt::relgcn_tc_bwd_kernel<64><<<grid, rgt::Cfg<64>::NT, rgt::Cfg<64>::B_SMEM_BYTES, st>>>(k);
    } else {
        cudaFuncSetAttribute(rgt::relgcn_tc_bwd_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, rgt::Cfg<128>::B_SMEM_BYTES);
        rgt::relgcn_tc_bwd_kernel<128><<<grid, rgt::Cfg<128>::NT, rgt::Cfg<128>::B_SMEM_BYTES, st>>>(k);
    }
    count_launch();
    if ((rc = check_launch("relgcn_tc_bwd_kernel"))) return rc;
    // parameter gradients: grouped contractions over the dumped panels, one layer at a time
    for (int l = 0; l < L; ++l) {
        if (a->d_self_W[l] || a->d_self_b[l]) {
            for (int mt = 0; mt < KP; mt += 2) {
                w2::Args g = {};
                g.A = k.st.Dp; g.a_ppt = 3 * KP; g.n_mt = 1;
                g.a_panel[0][0] = 2 * KP + mt; g.a_panel[0][1] = mt + 1 < KP ? 2 * KP + mt + 1 : -1;
                g.a_panel[1][0] = g.a_panel[1][1] = -1;
                g.nb = KP;
                for (int j = 0; j < KP; ++j) { g.B[j] = k.st.Xp; g.b_ppt[j] = KP; g.b_panel[j] = j; g.ldc[j] = H; }
                for (int bl = 0; bl < 2; ++bl) {
                    if (g.a_panel[0][bl] < 0) continue;
                    const long row0 = (long)(mt + bl) * 64;
                    for (int j = 0; j < KP; ++j) g.C[0][bl][j] = a->d_self_W[l] ? a->d_self_W[l] + row0 * H + j * 64 : nullptr;
                    g.bias[0][bl] = a->d_self_b[l] ? a->d_self_b[l] + row0 : nullptr;
                }
                g.bias_stride = 1;
                g.t0 = g.t1 = l; g.n_tiles = n_tiles;
                if ((rc = bmp_wgrad_panels(g, stream))) return rc;
            }
        }
        if (a->d_edge_W[l] || a->d_edge_b[l]) {
            for (int e = 0; e < 4; e += 2)
                for (int mt = 0; mt < KP; mt += 2) {
                    w2::Args g = {};
                    g.A = k.st.Pp; g.a_ppt = 4 * KP; g.n_mt = 2;
                    for (int m = 0; m < 2; ++m) {
                        g.a_panel[m][0] = (e + m) * KP + mt;
                        g.a_panel[m][1] = mt + 1 < KP ? (e + m) * KP + mt + 1 : -1;
                    }
                    g.nb = KP;
                    for (int j = 0; j < KP; ++j) { g.B[j] = k.st.Xp; g.b_ppt[j] = KP; g.b_panel[j] = j; g.ldc[j] = 4 * H; }
                    for (int m = 0; m < 2; ++m)
                        for (int bl = 0; bl < 2; ++bl) {
                            if (g.a_panel[m][bl] < 0) continue;
                            const long c0 = (long)(mt + bl) * 64;
                            for (int j = 0; j < KP; ++j) g.C[m][bl][j] = a->d_edge_W[l] ? a->d_edge_W[l] + (c0 * 4 + (e + m)) * H + j * 64 : nullptr;
                            g.bias[m][bl] = a->d_edge_b[l] ? a->d_edge_b[l] + c0 * 4 + (e + m) : nullptr;
                        }
                    g.bias_stride = 4;
                    g.t0 = g.t1 = l; g.n_tiles = n_tiles;
                    if ((rc = bmp_wgrad_panels(g, stream))) return rc;
                }
        }
    }
    return BMP_OK;
}
