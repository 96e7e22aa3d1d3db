// wgrad_tc2.cu -- parameter-gradient contraction over the PANEL stash (BMP_MODE_BF16, stash v2).
//
// The tcgen05 encoder kernels dump their bf16 operand panels ([128 rows][64 cols], 128-byte swizzle)
// verbatim to global memory (cp.async.bulk stores).  A 64-row half of such a panel is, byte for byte, an
// MN-major UMMA operand block [64 k-rows][64 columns], so C += A^T B needs no conversion at all here:
// one lane streams 8 KB blocks with cp.async.bulk into a 3-stage ring, one lane issues M=128 x N x 16 UMMAs
// into TMEM accumulators that live for the CTA's whole row range (split over CTAs), four warps add the tiles
// into C with 128-bit fp32 atomics.  One launch contracts up to two M tiles (2 x 2 A blocks) against up to six
// B blocks drawn from different panel arrays, so every operand byte is read once per launch: the kernel is
// HBM-bound and the launches are grouped to minimise re-reads (ggnn_tc_bwd.cu).  A block can feed two targets
// (W_r[:, :H] and U_r see the same sum when the GRU state is the step input).  Bias gradients (column sums of
// A) come from one extra N=16 UMMA per M tile against a block of ones.
#include <cstdlib>
#include "tc_common.cuh"
#include "det.cuh"

namespace bmp {
namespace w2 {
using namespace tc;

constexpr int BLK = 64 * 128;          // 8 KB operand block
constexpr int STAGES = 3;
constexpr int NTH = 192;               // warps 0-3 epilogue, 4 TMA, 5 MMA

__global__ void __launch_bounds__(NTH, 1) wgrad2_kernel(const __grid_constant__ Multi mm) {
    int ci = 0;
    while (ci + 1 < mm.n && (int)blockIdx.x >= mm.cta0[ci + 1]) ++ci;
    const Args &a = mm.cls[ci];
    const long k0 = (long)blockIdx.x - mm.cta0[ci], kn = mm.cta0[ci + 1] - mm.cta0[ci];      // this CTA: units k0, k0 + kn, ...
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const int NB = a.nb, NMT = a.n_mt, NA = 2 * NMT;
    const int stage_bytes = (NA + NB) * BLK;
    const uint32_t s_ones = sbase + STAGES * stage_bytes;
    const uint32_t s_bar = s_ones + BLK;
    auto FULL = [&](int s) { return s_bar + 8u * s; };
    auto EMPTY = [&](int s) { return s_bar + 8u * (STAGES + s); };
    const uint32_t DONE = s_bar + 8u * (2 * STAGES);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + STAGES * stage_bytes + BLK + 8 * (2 * STAGES + 1) + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long total = (long)(a.t1 - a.t0 + 1) * a.n_tiles * 2;
    bool want_bias = false;
    for (int m = 0; m < 2; ++m)
        for (int b = 0; b < 2; ++b) want_bias |= a.bias[m][b] != nullptr || a.bias2[m][b] != nullptr;
    // accumulator columns: one M tile -> [0, 64 nb) + bias at 496 ; two M tiles -> [256 mt, 256 mt + 64 nb) + bias at 256 mt + 240
    auto col_of = [&](int mt) -> uint32_t { return (uint32_t)mt * 256u; };
    auto bias_col = [&](int mt) -> uint32_t { return NMT == 1 ? 496u : (uint32_t)mt * 256u + 240u; };

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(FULL(s), 1); mbar_init(EMPTY(s), 1); }
        mbar_init(DONE, 1);
        fence_mbar_init();
    }
    // a block of bf16 ones (B operand of the bias column-sum UMMA)
    for (int i = tid; i < BLK / 4; i += NTH) reinterpret_cast<uint32_t *>(smem + STAGES * stage_bytes)[i] = 0x3F803F80u;
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "n"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 4) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            int nblk = NB;
            for (int m = 0; m < NMT; ++m) nblk += (a.a_panel[m][0] >= 0) + (a.a_panel[m][1] >= 0);
            for (long c = k0; c < total; c += kn) {
                const long tt = c / 2;                       // (step, tile) index
                const int half = (int)(c & 1);
                const long step = tt / a.n_tiles, tile = tt % a.n_tiles;
                const long tbase = ((long)(a.t0 + step) * a.n_tiles + tile);
                mbar_wait(EMPTY(stage), phase ^ 1);
                mbar_expect_tx(FULL(stage), nblk * BLK);
                const uint32_t dst = sbase + stage * stage_bytes;
                for (int m = 0; m < NMT; ++m)
                    for (int b = 0; b < 2; ++b)
                        if (a.a_panel[m][b] >= 0)
                            tma_bulk_g2s(dst + (2 * m + b) * BLK, a.A + (tbase * a.a_ppt + a.a_panel[m][b]) * (long)PANEL_BYTES + half * BLK, BLK, FULL(stage));
                for (int j = 0; j < NB; ++j)
                    tma_bulk_g2s(dst + (NA + j) * BLK, a.B[j] + (tbase * a.b_ppt[j] + a.b_panel[j]) * (long)PANEL_BYTES + half * BLK, BLK, FULL(stage));
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {
            const int n1 = NB > 4 ? 4 : NB, n2 = NB - n1;        // UMMA N <= 256: B blocks in two groups
            const uint32_t idN1 = idesc2(n1 * 64, 1, 1), idN2 = idesc2(n2 > 0 ? n2 * 64 : 64, 1, 1), id16 = idesc2(16, 1, 1);
            uint32_t stage = 0, phase = 0;
            // MN-major SW128 blocks: LBO = 8 KB (next 64-column block), SBO = 1024 B (8 k-rows)
            auto desc = [](uint32_t saddr) -> uint64_t {
                return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(BLK >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
            };
            bool first = true;
            for (long c = k0; c < total; c += kn) {
                mbar_wait(FULL(stage), phase);
                tc_fence_after();
                const uint32_t s0 = sbase + stage * stage_bytes, sb = s0 + NA * BLK;
                for (int m = 0; m < NMT; ++m) {
                    const uint32_t sa = s0 + 2 * m * BLK;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t acc = first && k == 0 ? 0u : 1u;
                        tc_mma(tmem + col_of(m), desc(sa + k * 2048), desc(sb + k * 2048), idN1, acc);
                        if (n2 > 0) tc_mma(tmem + col_of(m) + 256, desc(sa + k * 2048), desc(sb + 4 * BLK + k * 2048), idN2, acc);
                        if (want_bias) tc_mma(tmem + bias_col(m), desc(sa + k * 2048), desc(s_ones + k * 2048), id16, acc);
                    }
                }
                first = false;
                tc_commit(EMPTY(stage));
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            tc_commit(DONE);
        }
    } else {
        mbar_wait(DONE, 0);
        tc_fence_after();
        if (k0 < total) {
            const int q = warp, blk = q >> 1, r = (q & 1) * 32 + lane;     // TMEM lane 32q+lane = A column = C row
            const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
            // deterministic mode: this CTA's slot; target (m, blk, j) at ((2m + blk) NB + j) 4096 + 64 r, bias row r of (m, blk)
            // after the 2 NMT NB targets.  C and C2 of a target get the same partial, so they share it.
            float *slot = mm.part[ci] ? mm.part[ci] + k0 * mm.plen[ci] : nullptr;
            for (int m = 0; m < NMT; ++m) {
                if (a.a_panel[m][blk] < 0) continue;
                for (int j = 0; j < NB; ++j) {
                    float *d1 = a.C[m][blk][j] ? a.C[m][blk][j] + (long)r * a.ldc[j] : nullptr;
                    float *d2 = a.C2[m][blk][j] ? a.C2[m][blk][j] + (long)r * a.ldc2[j] : nullptr;
                    if (!d1 && !d2) continue;
                    float *sp = slot ? slot + ((long)(2 * m + blk) * NB + j) * 4096 + 64 * r : nullptr;
                    for (int cc = 0; cc < 64; cc += 32) {
                        uint32_t v[32];
                        tc_ld32(t_lane + col_of(m) + j * 64 + cc, v);
                        tc_wait_ld();
#pragma unroll
                        for (int x = 0; x < 32; x += 4) {     // 128-bit vector reductions (sm_90+): 4x fewer L2 atomic operations
                            const float4 f = make_float4(__uint_as_float(v[x]), __uint_as_float(v[x + 1]), __uint_as_float(v[x + 2]), __uint_as_float(v[x + 3]));
                            if (sp) {
                                det_put4(nullptr, sp + cc + x, f);
                            } else {
                                if (d1) atomicAdd(reinterpret_cast<float4 *>(d1 + cc + x), f);
                                if (d2) atomicAdd(reinterpret_cast<float4 *>(d2 + cc + x), f);
                            }
                        }
                    }
                }
                if (a.bias[m][blk] || a.bias2[m][blk]) {
                    uint32_t w[16];
                    tc_ld16(t_lane + bias_col(m), w);
                    tc_wait_ld();
                    if (slot) {
                        det_put(nullptr, slot + (long)NMT * 2 * NB * 4096 + (2 * m + blk) * 64 + r, __uint_as_float(w[0]));
                    } else {
                        if (a.bias[m][blk]) atomicAdd(a.bias[m][blk] + (long)r * a.bias_stride, __uint_as_float(w[0]));
                        if (a.bias2[m][blk]) atomicAdd(a.bias2[m][blk] + (long)r * a.bias_stride, __uint_as_float(w[0]));
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512));
    }
}

}  // namespace w2
}  // namespace bmp

using namespace bmp;

// Grouped contractions over the panel stash (see w2::Args / w2::Multi in tc_common.cuh): n classes over the same (step, tile)
// range in one launch.  The caller fills the operand / target descriptions; t0, t1, n_tiles must agree between the classes.
int bmp_wgrad_panels_multi(w2::Args *list, int n, void *stream) {
    if (n < 1 || n > w2::MAX_CLASSES) { set_error("bmp_wgrad_panels: %d classes (1..%d)", n, w2::MAX_CLASSES); return BMP_EINVAL; }
    for (int c = 0; c < n; ++c) {
        const w2::Args &k = list[c];
        if (!k.A || k.nb < 1 || k.nb > 6 || k.n_mt < 1 || k.n_mt > 2 || (k.n_mt == 2 && k.nb > 3) || k.t0 != list[0].t0 ||
            k.t1 != list[0].t1 || k.n_tiles != list[0].n_tiles) {
            set_error("bmp_wgrad_panels: bad arguments");
            return BMP_EINVAL;
        }
    }
    if (list[0].t1 < list[0].t0 || list[0].n_tiles <= 0) return BMP_OK;
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const long total = (long)(list[0].t1 - list[0].t0 + 1) * list[0].n_tiles * 2;
    w2::Multi m = {};
    m.n = n;
    // CTAs per class in proportion to the 8 KB blocks a class loads per unit (all classes then advance at the same unit rate)
    int blocks[w2::MAX_CLASSES], sum = 0, smem = 0;
    for (int c = 0; c < n; ++c) {
        int na = 0;
        for (int mt = 0; mt < list[c].n_mt; ++mt) na += (list[c].a_panel[mt][0] >= 0) + (list[c].a_panel[mt][1] >= 0);
        blocks[c] = na + list[c].nb;
        sum += blocks[c];
        const int need = w2::STAGES * (2 * list[c].n_mt + list[c].nb) * w2::BLK + w2::BLK + 256 + 1024;
        smem = need > smem ? need : smem;
    }
    long budget = sms;
    if (budget > (total + 7) / 8 * n) budget = (total + 7) / 8 * n;       // small problems: at least ~8 units per CTA
    if (budget < n) budget = n;
    // largest-remainder split of `budget` CTAs (never more than one wave: every CTA must be resident from the start)
    long share[w2::MAX_CLASSES], rem[w2::MAX_CLASSES], given = 0;
    for (int c = 0; c < n; ++c) {
        share[c] = budget * blocks[c] / sum;
        rem[c] = budget * blocks[c] % sum;
        if (share[c] < 1) { share[c] = 1; rem[c] = -1; }
        given += share[c];
    }
    while (given < budget) {
        int best = 0;
        for (int c = 1; c < n; ++c) if (rem[c] > rem[best]) best = c;
        if (rem[best] < 0) break;
        ++share[best]; rem[best] = -1; ++given;
    }
    while (given > budget) {          // the >= 1 floor overshot: take from the largest class
        int big = 0;
        for (int c = 1; c < n; ++c) if (share[c] > share[big]) big = c;
        if (share[big] <= 1) break;
        --share[big]; --given;
    }
    int used = 0;
    for (int c = 0; c < n; ++c) {
        long ctas = share[c] > total ? total : share[c];
        m.cta0[c] = used;
        used += (int)ctas;
        m.cls[c] = list[c];
    }
    m.cta0[n] = used;
    Partials pt((cudaStream_t)stream);
    if (det_on())
        for (int c = 0; c < n; ++c) {
            m.plen[c] = (long)list[c].n_mt * 2 * list[c].nb * 4096 + list[c].n_mt * 2 * 64;
            if (!(m.part[c] = pt.take((m.cta0[c + 1] - m.cta0[c]) * m.plen[c]))) return BMP_EINVAL;
        }
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(w2::wgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, w2::STAGES * 8 * w2::BLK + w2::BLK + 256 + 1024);
        attr = true;
    }
    ProfScope prof(BMP_PROF_WGRAD, (cudaStream_t)stream);
    w2::wgrad2_kernel<<<(unsigned)used, w2::NTH, smem, (cudaStream_t)stream>>>(m);
    count_launch();
    int rc = check_launch("wgrad2_kernel");
    if (rc || !det_on()) return rc;
    for (int c = 0; c < n; ++c) {
        const w2::Args &k = list[c];
        const int parts = m.cta0[c + 1] - m.cta0[c], NB = k.nb;
        for (int mt = 0; mt < k.n_mt; ++mt)
            for (int blk = 0; blk < 2; ++blk) {
                if (k.a_panel[mt][blk] < 0) continue;
                for (int j = 0; j < NB; ++j) {
                    const float *src = m.part[c] + ((long)(2 * mt + blk) * NB + j) * 4096;
                    pt.add(k.C[mt][blk][j], k.ldc[j], 64, 64, src, parts, m.plen[c]);
                    pt.add(k.C2[mt][blk][j], k.ldc2[j], 64, 64, src, parts, m.plen[c]);
                }
                const float *bsrc = m.part[c] + (long)k.n_mt * 2 * NB * 4096 + (2 * mt + blk) * 64;
                pt.add(k.bias[mt][blk], k.bias_stride, 64, 1, bsrc, parts, m.plen[c]);
                pt.add(k.bias2[mt][blk], k.bias_stride, 64, 1, bsrc, parts, m.plen[c]);
            }
    }
    return pt.reduce("det_reduce_kernel (bmp_wgrad_panels)");
}

int bmp_wgrad_panels(w2::Args &k, void *stream) { return bmp_wgrad_panels_multi(&k, 1, stream); }
