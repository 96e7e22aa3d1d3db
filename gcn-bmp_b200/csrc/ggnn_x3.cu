// ggnn_x3.cu -- BMP_MODE_F32 GGNN encoder with every H x H contraction on tcgen05 at fp32-grade accuracy.
//
// Same arithmetic as ggnn.cu (models/update/ggnn_update.py:31-63, models/models/ggnn.py:72-106) and the same fp32 stash
// (Hs / Ms / Gs / RSs / Ps / dHs as include/gcnbmp.h describes them), but the dense products run on the tensor cores:
// every fp32 operand is split into a bf16 hi / lo pair (x = hi + lo up to 2^-17 relative) and each product is three
// UMMAs, hi.hi + lo.hi + hi.lo, into an fp32 TMEM accumulator (the lo.lo term is below fp32 rounding).  The step is a
// short sequence of launches over the FLAT row space (rows = mb * N atoms; the GEMMs never see molecule boundaries):
//
//   forward step t        agg          AH_e = A_e h_t (non-zeros of the dense adjacency through bit masks, FFMA), deg_e = A_e 1
//                         rowgemm3     m   = [AH_0 .. AH_3 | deg] [W_0 .. W_3 | b]^T  (the bias rides as a K block)  -> Ms[t]
//                         rowgemm3     r,z = sigma([h | m] [W_r + U_r | ..]^T + b), r*h                -> Gs[t], RSs[t]
//                         rowgemm3     hb  = tanh([h | m | r*h] [W | U]^T + b), h' = z hb + (1 - z) h  -> Gs[t], Hs[t+1]
//   backward step t       gate_bwd     delta_z, delta_h, g (1 - z)            (pointwise)
//                         rowgemm3     q = delta_h U -> delta_r, ds += q r
//                         rowgemm3     dh_x = [dz | dh | dr] [W_z + U_z | W | W_r + U_r]_h (+ ds) ; dm = [..] [..]_m
//                         agg          P_e = A_e^T dm                                                  -> Ps[t]
//                         rowgemm3     dHs[t] += dh_x + sum_e P_e W_e
// The parameter gradients stay where they were: bmp_ggnn_backward's contractions over the stash (bmp_wgrad_tc3).
//
// rowgemm3: one persistent CTA per SM; a work item = (128-row tile, job), jobs of one launch interleaved so the CTAs that
// share an A tile run at the same time (second reader hits L2).  Warp roles: 8 epilogue warps (TMEM lane quarter x column half),
// 6 converter warps (fp32 rows, landed in a two-deep shared-memory ring by one cp.async.bulk copy per row, -> hi / lo
// SW128 K-major panels), one producer warp (fp32 A rows and packed hi / lo weight k-tiles, cp.async.bulk + mbarrier), one MMA lane.  Two 128-column
// TMEM accumulators alternate between consecutive items, so an item's epilogue overlaps the next item's MMAs.
#include <cstdio>
#include <cstring>
#include <cuda.h>
#include "tc_common.cuh"

namespace bmp {
namespace x3 {
using namespace tc;

constexpr int MAXB = 6, MAXJ = 4;
constexpr int STAGES = 2;
constexpr int STAGE_BYTES = 2 * PANEL_BYTES;      // converted A operand: [A_hi | A_lo]
constexpr int WDEPTH = 3;                         // packed weight k-tiles in flight (own ring: the L2 latency of a tile is hidden)
constexpr int F32_DEPTH = 2;                      // fp32 A k-tiles in flight per CTA (cp.async.bulk row copies)
constexpr int WSLOT = 2 * PANEL_BYTES;            // one packed weight k-tile: hi (n x 64 bf16, SW128) then lo
constexpr int NEPI_W = 8, NCONV_W = 6;
constexpr int NT = 32 * (NEPI_W + NCONV_W + 2);   // 512 threads: 128 registers each
constexpr int NCONV = 32 * NCONV_W;
constexpr int NU = (2048 + NCONV - 1) / NCONV;    // float4 of a 128 x 64 fp32 k-tile per converter thread (last round partial)
constexpr int F32_SLOT = 128 * 256;                // one fp32 A k-tile: 128 rows x 64 floats, row-major (a bulk copy per row)
constexpr int OFF_WR = STAGES * STAGE_BYTES;        // weight ring: WDEPTH x [W_hi | W_lo]
constexpr int OFF_F32 = OFF_WR + WDEPTH * 2 * PANEL_BYTES;
constexpr int OFF_BAR = OFF_F32 + F32_DEPTH * F32_SLOT;
constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;

enum { EPI_MSG = 0, EPI_R, EPI_Z, EPI_HB, EPI_Q, EPI_DHX, EPI_DM, EPI_DHMSG, EPI_LIN /* accumulator + bias */, EPI_TANH /* tanh(accumulator + bias) */ };

struct Job {
    const float *A[MAXB];            // K-block b: (rows, 64 * kt[b]) fp32, leading dimension lda[b]
    int lda[MAXB], kt[MAXB], nblk;
    const uint8_t *wimg;             // packed weight k-tiles of this job (and column chunk) in consumption order
    int epi;
    const float *bias, *bias2;       // per output column (pointers already at column n0), either may be NULL
    const float *in0, *in1, *in2;    // epilogue inputs, row-major, pointers at (row 0, column n0)
    int li0, li1, li2;
    float *out0, *out1, *out2;
    int lo0, lo1, lo2;
};
struct Args {
    CUtensorMap tmap[MAXJ][MAXB];    // K-block b of job j as a 2-D fp32 tensor (rows x 64 kt[b] columns, row stride lda[b]); box 128 x 64
    Job job[MAXJ];
    int njobs, NC;                   // NC = columns per job: 64 or 128
    long rows;
    long long *dbg;                  // optional wait-cycle counters of CTA 0 (tools/x3_check.py --waits)
};

// ------------------------------------------------------------------------------------------------ rowgemm3
__device__ __forceinline__ float sigmoid_x3(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
// 1 - 2 / (1 + e^{2x}): absolute error at the fp32 rounding level of the result's range
__device__ __forceinline__ float tanh_x3(float x) { return 1.f - __fdividef(2.f, 1.f + __expf(2.f * x)); }
// tcgen05.ld 16x256b.x2: 16 TMEM lanes x 16 columns; thread t gets, for column group j (8 columns) and row half rh,
// registers 4 j + 2 rh + {0, 1} = (lane t / 4 + 8 rh, columns 8 j + 2 (t % 4) + {0, 1})
__device__ __forceinline__ void tc_ld_16x256b_x2(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <bool DBG>
__global__ void __launch_bounds__(NT, 1) rowgemm3_kernel(const __grid_constant__ Args a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_bar = sbase + OFF_BAR;
    auto FULL = [&](int s) { return s_bar + 8u * s; };
    auto EMPTY = [&](int s) { return s_bar + 8u * (STAGES + s); };
    auto ACCF = [&](int b) { return s_bar + 8u * (2 * STAGES + b); };
    auto ACCE = [&](int b) { return s_bar + 8u * (2 * STAGES + 2 + b); };
    auto F32F = [&](int d) { return s_bar + 8u * (2 * STAGES + 4 + d); };
    auto F32E = [&](int d) { return s_bar + 8u * (2 * STAGES + 4 + F32_DEPTH + d); };
    auto WFULL = [&](int d) { return s_bar + 8u * (2 * STAGES + 4 + 2 * F32_DEPTH + d); };
    auto WEMPTY = [&](int d) { return s_bar + 8u * (2 * STAGES + 4 + 2 * F32_DEPTH + WDEPTH + d); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_BAR + 8 * (2 * STAGES + 4 + 2 * F32_DEPTH + 2 * WDEPTH) + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int NC = a.NC, njobs = a.njobs;
    const long nrows = a.rows;
    const long ntiles = (nrows + 127) / 128, nitems = ntiles * njobs;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(FULL(s), NCONV_W); mbar_init(EMPTY(s), 1); }
        for (int d = 0; d < WDEPTH; ++d) { mbar_init(WFULL(d), 1); mbar_init(WEMPTY(d), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(ACCF(b), 1); mbar_init(ACCE(b), NEPI_W); }
        for (int d = 0; d < F32_DEPTH; ++d) { mbar_init(F32F(d), 1); mbar_init(F32E(d), NCONV_W); }
        fence_mbar_init();
    }
    if (warp == NEPI_W + NCONV_W + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == NEPI_W + NCONV_W) {
        // ===================== producer (whole warp): per k-tile the fp32 A rows (one 256-byte bulk copy per row, four
        // rows per lane, into the fp32 ring) and the packed hi / lo weight tile (lane 0, into the operand stage)
        uint32_t stage = 0, phase = 0, slot = 0, fphase = 0;
        const uint32_t wb = (uint32_t)NC * 128u;
        for (long w = blockIdx.x; w < nitems; w += gridDim.x) {
            const Job &J = a.job[(int)(w % njobs)];
            const long row0 = (w / njobs) * 128;
            const int left = nrows - row0 >= 128 ? 128 : (int)(nrows - row0);
            {   // the item's epilogue inputs towards L2
                const int lpr = NC / 32;
                for (int idx = lane; idx < left * lpr; idx += 32) {
                    const long row = row0 + idx / lpr;
                    const int c0 = (idx % lpr) * 32;
                    if (J.in0) prefetch_l2(J.in0 + row * J.li0 + c0);
                    if (J.in1) prefetch_l2(J.in1 + row * J.li1 + c0);
                    if (J.in2) prefetch_l2(J.in2 + row * J.li2 + c0);
                }
            }
            int k = 0;
            for (int b = 0; b < J.nblk; ++b) {
                for (int kb = 0; kb < J.kt[b]; ++kb, ++k) {
                    if (lane == 0) {
                        mbar_wait_sleep(F32E(slot), fphase ^ 1, 100);
                        mbar_expect_tx(F32F(slot), (uint32_t)F32_SLOT);
                        // one tensor copy: 128 rows x 64 floats, rows past the end arrive as zeros
                        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                                     ::"r"(sbase + OFF_F32 + slot * F32_SLOT), "l"(&a.tmap[(int)(w % njobs)][b]), "r"(kb * 64), "r"((int)row0),
                                       "r"(F32F(slot)) : "memory");
                    }
                    if (++slot == F32_DEPTH) { slot = 0; fphase ^= 1; }
                    if (lane == 0) {
                        mbar_wait_sleep(WEMPTY(stage), phase ^ 1, 100);
                        mbar_expect_tx(WFULL(stage), 2 * wb);
                        const uint32_t wd = sbase + OFF_WR + stage * 2 * PANEL_BYTES;
                        tma_bulk_g2s(wd, J.wimg + (size_t)k * WSLOT, wb, WFULL(stage));
                        tma_bulk_g2s(wd + PANEL_BYTES, J.wimg + (size_t)k * WSLOT + PANEL_BYTES, wb, WFULL(stage));
                    }
                    if (++stage == WDEPTH) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == NEPI_W + NCONV_W + 1) {
        // ===================== MMA issuer
        if (lane == 0) {
            const uint32_t ID = idesc(NC, 0);
            uint32_t stage = 0, phase = 0, ws = 0, wphase = 0, it = 0;
            const bool dbg = DBG && blockIdx.x == 0;
            long long t_all = dbg ? clock64() : 0, w_full = 0, w_wfull = 0, w_acce = 0, t0 = 0;
            for (long w = blockIdx.x; w < nitems; w += gridDim.x, ++it) {
                const Job &J = a.job[(int)(w % njobs)];
                int nk = 0;
                for (int b = 0; b < J.nblk; ++b) nk += J.kt[b];
                const uint32_t buf = it & 1, use = it >> 1;
                if (dbg) t0 = clock64();
                mbar_wait_sleep(ACCE(buf), (use & 1) ^ 1, 100);           // the epilogue has drained this accumulator's previous item
                if (dbg) w_acce += clock64() - t0;
                tc_fence_after();
                const uint32_t d = tmem + buf * 128;
                for (int k = 0; k < nk; ++k) {
                    if (dbg) t0 = clock64();
                    mbar_wait(WFULL(ws), wphase);
                    if (dbg) { w_wfull += clock64() - t0; t0 = clock64(); }
                    mbar_wait(FULL(stage), phase);
                    if (dbg) w_full += clock64() - t0;
                    tc_fence_after();
                    const uint32_t sa = sbase + stage * STAGE_BYTES, sw = sbase + OFF_WR + ws * 2 * PANEL_BYTES;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t ah = desc_kmajor(sa + ks * 32), al = desc_kmajor(sa + PANEL_BYTES + ks * 32);
                        const uint64_t wh = desc_kmajor(sw + ks * 32), wl = desc_kmajor(sw + PANEL_BYTES + ks * 32);
                        tc_mma(d, ah, wh, ID, (k | ks) ? 1u : 0u);      // hi . hi
                        tc_mma(d, al, wh, ID, 1u);                      // lo . hi
                        tc_mma(d, ah, wl, ID, 1u);                      // hi . lo
                    }
                    tc_commit(EMPTY(stage));
                    tc_commit(WEMPTY(ws));
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                    if (++ws == WDEPTH) { ws = 0; wphase ^= 1; }
                }
                tc_commit(ACCF(buf));
            }
            if (dbg) { a.dbg[0] = clock64() - t_all; a.dbg[1] = w_full; a.dbg[2] = w_acce; a.dbg[7] = w_wfull; }
        }
    } else if (warp >= NEPI_W) {
        // ===================== converters: fp32 rows -> bf16 hi / lo K-major panels
        // Thread ct owns the 16-byte piece p = ct & 15 of the rows r0 + 12 u (r0 = ct >> 4, u = 0..10; the last round
        // only for ct < 128): fp32 source and swizzled panel offset are a base plus a constant per round.
        const int ct = tid - 32 * NEPI_W;
        const int r0 = ct >> 4, p = ct & 15;
        const bool last_round = ct < 2048 - (NU - 1) * NCONV;
        const uint32_t sw_a = (uint32_t)r0 * 128u + ((((uint32_t)(p >> 1)) ^ ((uint32_t)r0 & 7u)) << 4) + (uint32_t)(p & 1) * 8u;
        const uint32_t sw_b = (uint32_t)r0 * 128u + ((((uint32_t)(p >> 1)) ^ ((uint32_t)(r0 + 4) & 7u)) << 4) + (uint32_t)(p & 1) * 8u;
        const uint32_t f32_mine = sbase + OFF_F32 + (uint32_t)r0 * 256u + (uint32_t)p * 16u;
        const bool dbg = DBG && blockIdx.x == 0 && ct == 0;
        long long w_empty = 0, w_conv = 0, t0 = 0;
        uint32_t stage = 0, phase = 0, slot = 0, fphase = 0;
        for (long w = blockIdx.x; w < nitems; w += gridDim.x) {
            const Job &J = a.job[(int)(w % njobs)];
            int nk = 0;
            for (int b = 0; b < J.nblk; ++b) nk += J.kt[b];
            for (int k = 0; k < nk; ++k) {
                if (dbg) t0 = clock64();
                mbar_wait(F32F(slot), fphase);
                mbar_wait(EMPTY(stage), phase ^ 1);
                if (dbg) { w_empty += clock64() - t0; t0 = clock64(); }
                const uint32_t hi = sbase + stage * STAGE_BYTES, mine = f32_mine + slot * F32_SLOT;
#pragma unroll
                for (int u = 0; u < NU; ++u) {
                    if (u == NU - 1 && !last_round) break;
                    float4 x;
                    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(mine + (uint32_t)u * (12u * 256u)));
                    const uint32_t off = hi + ((u & 1) ? sw_b : sw_a) + (uint32_t)u * (12u * 128u);
                    const uint32_t hx = pack_bf16(x.x, x.y), hy = pack_bf16(x.z, x.w);
                    const uint32_t lx = pack_bf16(x.x - __uint_as_float(hx << 16), x.y - __uint_as_float(hx & 0xFFFF0000u));
                    const uint32_t ly = pack_bf16(x.z - __uint_as_float(hy << 16), x.w - __uint_as_float(hy & 0xFFFF0000u));
                    asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(off), "r"(hx), "r"(hy) : "memory");
                    asm volatile("st.shared.v2.b32 [%0], {%1,%2};" ::"r"(off + PANEL_BYTES), "r"(lx), "r"(ly) : "memory");
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { mbar_arrive(F32E(slot)); mbar_arrive(FULL(stage)); }
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
                if (++slot == F32_DEPTH) { slot = 0; fphase ^= 1; }
                if (dbg) w_conv += clock64() - t0;
            }
        }
        if (dbg) { a.dbg[3] = w_empty; a.dbg[4] = w_conv; }
    } else {
        // ===================== epilogue: TMEM -> pointwise -> global
        // warp = TMEM lane quarter (warp & 3) x column half (warp >> 2); 16-column chunks read with the 16x256b shape: a
        // thread holds column PAIRS of four rows (lane / 4 + 8 rr), so four lanes cover one 32-byte sector of a row and every
        // global access of the warp moves eight full sectors -- no transposition through shared memory.
        const int q = warp & 3, half = warp >> 2;
        const int tr = lane >> 2, tc2 = (lane & 3) * 2;
        const int nch = NC / 32;                               // chunks of this warp
        uint32_t it = 0;
        const bool dbg = DBG && blockIdx.x == 0 && tid == 0;
        long long w_accf = 0, w_epi = 0, t0 = 0;
        for (long w = blockIdx.x; w < nitems; w += gridDim.x, ++it) {
            const Job &J = a.job[(int)(w % njobs)];
            const int epi = J.epi;
            if (dbg) t0 = clock64();
            const long wrow = (w / njobs) * 128 + 32 * q + tr;       // first of this thread's four rows (+ 8 rr)
            const int live = nrows > wrow ? (int)((nrows - wrow + 7) >> 3) : 0;   // rows rr < live exist
            const uint32_t buf = it & 1, use = it >> 1;
            const bool u0 = epi == EPI_R || epi == EPI_HB || epi == EPI_Q || epi == EPI_DHMSG || (epi == EPI_DHX && J.in0);
            const bool u1 = (epi == EPI_HB && J.in1) || epi == EPI_Q || epi == EPI_DHMSG;
            const bool u2 = epi == EPI_Q;
            mbar_wait_sleep(ACCF(buf), use & 1, 100);
            if (dbg) { w_accf += clock64() - t0; t0 = clock64(); }
            tc_fence_after();
            for (int cc = 0; cc < nch; ++cc) {
                const int c0 = half * (NC / 2) + cc * 16, col = c0 + tc2;
                auto LD = [&](const float *p, int ld, float2 (&x)[4][2]) {
                    const float *b = p + wrow * ld + col;
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr)
#pragma unroll
                        for (int j = 0; j < 2; ++j)
                            x[rr][j] = rr < live ? __ldg(reinterpret_cast<const float2 *>(b + (long)(8 * rr) * ld + 8 * j)) : make_float2(0.f, 0.f);
                };
                auto ST = [&](float *p, int ld, const float2 (&x)[4][2]) {
                    float *b = p + wrow * ld + col;
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr)
#pragma unroll
                        for (int j = 0; j < 2; ++j)
                            if (rr < live) *reinterpret_cast<float2 *>(b + (long)(8 * rr) * ld + 8 * j) = x[rr][j];
                };
                // the global inputs of the chunk are requested before the accumulator is read
                float2 x0[4][2], x1[4][2], x2[4][2], f[4][2];
                if (u0) LD(J.in0, J.li0, x0);
                if (u1) LD(J.in1, J.li1, x1);
                if (u2) LD(J.in2, J.li2, x2);
                {
                    uint32_t v0[8], v1[8];
                    tc_ld_16x256b_x2(tmem + ((uint32_t)(32 * q) << 16) + buf * 128 + c0, v0);
                    tc_ld_16x256b_x2(tmem + ((uint32_t)(32 * q + 16) << 16) + buf * 128 + c0, v1);
                    tc_wait_ld();
#pragma unroll
                    for (int j = 0; j < 2; ++j)
#pragma unroll
                        for (int rh = 0; rh < 2; ++rh) {
                            f[rh][j] = make_float2(__uint_as_float(v0[4 * j + 2 * rh]), __uint_as_float(v0[4 * j + 2 * rh + 1]));
                            f[2 + rh][j] = make_float2(__uint_as_float(v1[4 * j + 2 * rh]), __uint_as_float(v1[4 * j + 2 * rh + 1]));
                        }
                }
                if (cc == nch - 1) {                                 // every TMEM read of this item is done
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(ACCE(buf));
                }
                if (epi == EPI_R || epi == EPI_Z || epi == EPI_HB || epi == EPI_LIN || epi == EPI_TANH) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        float2 b2 = make_float2(0.f, 0.f);
                        if (J.bias) b2 = __ldg(reinterpret_cast<const float2 *>(J.bias + col + 8 * j));
                        if (J.bias2) {
                            const float2 t2 = __ldg(reinterpret_cast<const float2 *>(J.bias2 + col + 8 * j));
                            b2.x += t2.x; b2.y += t2.y;
                        }
#pragma unroll
                        for (int rr = 0; rr < 4; ++rr) { f[rr][j].x += b2.x; f[rr][j].y += b2.y; }
                    }
                }
#define X3_EACH(expr)                                  \
    _Pragma("unroll") for (int rr = 0; rr < 4; ++rr)   \
    _Pragma("unroll") for (int j = 0; j < 2; ++j) { expr; }
                switch (epi) {
                    case EPI_R: {               // x0 = state
                        X3_EACH(f[rr][j].x = sigmoid_x3(f[rr][j].x); f[rr][j].y = sigmoid_x3(f[rr][j].y);
                                x0[rr][j].x *= f[rr][j].x; x0[rr][j].y *= f[rr][j].y)
                        ST(J.out0, J.lo0, f);
                        ST(J.out1, J.lo1, x0);
                        break;
                    }
                    case EPI_Z: {
                        X3_EACH(f[rr][j].x = sigmoid_x3(f[rr][j].x); f[rr][j].y = sigmoid_x3(f[rr][j].y))
                        ST(J.out0, J.lo0, f);
                        if (J.out1) {           // stateless step: zero r slot and r*state (keeps the merged wgrad contractions exact)
                            X3_EACH(f[rr][j] = make_float2(0.f, 0.f))
                            ST(J.out1, J.lo1, f);
                            ST(J.out2, J.lo2, f);
                        }
                        break;
                    }
                    case EPI_HB: {              // x0 = z, x1 = state
                        X3_EACH(f[rr][j].x = tanh_x3(f[rr][j].x); f[rr][j].y = tanh_x3(f[rr][j].y))
                        ST(J.out0, J.lo0, f);
                        if (u1) {
                            X3_EACH(f[rr][j].x = x0[rr][j].x * f[rr][j].x + (1.f - x0[rr][j].x) * x1[rr][j].x;
                                    f[rr][j].y = x0[rr][j].y * f[rr][j].y + (1.f - x0[rr][j].y) * x1[rr][j].y)
                        } else {
                            X3_EACH(f[rr][j].x *= x0[rr][j].x; f[rr][j].y *= x0[rr][j].y)
                        }
                        ST(J.out1, J.lo1, f);
                        if (J.out2) ST(J.out2, J.lo2, f);
                        break;
                    }
                    case EPI_Q: {               // x0 = state, x1 = r, x2 = ds
                        X3_EACH(x2[rr][j].x += f[rr][j].x * x1[rr][j].x; x2[rr][j].y += f[rr][j].y * x1[rr][j].y;
                                f[rr][j].x *= x0[rr][j].x * x1[rr][j].x * (1.f - x1[rr][j].x);
                                f[rr][j].y *= x0[rr][j].y * x1[rr][j].y * (1.f - x1[rr][j].y))
                        ST(J.out0, J.lo0, f);
                        ST(J.out1, J.lo1, x2);
                        break;
                    }
                    case EPI_DHX: {
                        if (u0) { X3_EACH(f[rr][j].x += x0[rr][j].x; f[rr][j].y += x0[rr][j].y) }
                        ST(J.out0, J.lo0, f);
                        break;
                    }
                    case EPI_DHMSG: {
                        X3_EACH(f[rr][j].x += x0[rr][j].x + x1[rr][j].x; f[rr][j].y += x0[rr][j].y + x1[rr][j].y)
                        ST(J.out0, J.lo0, f);
                        break;
                    }
                    case EPI_TANH: {
                        X3_EACH(f[rr][j].x = tanh_x3(f[rr][j].x); f[rr][j].y = tanh_x3(f[rr][j].y))
                        ST(J.out0, J.lo0, f);
                        break;
                    }
                    default:                    // EPI_MSG (bias rides in the K stream), EPI_DM, EPI_LIN: the accumulator as it is
                        ST(J.out0, J.lo0, f);
                        break;
                }
#undef X3_EACH
            }
            if (dbg) w_epi += clock64() - t0;
        }
        if (dbg) { a.dbg[5] = w_accf; a.dbg[6] = w_epi; }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NEPI_W + NCONV_W + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256));
    }
}

// ------------------------------------------------------------------------------------------------ weight images
// Image of one step's parameters: the k-tiles of the eight jobs in consumption order, per 128-column output chunk.
//   job        K-blocks (each H/64 k-tiles)                           B element (n = output column, k = K index)
//   MSG        AH_0 .. AH_3, deg (one k-tile: columns 0-3 = deg_e)    msg_W[(n*4 + e)*H + k] ; msg_b[n*4 + k] (k < 4)
//   R          h, m                                                   W_r[n][k] + U_r[n][k] ; W_r[n][H + k]
//   Z          h, m                                                   W_z[n][k] (+ U_z[n][k] stateful) ; W_z[n][H + k]
//   HB         h, m, r*h                                              W[n][k] ; W[n][H + k] ; U[n][k]
//   Q          delta_h                                                U[k][n]
//   DHX        delta_z, delta_h, delta_r                              W_z[k][n] (+ U_z[k][n]) ; W[k][n] ; W_r[k][n] + U_r[k][n]
//   DM         delta_z, delta_h, delta_r                              W_z[k][H + n] ; W[k][H + n] ; W_r[k][H + n]
//   DHMSG      P_0 .. P_3                                             msg_W[(k*4 + e)*H + n]
__host__ __device__ inline int job_blocks(int j) { return (j == EPI_MSG || j == EPI_DHMSG) ? 4 : (j == EPI_Q ? 1 : (j == EPI_R || j == EPI_Z) ? 2 : 3); }
__host__ __device__ inline int job_ktiles(int j, int H) { return job_blocks(j) * (H / 64) + (j == EPI_MSG ? 1 : 0); }   // per column chunk
__host__ __device__ inline int job_tile0(int j, int H) {      // first k-tile of job j (chunk 0) inside an image
    const int hc = (H + 127) / 128;
    int t = 0;
    for (int i = 0; i < j; ++i) t += job_ktiles(i, H) * hc;
    return t;
}
__host__ __device__ inline int image_tiles(int H) { return job_tile0(8, H); }

struct PackArgs {
    const float *msg_W, *msg_b;
    bmp_gru_t g;
    int H, stateful;
    uint8_t *img;
};

__global__ void __launch_bounds__(256) pack_x3_kernel(const PackArgs a) {
    const int H = a.H, kb = H / 64, hc = (H + 127) / 128, NC = H < 128 ? H : 128;
    int tile = blockIdx.x, j = 0;
    while (j < 7 && tile >= job_tile0(j + 1, H)) ++j;
    const int local = tile - job_tile0(j, H), per = job_ktiles(j, H);
    const int nc = local / per, kk = local % per, b = kk / kb, kbase = (kk % kb) * 64;      // b == 4 (MSG only): the bias k-tile
    (void)hc;
    const bool st = a.stateful != 0;
    auto val = [&](int n, int k) -> float {       // n: global output column, k: column inside K-block b
        const bmp_gru_t &g = a.g;
        const long H2 = 2L * H;
        switch (j) {
            case EPI_MSG: return b < 4 ? a.msg_W[((long)n * 4 + b) * H + k] : (k < 4 && a.msg_b ? a.msg_b[(long)n * 4 + k] : 0.f);
            case EPI_R: return b == 0 ? (st ? g.W_r[n * H2 + k] + g.U_r[(long)n * H + k] : 0.f) : (st ? g.W_r[n * H2 + H + k] : 0.f);
            case EPI_Z: return b == 0 ? g.W_z[n * H2 + k] + (st ? g.U_z[(long)n * H + k] : 0.f) : g.W_z[n * H2 + H + k];
            case EPI_HB: return b == 0 ? g.W[n * H2 + k] : (b == 1 ? g.W[n * H2 + H + k] : (st ? g.U[(long)n * H + k] : 0.f));
            case EPI_Q: return st ? g.U[(long)k * H + n] : 0.f;
            case EPI_DHX:
                return b == 0 ? g.W_z[k * H2 + n] + (st ? g.U_z[(long)k * H + n] : 0.f)
                              : (b == 1 ? g.W[k * H2 + n] : (st ? g.W_r[k * H2 + n] + g.U_r[(long)k * H + n] : 0.f));
            case EPI_DM: return b == 0 ? g.W_z[k * H2 + H + n] : (b == 1 ? g.W[k * H2 + H + n] : (st ? g.W_r[k * H2 + H + n] : 0.f));
            default: return a.msg_W[((long)k * 4 + b) * H + n];
        }
    };
    uint8_t *dst = a.img + (size_t)tile * WSLOT;
    for (int idx = threadIdx.x; idx < NC * 8; idx += 256) {
        const int n = idx % NC, c8 = idx / NC;        // n fastest: the transposed jobs read consecutive addresses
        float v[8];
#pragma unroll
        for (int x = 0; x < 8; ++x) v[x] = val(nc * 128 + n, kbase + c8 * 8 + x);
        uint32_t h[4], l[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            h[x] = pack_bf16(v[2 * x], v[2 * x + 1]);
            l[x] = pack_bf16(v[2 * x] - __uint_as_float(h[x] << 16), v[2 * x + 1] - __uint_as_float(h[x] & 0xFFFF0000u));
        }
        const uint32_t off = sw128(n, c8 * 8);
        *reinterpret_cast<uint4 *>(dst + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4 *>(dst + PANEL_BYTES + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// ------------------------------------------------------------------------------------------------ adjacency products
// The adjacency is the reference's dense fp32 (mb,E,N,N) array, > 97 % zeros.  It is scanned ONCE per encoder call into bit masks
// (64 bits per row and per column of every bond type, 4 KB per molecule instead of 64 KB) plus a flag "some non-zero entry is not
// 1.0"; the per-step products then walk the set bits in ascending order -- the dense sum with the zeros skipped -- and touch the
// dense array again only when that flag is set (general fp32 weights).
// masks[mol][0][e][i][w] bit b = (A_e[i][64 w + b] != 0) ; masks[mol][1][e][j][w] bit b = (A_e[64 w + b][j] != 0) ; W = ceil(N / 64) words
__global__ void __launch_bounds__(256) adj_mask_kernel(const float *__restrict__ adj, unsigned long long *__restrict__ masks, int *nonbinary,
                                                       int mb, int N) {
    extern __shared__ unsigned long long cm[];                   // [4][N][W] column masks
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, W = (N + 63) >> 6, per = 4 * N * W;
    for (int mol = blockIdx.x; mol < mb; mol += gridDim.x) {
        __syncthreads();
        for (int idx = tid; idx < per; idx += 256) cm[idx] = 0ull;
        unsigned long long *out = masks + (size_t)mol * 2 * per;
        __syncthreads();
        bool odd = false;
        for (int idx = warp; idx < 4 * N; idx += 8) {
            const int e = idx / N, i = idx - e * N;
            const float *arow = adj + (((long)mol * 4 + e) * N + i) * N;
            for (int w = 0; w < W; ++w) {
                const int j0 = 64 * w + lane, j1 = j0 + 32;
                const float a0 = j0 < N ? __ldg(arow + j0) : 0.f, a1 = j1 < N ? __ldg(arow + j1) : 0.f;
                const unsigned long long m = (unsigned long long)__ballot_sync(0xffffffffu, a0 != 0.f) |
                                             ((unsigned long long)__ballot_sync(0xffffffffu, a1 != 0.f) << 32);
                if (lane == 0) out[(e * N + i) * W + w] = m;
                if (a0 != 0.f) atomicOr(&cm[(e * N + j0) * W + (i >> 6)], 1ull << (i & 63));
                if (a1 != 0.f) atomicOr(&cm[(e * N + j1) * W + (i >> 6)], 1ull << (i & 63));
                odd = odd || (a0 != 0.f && a0 != 1.f) || (a1 != 0.f && a1 != 1.f);
            }
        }
        if (__any_sync(0xffffffffu, odd) && lane == 0) *nonbinary = 1;
        __syncthreads();
        for (int idx = tid; idx < per; idx += 256) out[per + idx] = cm[idx];
    }
}

// BWD = false: dst[row i][e*H + c] = sum_j A_e[i][j] src[j][c]  (A_e h; deg[row][e] = sum_j A_e[i][j] into rows of 64 floats, the A
//              operand of the bias k-tile)
// BWD = true : dst[row j][e*H + c] = sum_i A_e[i][j] src[i][c]  (A_e^T dm)                                    one CTA per molecule
// cscale (mb, N) or NULL: every A_e[i][j] is taken times cscale[mol][j] (RelGCN's rescale_adj), deg included
template <bool BWD>
__global__ void __launch_bounds__(256) agg_kernel(const unsigned long long *__restrict__ masks, const int *__restrict__ nonbinary,
                                                  const float *__restrict__ adj, const float *__restrict__ src, float *__restrict__ dst,
                                                  float *__restrict__ deg, int mb, int N, int H, const float *__restrict__ cscale) {
    extern __shared__ __align__(16) float sh[];                  // [N][H]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, HV = H / 4, W = (N + 63) >> 6, per = 4 * N * W;
    const bool general = *nonbinary != 0;
    for (int mol = blockIdx.x; mol < mb; mol += gridDim.x) {
        __syncthreads();
        const float4 *s4 = reinterpret_cast<const float4 *>(src + (long)mol * N * H);
        for (int idx = tid; idx < N * HV; idx += 256) reinterpret_cast<float4 *>(sh)[idx] = __ldg(s4 + idx);
        __syncthreads();
        const unsigned long long *mk = masks + (size_t)mol * 2 * per + (BWD ? per : 0);
        const float *am = adj + (long)mol * 4 * N * N;
        const float *cs = cscale ? cscale + (long)mol * N : nullptr;
        for (int idx = warp; idx < 4 * N; idx += 8) {
            const int e = idx / N, x = idx - e * N;
            float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
            float d = 0.f;
            for (int w = 0; w < W; ++w) {
                unsigned long long m = __ldg(mk + (e * N + x) * W + w);
                while (m) {
                    const int y = 64 * w + __ffsll((long long)m) - 1;
                    m &= m - 1;
                    float v = general ? __ldg(am + ((long)e * N + (BWD ? y : x)) * N + (BWD ? x : y)) : 1.f;
                    if (cs) v *= cs[BWD ? x : y];
                    d += v;
                    const float4 *hr = reinterpret_cast<const float4 *>(sh + y * H);
                    if (lane < HV) {
                        const float4 t = hr[lane];
                        acc0.x = fmaf(v, t.x, acc0.x); acc0.y = fmaf(v, t.y, acc0.y); acc0.z = fmaf(v, t.z, acc0.z); acc0.w = fmaf(v, t.w, acc0.w);
                    }
                    if (lane + 32 < HV) {
                        const float4 t = hr[lane + 32];
                        acc1.x = fmaf(v, t.x, acc1.x); acc1.y = fmaf(v, t.y, acc1.y); acc1.z = fmaf(v, t.z, acc1.z); acc1.w = fmaf(v, t.w, acc1.w);
                    }
                }
            }
            float4 *out = reinterpret_cast<float4 *>(dst + ((long)mol * N + x) * 4 * H + (long)e * H);
            if (lane < HV) out[lane] = acc0;
            if (lane + 32 < HV) out[lane + 32] = acc1;
            if (!BWD && deg && lane == 0) deg[((long)mol * N + x) * 64 + e] = d;
        }
    }
}

// gate derivatives of one step: g = dL/dh_{t+1};  delta_h = g z (1 - hb^2), delta_z = g (hb - s) z (1 - z) over the z | hb
// slots of Gs[t];  ds = g (1 - z) (stateful steps)
__global__ void __launch_bounds__(256) gate_bwd_kernel(const float *__restrict__ g, float *__restrict__ Gt, const float *__restrict__ s,
                                                       float *__restrict__ ds, long rows, int H) {
    const int HV = H / 4;
    const long n = rows * HV;
    for (long idx = (long)blockIdx.x * 256 + threadIdx.x; idx < n; idx += (long)gridDim.x * 256) {
        const long row = idx / HV;
        const int c = (int)(idx - row * HV) * 4;
        const float4 gv = __ldg(reinterpret_cast<const float4 *>(g + row * H + c));
        float4 *zp = reinterpret_cast<float4 *>(Gt + row * 3 * H + H + c), *hp = reinterpret_cast<float4 *>(Gt + row * 3 * H + 2 * H + c);
        const float4 z = *zp, hb = *hp;
        const float4 sv = s ? __ldg(reinterpret_cast<const float4 *>(s + row * H + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 dz, dh, d;
#define BMP_X3_GATE(f)                                   \
        dz.f = gv.f * (hb.f - sv.f) * z.f * (1.f - z.f); \
        dh.f = gv.f * z.f * (1.f - hb.f * hb.f);         \
        d.f = gv.f * (1.f - z.f);
        BMP_X3_GATE(x) BMP_X3_GATE(y) BMP_X3_GATE(z) BMP_X3_GATE(w)
#undef BMP_X3_GATE
        *zp = dz;
        *hp = dh;
        if (s) *reinterpret_cast<float4 *>(ds + row * H + c) = d;
    }
}

// ------------------------------------------------------------------------------------------------ host side
static int sm_count() {
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    return sms;
}

// the row GEMMs never see molecule boundaries; the per-molecule adjacency products keep an N x H fp32 tile in shared memory
static bool shape_ok(int N, int H, int E) {
    return (H == 64 || H == 128 || H == 256) && E == 4 && N > 0 && N <= BMP_X3_MAX_ATOMS && (size_t)N * H * sizeof(float) <= 160 * 1024;
}
constexpr long MIN_ROWS = 128;      // one full row tile (the tensor-map box)

struct Layout {
    size_t img_bytes, tmp_off, deg_off, mask_off, mini_off, total;
    Layout(long rows, int mb, int N, int H, int T, bool inference) {
        img_bytes = (size_t)image_tiles(H) * WSLOT;
        tmp_off = (size_t)T * img_bytes;
        deg_off = tmp_off + (size_t)rows * 4 * H * sizeof(float);
        mask_off = deg_off + (((size_t)rows * 64 * sizeof(float) + 1023) & ~(size_t)1023);      // flag (256 B) + bit masks (4 KB per molecule at N = 64)
        mini_off = mask_off + 256 + (size_t)mb * 64 * N * ((N + 63) / 64);      // 2 x 4 x N x W words of 8 bytes
        total = mini_off + (inference ? (size_t)rows * 7 * H * sizeof(float) : 0) + 1024;
    }
};

static long long *g_dbg = nullptr;
static int g_dbg_slot = 0;

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// the driver entry point is looked up at run time: the library keeps loading on a machine without a driver
static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

static int launch_gemm(Args &g, cudaStream_t st) {
    g.dbg = g_dbg ? g_dbg + 8 * (g_dbg_slot++) : nullptr;
    EncodeTiledFn enc = encode_tiled();
    if (!enc) { set_error("rowgemm3: cuTensorMapEncodeTiled is not available"); return BMP_ECUDA; }
    for (int j = 0; j < g.njobs; ++j)
        for (int b = 0; b < g.job[j].nblk; ++b) {
            const Job &J = g.job[j];
            const cuuint64_t dims[2] = {(cuuint64_t)64 * J.kt[b], (cuuint64_t)g.rows};
            const cuuint64_t strides[1] = {(cuuint64_t)J.lda[b] * sizeof(float)};
            const cuuint32_t box[2] = {64, 128}, estr[2] = {1, 1};
            const CUresult r = enc(&g.tmap[j][b], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)J.A[b], dims, strides, box, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) { set_error("rowgemm3: cuTensorMapEncodeTiled failed (%d)", (int)r); return BMP_ECUDA; }
        }
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(rowgemm3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        cudaFuncSetAttribute(rowgemm3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
        attr = true;
    }
    const long items = ((g.rows + 127) / 128) * g.njobs;
    const int grid = (int)(items < sm_count() ? items : sm_count());
    if (g.dbg) rowgemm3_kernel<true><<<grid, NT, SMEM_BYTES, st>>>(g);
    else rowgemm3_kernel<false><<<grid, NT, SMEM_BYTES, st>>>(g);
    count_launch();
    return check_launch("rowgemm3_kernel");
}

static bool same_msg_b(const bmp_ggnn_fwd_t *a, int u, int t) { return a->msg_b[u] == a->msg_b[t]; }
// the backward struct carries no message bias: two steps that share W_m share their linear link, hence its bias, in every caller
// of this library; the forward (which packs the images both directions use) compares the pointer
static bool same_msg_b(const bmp_ggnn_bwd_t *, int, int) { return true; }

// step -> image index (steps that share every parameter pointer and the stateful flag share an image)
template <class S>
static void image_plan(const S *a, int *img_of) {
    for (int t = 0; t < a->n_steps; ++t) {
        img_of[t] = t;
        for (int u = 0; u < t; ++u)
            if (a->msg_W[u] == a->msg_W[t] && same_msg_b(a, u, t) && same_gru(a->gru[u], a->gru[t]) &&
                (a->stateful[u] != 0) == (a->stateful[t] != 0)) {
                img_of[t] = img_of[u];
                break;
            }
    }
}

static const float *msg_b_of(const bmp_ggnn_fwd_t *a, int t) { return a->msg_b[t]; }
static const float *msg_b_of(const bmp_ggnn_bwd_t *, int) { return nullptr; }      // the backward jobs do not use the bias tile

template <class S>
static int pack_images(const S *a, uint8_t *ws, const Layout &L, const int *img_of, cudaStream_t st) {
    for (int t = 0; t < a->n_steps; ++t) {
        if (img_of[t] != t) continue;
        PackArgs p;
        p.msg_W = a->msg_W[t];
        p.msg_b = msg_b_of(a, t);
        p.g = a->gru[t];
        p.H = a->hidden;
        p.stateful = a->stateful[t];
        p.img = ws + (size_t)t * L.img_bytes;
        pack_x3_kernel<<<image_tiles(a->hidden), 256, 0, st>>>(p);
        count_launch();
    }
    return check_launch("pack_x3_kernel");
}

static const uint8_t *job_img(const uint8_t *img, int j, int nc, int H) {
    return img + ((size_t)job_tile0(j, H) + (size_t)nc * job_ktiles(j, H)) * WSLOT;
}

}  // namespace x3
}  // namespace bmp

using namespace bmp;
using namespace bmp::x3;

// debug: p = device buffer of 8 x n long long; every rowgemm3 launch after this call fills the next 8-slot record
extern "C" void bmp_debug_set_buffer_x3(void *p) { g_dbg = (long long *)p; g_dbg_slot = 0; }

// ------------------------------------------------------------------------------------------------ gated read-out (forward)
// models/readout/ggnn_readout.py:42-58 (R1) and models/ggnn_att.py:338-346 (R2) in BMP_MODE_F32: the two linears over all atoms are row
// GEMMs on the same split-bf16 kernel (pre-activations to a workspace), the gate product and the sum over a molecule's atoms a
// small kernel.  The backward stays the kernel of readout.cu (it needs h, h0, the weights and g only).
namespace bmp {
namespace x3 {

// W (n_out, ldw) row-major, columns [k0, k0 + 64 kt): k-tiles [nc][kk] of the B operand (n = output column)
__global__ void __launch_bounds__(256) pack_lin_kernel(const float *__restrict__ W, int ldw, int n_out, int k0, int kt, uint8_t *img) {
    const int tile = blockIdx.x, nc = tile / kt, kk = tile % kt, NC = n_out < 128 ? n_out : 128;
    uint8_t *dst = img + (size_t)tile * WSLOT;
    for (int idx = threadIdx.x; idx < NC * 8; idx += 256) {
        const int c8 = idx % 8, n = idx / 8;          // k fastest: consecutive addresses of one weight row
        const float *src = W + (long)(nc * 128 + n) * ldw + k0 + kk * 64 + c8 * 8;
        const float4 a = __ldg(reinterpret_cast<const float4 *>(src)), b = __ldg(reinterpret_cast<const float4 *>(src) + 1);
        const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t h[4], l[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            h[x] = pack_bf16(v[2 * x], v[2 * x + 1]);
            l[x] = pack_bf16(v[2 * x] - __uint_as_float(h[x] << 16), v[2 * x + 1] - __uint_as_float(h[x] & 0xFFFF0000u));
        }
        const uint32_t off = sw128(n, c8 * 8);
        *reinterpret_cast<uint4 *>(dst + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4 *>(dst + PANEL_BYTES + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// g[mol][o] = act_agg( sum_n sigmoid(pi[row][o]) * act(pj[row][o]) * mask[row] )
__global__ void __launch_bounds__(256) readout_reduce_kernel(const float *__restrict__ pi, const float *__restrict__ pj,
                                                             const float *__restrict__ mask, float *__restrict__ g, int mb, int N, int O,
                                                             int act, int act_agg) {
    for (int mol = blockIdx.x; mol < mb; mol += gridDim.x)
        for (int o = threadIdx.x; o < O; o += 256) {
            float s = 0.f;
            for (int n = 0; n < N; ++n) {
                const long row = (long)mol * N + n;
                const float v = sigmoidf_(__ldg(pi + row * O + o)) * act_fwd(act, __ldg(pj + row * O + o));
                s += mask ? v * __ldg(mask + row) : v;
            }
            g[(long)mol * O + o] = act_fwd(act_agg, s);
        }
}

static bool readout_ok(int mb, int N, int H, int O, int variant) {
    return (H == 64 || H == 128 || H == 256) && (O == 64 || O == 128 || O == 256) && (long)mb * N >= MIN_ROWS &&
           (variant == BMP_READOUT_R1 || variant == BMP_READOUT_R2);
}
static size_t readout_img_tiles(int H, int O, bool has_h0, int variant) {
    const int hc = (O + 127) / 128, kb = H / 64;
    const int blk_i = has_h0 ? 2 : 1, blk_j = (has_h0 && variant == BMP_READOUT_R1) ? 2 : 1;
    return (size_t)(blk_i + blk_j) * kb * hc;
}

}  // namespace x3
}  // namespace bmp

// Bytes of workspace the tensor-core fp32 read-out forward needs (weight images + the two pre-activation arrays); 0 = not covered.
extern "C" size_t bmp_readout_x3_workspace_bytes(int mb, int n_atoms, int hidden, int out_dim, int variant, int has_h0) {
    if (!readout_ok(mb, n_atoms, hidden, out_dim, variant)) return 0;
    return readout_img_tiles(hidden, out_dim, has_h0 != 0, variant) * WSLOT + 2 * (size_t)mb * n_atoms * out_dim * sizeof(float) + 4096;
}

bool bmp_readout_x3_usable(const bmp_readout_fwd_t *a) {
    if (a->mode != BMP_MODE_F32 || !a->tc_workspace || !readout_ok(a->mb, a->n_atoms, a->hidden, a->out_dim, a->variant)) return false;
    if (!aligned16({a->b_i, a->b_j})) return false;
    return a->tc_workspace_bytes >= bmp_readout_x3_workspace_bytes(a->mb, a->n_atoms, a->hidden, a->out_dim, a->variant, a->h0 != nullptr);
}

int bmp_readout_forward_x3(const bmp_readout_fwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int H = a->hidden, O = a->out_dim, N = a->n_atoms, NC = O < 128 ? O : 128, hc = (O + 127) / 128, kb = H / 64;
    const long rows = (long)a->mb * N;
    const bool has_h0 = a->h0 != nullptr;
    const int blk[2] = {has_h0 ? 2 : 1, (has_h0 && a->variant == BMP_READOUT_R1) ? 2 : 1};
    const int Kin[2] = {blk[0] * H, blk[1] * H};
    const float *W[2] = {a->W_i, a->W_j}, *bias[2] = {a->b_i, a->b_j};
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 1023) & ~(uintptr_t)1023);
    uint8_t *img[2] = {ws, ws + (size_t)blk[0] * kb * hc * WSLOT};
    float *pre = reinterpret_cast<float *>(ws + readout_img_tiles(H, O, has_h0, a->variant) * WSLOT);
    float *pre_ij[2] = {pre, pre + (size_t)rows * O};
    int rc;
    if (!a->tc_images_ready) {
        for (int w = 0; w < 2; ++w) {
            // image of linear w: per column chunk the k-tiles of its K blocks in consumption order = all kt = blk * kb tiles of the row
            pack_lin_kernel<<<blk[w] * kb * hc, 256, 0, st>>>(W[w], Kin[w], O, 0, blk[w] * kb, img[w]);
            count_launch();
        }
        if ((rc = check_launch("pack_lin_kernel"))) return rc;
    }
    Args ga;
    memset(&ga, 0, sizeof(ga));
    ga.rows = rows; ga.NC = NC;
    int nj = 0;
    for (int nc = 0; nc < hc; ++nc)
        for (int w = 0; w < 2; ++w) {
            Job &J = ga.job[nj++];
            J.nblk = blk[w];
            J.A[0] = a->h; J.A[1] = a->h0; J.lda[0] = J.lda[1] = H; J.kt[0] = J.kt[1] = kb;
            J.wimg = img[w] + (size_t)nc * blk[w] * kb * WSLOT;
            J.epi = EPI_LIN;
            J.bias = bias[w] ? bias[w] + nc * 128 : nullptr;
            J.out0 = pre_ij[w] + nc * 128; J.lo0 = O;
        }
    ga.njobs = nj;
    if ((rc = launch_gemm(ga, st))) return rc;
    const int grid = a->mb < 8 * sm_count() ? a->mb : 8 * sm_count();
    readout_reduce_kernel<<<grid, 256, 0, st>>>(pre_ij[0], pre_ij[1], a->is_real_node, a->g, a->mb, N, O, a->act, a->act_agg);
    count_launch();
    return check_launch("readout_reduce_kernel");
}

// Bytes of workspace the tensor-core fp32 path needs (weight images + per-step temporaries [+ a one-step stash for
// inference]); 0 = shape not covered (the FFMA kernels of ggnn.cu run instead).
extern "C" size_t bmp_ggnn_x3_workspace_bytes(int mb, int n_atoms, int hidden, int n_edge, int n_steps, int inference) {
    if (!shape_ok(n_atoms, hidden, n_edge) || (long)mb * n_atoms < MIN_ROWS || n_steps <= 0 || n_steps > BMP_MAX_STEPS) return 0;
    return Layout((long)mb * n_atoms, mb, n_atoms, hidden, n_steps, inference != 0).total;
}

bool bmp_ggnn_x3_usable(int mb, int N, int H, int E, int T, const void *ws, size_t ws_bytes, const void *state_in, bool inference) {
    if (!ws || state_in || !shape_ok(N, H, E) || (long)mb * N < MIN_ROWS) return false;
    return ws_bytes >= Layout((long)mb * N, mb, N, H, T, inference).total;
}

int bmp_ggnn_forward_x3(const bmp_ggnn_fwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int H = a->hidden, N = a->n_atoms, T = a->n_steps, NC = H < 128 ? H : 128, hc = (H + 127) / 128, kb = H / 64;
    const long rows = (long)a->mb * N;
    const bool inference = !a->Hs;
    if (!inference && (!a->Ms || !a->Gs || !a->RSs)) { set_error("bmp_ggnn_forward: partial stash"); return BMP_EINVAL; }
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 1023) & ~(uintptr_t)1023);
    const Layout L(rows, a->mb, N, H, T, inference);
    int img_of[BMP_MAX_STEPS];
    image_plan(a, img_of);
    int rc;
    if (!a->tc_images_ready && (rc = pack_images(a, ws, L, img_of, st))) return rc;
    float *AH = reinterpret_cast<float *>(ws + L.tmp_off), *deg = reinterpret_cast<float *>(ws + L.deg_off);
    float *mini = reinterpret_cast<float *>(ws + L.mini_off);
    const size_t RH = (size_t)rows * H;
    auto Hs_at = [&](int t) { return inference ? mini + (size_t)(t & 1) * RH : a->Hs + (size_t)t * RH; };
    auto Ms_at = [&](int t) { return inference ? mini + 2 * RH : a->Ms + (size_t)t * RH; };
    auto Gs_at = [&](int t) { return inference ? mini + 3 * RH : a->Gs + (size_t)t * 3 * RH; };
    auto RS_at = [&](int t) { return inference ? mini + 6 * RH : a->RSs + (size_t)t * RH; };

    if (a->atoms) {
        if ((rc = bmp_embed_forward(a->atoms, a->embed_W, Hs_at(0), (int)rows, H, a->n_atom_types, stream))) return rc;
    } else {
        cudaMemcpyAsync(Hs_at(0), a->h_in, RH * sizeof(float), cudaMemcpyDeviceToDevice, st);
    }
    if (a->h0_out) cudaMemcpyAsync(a->h0_out, Hs_at(0), RH * sizeof(float), cudaMemcpyDeviceToDevice, st);

    cudaMemsetAsync(deg, 0, (size_t)rows * 64 * sizeof(float), st);
    int *flag = reinterpret_cast<int *>(ws + L.mask_off);
    unsigned long long *masks = reinterpret_cast<unsigned long long *>(ws + L.mask_off + 256);
    const size_t agg_smem = (size_t)N * H * sizeof(float);
    cudaFuncSetAttribute(agg_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)agg_smem);
    const int agg_grid = a->mb < 8 * sm_count() ? a->mb : 8 * sm_count();
    cudaMemsetAsync(flag, 0, 256, st);
    adj_mask_kernel<<<agg_grid, 256, (size_t)32 * N * ((N + 63) / 64), st>>>(a->adj, masks, flag, a->mb, N);
    count_launch();
    if ((rc = check_launch("adj_mask_kernel"))) return rc;
    for (int t = 0; t < T; ++t) {
        const bool stf = a->stateful[t] != 0;
        const uint8_t *img = ws + (size_t)img_of[t] * L.img_bytes;
        const bmp_gru_t &G = a->gru[t];
        float *h = Hs_at(t), *hn = Hs_at(t + 1), *m = Ms_at(t), *g = Gs_at(t), *rs = RS_at(t);
        agg_kernel<false><<<agg_grid, 256, agg_smem, st>>>(masks, flag, a->adj, h, AH, t == 0 ? deg : nullptr, a->mb, N, H, nullptr);
        count_launch();
        if ((rc = check_launch("agg_kernel"))) return rc;
        Args ga;
        // ---- message
        memset(&ga, 0, sizeof(ga));
        ga.rows = rows; ga.NC = NC; ga.njobs = hc;
        for (int nc = 0; nc < hc; ++nc) {
            Job &J = ga.job[nc];
            J.nblk = 5;
            for (int e = 0; e < 4; ++e) { J.A[e] = AH + (size_t)e * H; J.lda[e] = 4 * H; J.kt[e] = kb; }
            J.A[4] = deg; J.lda[4] = 64; J.kt[4] = 1;
            J.wimg = job_img(img, EPI_MSG, nc, H);
            J.epi = EPI_MSG;
            J.out0 = m + nc * 128; J.lo0 = H;
        }
        if ((rc = launch_gemm(ga, st))) return rc;
        // ---- reset (stateful) and update gates
        memset(&ga, 0, sizeof(ga));
        ga.rows = rows; ga.NC = NC;
        int nj = 0;
        for (int nc = 0; nc < hc; ++nc) {
            if (stf) {
                Job &J = ga.job[nj++];
                J.nblk = 2;
                J.A[0] = h; J.A[1] = m; J.lda[0] = J.lda[1] = H; J.kt[0] = J.kt[1] = kb;
                J.wimg = job_img(img, EPI_R, nc, H);
                J.epi = EPI_R;
                J.bias = G.b_Wr + nc * 128; J.bias2 = G.b_Ur + nc * 128;
                J.in0 = h + nc * 128; J.li0 = H;
                J.out0 = g + nc * 128; J.lo0 = 3 * H;
                J.out1 = rs + nc * 128; J.lo1 = H;
            }
            Job &J = ga.job[nj++];
            J.nblk = 2;
            J.A[0] = h; J.A[1] = m; J.lda[0] = J.lda[1] = H; J.kt[0] = J.kt[1] = kb;
            J.wimg = job_img(img, EPI_Z, nc, H);
            J.epi = EPI_Z;
            J.bias = G.b_Wz + nc * 128; J.bias2 = stf ? G.b_Uz + nc * 128 : nullptr;
            J.out0 = g + H + nc * 128; J.lo0 = 3 * H;
            if (!stf) { J.out1 = g + nc * 128; J.lo1 = 3 * H; J.out2 = rs + nc * 128; J.lo2 = H; }
        }
        ga.njobs = nj;
        if ((rc = launch_gemm(ga, st))) return rc;
        // ---- candidate and the new state
        memset(&ga, 0, sizeof(ga));
        ga.rows = rows; ga.NC = NC; ga.njobs = hc;
        for (int nc = 0; nc < hc; ++nc) {
            Job &J = ga.job[nc];
            J.nblk = stf ? 3 : 2;
            J.A[0] = h; J.A[1] = m; J.A[2] = rs; J.lda[0] = J.lda[1] = J.lda[2] = H; J.kt[0] = J.kt[1] = J.kt[2] = kb;
            J.wimg = job_img(img, EPI_HB, nc, H);
            J.epi = EPI_HB;
            J.bias = G.b_W + nc * 128; J.bias2 = stf ? G.b_U + nc * 128 : nullptr;
            J.in0 = g + H + nc * 128; J.li0 = 3 * H;
            J.in1 = stf ? h + nc * 128 : nullptr; J.li1 = H;
            J.out0 = g + 2 * H + nc * 128; J.lo0 = 3 * H;
            J.out1 = hn + nc * 128; J.lo1 = H;
            if (t == T - 1 && a->h_out) { J.out2 = a->h_out + nc * 128; J.lo2 = H; }
        }
        if ((rc = launch_gemm(ga, st))) return rc;
    }
    return BMP_OK;
}

// data part of the backward: Gs <- delta_r | delta_z | delta_h, Ps <- A_e^T dm, dHs[0] <- total gradient w.r.t. h_0
int bmp_ggnn_backward_x3(const bmp_ggnn_bwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int H = a->hidden, N = a->n_atoms, T = a->n_steps, NC = H < 128 ? H : 128, hc = (H + 127) / 128, kb = H / 64;
    const long rows = (long)a->mb * N;
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 1023) & ~(uintptr_t)1023);
    const Layout L(rows, a->mb, N, H, T, false);
    int img_of[BMP_MAX_STEPS];
    image_plan(a, img_of);
    int rc;
    if (!a->tc_images_ready && (rc = pack_images(a, ws, L, img_of, st))) return rc;
    const size_t RH = (size_t)rows * H;
    float *tmp = reinterpret_cast<float *>(ws + L.tmp_off);
    float *ds = tmp, *dhx = tmp + RH, *dm = tmp + 2 * RH;
    int *flag = reinterpret_cast<int *>(ws + L.mask_off);
    unsigned long long *masks = reinterpret_cast<unsigned long long *>(ws + L.mask_off + 256);
    const size_t agg_smem = (size_t)N * H * sizeof(float);
    cudaFuncSetAttribute(agg_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)agg_smem);
    const int agg_grid = a->mb < 8 * sm_count() ? a->mb : 8 * sm_count();
    cudaMemsetAsync(flag, 0, 256, st);        // the masks are rebuilt: the workspace need not be the forward's
    adj_mask_kernel<<<agg_grid, 256, (size_t)32 * N * ((N + 63) / 64), st>>>(a->adj, masks, flag, a->mb, N);
    count_launch();
    if ((rc = check_launch("adj_mask_kernel"))) return rc;
    for (int t = T - 1; t >= 0; --t) {
        const bool stf = a->stateful[t] != 0;
        const uint8_t *img = ws + (size_t)img_of[t] * L.img_bytes;
        float *Gt = a->Gs + (size_t)t * 3 * RH;
        const float *s = a->Hs + (size_t)t * RH;
        const float *g = a->dHs + (size_t)(t + 1) * RH;
        float *gout = a->dHs + (size_t)t * RH;
        const long nvec = rows * (H / 4);
        const int pgrid = (int)((nvec + 255) / 256 < 16L * sm_count() ? (nvec + 255) / 256 : 16L * sm_count());
        gate_bwd_kernel<<<pgrid, 256, 0, st>>>(g, Gt, stf ? s : nullptr, ds, rows, H);
        count_launch();
        if ((rc = check_launch("gate_bwd_kernel"))) return rc;
        Args ga;
        if (stf) {
            memset(&ga, 0, sizeof(ga));
            ga.rows = rows; ga.NC = NC; ga.njobs = hc;
            for (int nc = 0; nc < hc; ++nc) {
                Job &J = ga.job[nc];
                J.nblk = 1;
                J.A[0] = Gt + 2 * H; J.lda[0] = 3 * H; J.kt[0] = kb;
                J.wimg = job_img(img, EPI_Q, nc, H);
                J.epi = EPI_Q;
                J.in0 = s + nc * 128; J.li0 = H;
                J.in1 = Gt + nc * 128; J.li1 = 3 * H;
                J.in2 = ds + nc * 128; J.li2 = H;
                J.out0 = Gt + nc * 128; J.lo0 = 3 * H;
                J.out1 = ds + nc * 128; J.lo1 = H;
            }
            if ((rc = launch_gemm(ga, st))) return rc;
        }
        // ---- dh_x (+ ds) and dm
        memset(&ga, 0, sizeof(ga));
        ga.rows = rows; ga.NC = NC;
        int nj = 0;
        for (int nc = 0; nc < hc; ++nc)
            for (int which = 0; which < 2; ++which) {
                Job &J = ga.job[nj++];
                J.nblk = stf ? 3 : 2;
                J.A[0] = Gt + H; J.A[1] = Gt + 2 * H; J.A[2] = Gt;
                J.lda[0] = J.lda[1] = J.lda[2] = 3 * H; J.kt[0] = J.kt[1] = J.kt[2] = kb;
                J.wimg = job_img(img, which ? EPI_DM : EPI_DHX, nc, H);
                J.epi = which ? EPI_DM : EPI_DHX;
                if (!which && stf) { J.in0 = ds + nc * 128; J.li0 = H; }
                J.out0 = (which ? dm : dhx) + nc * 128; J.lo0 = H;
            }
        ga.njobs = nj;
        if ((rc = launch_gemm(ga, st))) return rc;
        agg_kernel<true><<<agg_grid, 256, agg_smem, st>>>(masks, flag, a->adj, dm, a->Ps + (size_t)t * 4 * RH, nullptr, a->mb, N, H, nullptr);
        count_launch();
        if ((rc = check_launch("agg_kernel"))) return rc;
        // ---- dHs[t] += dh_x + sum_e P_e W_e
        memset(&ga, 0, sizeof(ga));
        ga.rows = rows; ga.NC = NC; ga.njobs = hc;
        for (int nc = 0; nc < hc; ++nc) {
            Job &J = ga.job[nc];
            J.nblk = 4;
            for (int e = 0; e < 4; ++e) { J.A[e] = a->Ps + (size_t)t * 4 * RH + (size_t)e * H; J.lda[e] = 4 * H; J.kt[e] = kb; }
            J.wimg = job_img(img, EPI_DHMSG, nc, H);
            J.epi = EPI_DHMSG;
            J.in0 = dhx + nc * 128; J.li0 = H;
            J.in1 = gout + nc * 128; J.li1 = H;
            J.out0 = gout + nc * 128; J.lo0 = H;
        }
        if ((rc = launch_gemm(ga, st))) return rc;
    }
    return BMP_OK;
}

// ------------------------------------------------------------------------------------------------ RelGCN encoder (BMP_MODE_F32, 65..256 atoms)
// models/relgcn.py:61-73 and models/update/relgcn_update.py:24-44 for molecules the one-CTA-per-molecule FFMA kernels of relgcn.cu
// cannot hold.  A layer is the GGNN message with a self term and no gate:
//   forward layer l     agg        AH_e = A_e h_l, deg_e = A_e 1                       (rescale_adj: A_e[i][j] times cs[j])
//                       rowgemm3   h_{l+1} = act([h_l | AH_0 .. AH_3 | deg] [W_s | W_0 .. W_3 | b_e]^T + b_s)
//   backward layer l    delta      d = g * act'(h_{l+1})                               (pointwise)
//                       agg        P_e = A_e^T d
//                       rowgemm3   g <- [d | P_0 .. P_3] [W_s | W_0 .. W_3]             (the transposed packing)
//                       dW_s += d^T h_l, db_s += sum d, dW_e += P_e^T h_l, db_e += sum P_e (bmp_wgrad_tc3 over the caller's Hs)
// Every layer runs at one padded width Cp (the widest channel count rounded up to 64, 128 or 256): padded channels meet zero
// weights and zero bias, so they stay exactly 0 under identity and tanh.  The caller's buffers (Hs, h_out, d_h0) keep the
// unpadded widths of ch[]; batches of fewer than 128 rows run the GEMMs over one zero-padded 128-row tile.
namespace bmp {
namespace x3 {

static int relgcn_cpad(int cmax) { return cmax <= 64 ? 64 : (cmax <= 128 ? 128 : (cmax <= 256 ? 256 : 0)); }
static bool relgcn_shape_ok(int mb, int N, int cmax, int L) {
    const int Cp = relgcn_cpad(cmax);
    return mb > 0 && N > BMP_MAX_ATOMS && N <= BMP_X3_MAX_ATOMS && cmax > 0 && Cp > 0 && L > 0 && L <= BMP_MAX_STEPS &&
           (size_t)N * Cp * sizeof(float) <= 160 * 1024;
}
__host__ __device__ inline int relgcn_ftiles(int Cp) { return ((Cp + 127) / 128) * (5 * (Cp / 64) + 1); }   // forward job: h, AH_0..3, deg (bias tile)
__host__ __device__ inline int relgcn_btiles(int Cp) { return ((Cp + 127) / 128) * (5 * (Cp / 64)); }       // backward job: d, P_0..3

struct RLayout {
    size_t layer_img, bias_off, cs_off, mask_off, deg_off, ah_off, x_off, total;
    long rg;                                   // GEMM rows: at least one full 128-row tile
    RLayout(int mb, int N, int Cp, int L) {
        auto up = [](size_t x) { return (x + 1023) & ~(size_t)1023; };
        const long rows = (long)mb * N;
        rg = rows > MIN_ROWS ? rows : MIN_ROWS;
        layer_img = (size_t)(relgcn_ftiles(Cp) + relgcn_btiles(Cp)) * WSLOT;
        bias_off = (size_t)L * layer_img;
        cs_off = up(bias_off + (size_t)L * Cp * sizeof(float));
        mask_off = up(cs_off + (size_t)rows * sizeof(float));
        deg_off = up(mask_off + 256 + (size_t)mb * 64 * N * ((N + 63) / 64));
        ah_off = up(deg_off + (size_t)rg * 64 * sizeof(float));
        x_off = up(ah_off + (size_t)rg * 4 * Cp * sizeof(float));
        total = x_off + 2 * (size_t)rg * Cp * sizeof(float) + 1024;
    }
};

struct PackRelgcn {
    const float *Ws, *bs, *We, *be;       // (Cout, Cin), (Cout), (Cout * 4, Cin) rows c * 4 + e, (Cout * 4)
    int Cin, Cout, Cp, first;             // first: tile of blockIdx.x 0 (the backward packs only its own tiles)
    uint8_t *img;
    float *bias;                          // (Cp) b_s zero-padded
};

// One layer's image: the forward job's k-tiles per 128-column chunk (h, AH_0 .. AH_3, the bias tile of deg), then the backward job's
// (d, P_0 .. P_3).  B element (n = output column, k = column inside K-block b):
//   forward   W_s[n][k] ; W_e[n][k] = We[(n*4 + e)*Cin + k] ; b_e[n*4 + k] (k < 4)
//   backward  W_s[k][n] ; W_e[k][n]
__global__ void __launch_bounds__(256) pack_relgcn_kernel(const PackRelgcn p) {
    const int Cp = p.Cp, kb = Cp / 64, hc = (Cp + 127) / 128, NC = Cp < 128 ? Cp : 128;
    const int tile = blockIdx.x + p.first;
    const bool bwd = tile >= relgcn_ftiles(Cp);
    const int per = 5 * kb + (bwd ? 0 : 1), local = bwd ? tile - relgcn_ftiles(Cp) : tile;
    const int nc = local / per, kk = local % per, b = kk / kb, kbase = (kk % kb) * 64;
    (void)hc;
    auto val = [&](int n, int k) -> float {
        if (!bwd) {
            if (n >= p.Cout) return 0.f;
            if (b == 5) return k < 4 && p.be ? p.be[(long)n * 4 + k] : 0.f;
            if (k >= p.Cin) return 0.f;
            return b == 0 ? p.Ws[(long)n * p.Cin + k] : p.We[((long)n * 4 + b - 1) * p.Cin + k];
        }
        if (n >= p.Cin || k >= p.Cout) return 0.f;
        return b == 0 ? p.Ws[(long)k * p.Cin + n] : p.We[((long)k * 4 + b - 1) * p.Cin + n];
    };
    uint8_t *dst = p.img + (size_t)tile * WSLOT;
    for (int idx = threadIdx.x; idx < NC * 8; idx += 256) {
        const int n = idx % NC, c8 = idx / NC;
        float v[8];
#pragma unroll
        for (int x = 0; x < 8; ++x) v[x] = val(nc * 128 + n, kbase + c8 * 8 + x);
        uint32_t h[4], l[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            h[x] = pack_bf16(v[2 * x], v[2 * x + 1]);
            l[x] = pack_bf16(v[2 * x] - __uint_as_float(h[x] << 16), v[2 * x + 1] - __uint_as_float(h[x] & 0xFFFF0000u));
        }
        const uint32_t off = sw128(n, c8 * 8);
        *reinterpret_cast<uint4 *>(dst + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4 *>(dst + PANEL_BYTES + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    if (tile == 0)
        for (int i = threadIdx.x; i < Cp; i += 256) p.bias[i] = i < p.Cout && p.bs ? p.bs[i] : 0.f;
}

// x[r][c] = h_0[r][c] for c < C0, 0 for the padded channels; h_0 = embed_W[clamp(atoms[r])] or h_in[r]
__global__ void __launch_bounds__(256) relgcn_input_kernel(const int32_t *__restrict__ atoms, const float *__restrict__ embed_W, int n_types,
                                                           const float *__restrict__ h_in, float *__restrict__ x, long rows, int C0, int Cp) {
    for (long idx = (long)blockIdx.x * 256 + threadIdx.x; idx < rows * Cp; idx += (long)gridDim.x * 256) {
        const long r = idx / Cp;
        const int c = (int)(idx - r * Cp);
        float v = 0.f;
        if (c < C0) {
            if (atoms) {
                int id = atoms[r];
                id = id < 0 ? 0 : (id >= n_types ? n_types - 1 : id);
                v = __ldg(embed_W + (long)id * C0 + c);
            } else {
                v = __ldg(h_in + r * C0 + c);
            }
        }
        x[idx] = v;
    }
}

// d[r][c] = g[r][c] * act'(y[r][c]) for c < C (y = the layer output, row stride C; g row stride ldg), 0 for the padded channels
__global__ void __launch_bounds__(256) relgcn_delta_kernel(const float *__restrict__ g, int ldg, const float *__restrict__ y,
                                                           float *__restrict__ d, long rows, int C, int Cp, int act) {
    const int CV = Cp / 4;
    for (long idx = (long)blockIdx.x * 256 + threadIdx.x; idx < rows * CV; idx += (long)gridDim.x * 256) {
        const long r = idx / CV;
        const int c = (int)(idx - r * CV) * 4;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < C) {
            const float4 gv = __ldg(reinterpret_cast<const float4 *>(g + r * ldg + c));
            const float4 yv = __ldg(reinterpret_cast<const float4 *>(y + r * C + c));
            o = make_float4(gv.x * act_bwd(act, yv.x, yv.x), gv.y * act_bwd(act, yv.y, yv.y), gv.z * act_bwd(act, yv.z, yv.z),
                            gv.w * act_bwd(act, yv.w, yv.w));
        }
        *reinterpret_cast<float4 *>(d + r * Cp + c) = o;
    }
}

// cs[mol][j] = 1 / sum_{e,i} A[mol][e][i][j] (1 where the sum is 0)
__global__ void __launch_bounds__(256) relgcn_colscale_kernel(const float *__restrict__ adj, float *__restrict__ cs, int mb, int N) {
    __shared__ float part[4][64], inv[BMP_X3_MAX_ATOMS];
    for (int mol = blockIdx.x; mol < mb; mol += gridDim.x) {
        column_inverse_degree(adj + (long)mol * 4 * N * N, 4, N, part, inv);
        for (int j = threadIdx.x; j < N; j += 256) cs[(long)mol * N + j] = inv[j];
    }
}

static int relgcn_cmax(const int *ch, int L) {
    int c = 0;
    for (int l = 0; l <= L; ++l) c = ch[l] > c ? ch[l] : c;
    return c;
}

// (rows, C) row-major <- the first C columns of (rows, Cp)
static int copy_cols(float *dst, int C, const float *src, int Cp, long rows, cudaStream_t st) {
    if (cudaMemcpy2DAsync(dst, (size_t)C * sizeof(float), src, (size_t)Cp * sizeof(float), (size_t)C * sizeof(float), (size_t)rows,
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        set_error("relgcn x3: cudaMemcpy2DAsync failed");
        return BMP_ECUDA;
    }
    return BMP_OK;
}

// the adjacency side shared by forward and backward: bit masks + general-weight flag, and the column scales of rescale_adj
static int relgcn_adjacency(const float *adj, int mb, int N, bool scale, uint8_t *ws, const RLayout &R, cudaStream_t st) {
    int *flag = reinterpret_cast<int *>(ws + R.mask_off);
    const int grid = mb < 8 * sm_count() ? mb : 8 * sm_count();
    cudaMemsetAsync(flag, 0, 256, st);
    adj_mask_kernel<<<grid, 256, (size_t)32 * N * ((N + 63) / 64), st>>>(adj, reinterpret_cast<unsigned long long *>(ws + R.mask_off + 256),
                                                                         flag, mb, N);
    count_launch();
    int rc;
    if ((rc = check_launch("adj_mask_kernel"))) return rc;
    if (scale) {
        relgcn_colscale_kernel<<<grid, 256, 0, st>>>(adj, reinterpret_cast<float *>(ws + R.cs_off), mb, N);
        count_launch();
        if ((rc = check_launch("relgcn_colscale_kernel"))) return rc;
    }
    return BMP_OK;
}

static int relgcn_pack(const float *const *Ws, const float *const *bs, const float *const *We, const float *const *be, const int *ch,
                       int L, int Cp, bool backward, uint8_t *ws, const RLayout &R, cudaStream_t st) {
    for (int l = 0; l < L; ++l) {
        PackRelgcn p;
        p.Ws = Ws[l]; p.bs = bs ? bs[l] : nullptr; p.We = We[l]; p.be = be ? be[l] : nullptr;
        p.Cin = ch[l]; p.Cout = ch[l + 1]; p.Cp = Cp;
        p.first = backward ? relgcn_ftiles(Cp) : 0;
        p.img = ws + (size_t)l * R.layer_img;
        p.bias = reinterpret_cast<float *>(ws + R.bias_off) + (size_t)l * Cp;
        pack_relgcn_kernel<<<backward ? relgcn_btiles(Cp) : relgcn_ftiles(Cp), 256, 0, st>>>(p);
        count_launch();
    }
    return check_launch("pack_relgcn_kernel");
}

static int pointwise_grid(long n) {
    const long g = (n + 255) / 256;
    return (int)(g < 16L * sm_count() ? g : 16L * sm_count());
}

}  // namespace x3
}  // namespace bmp

// Bytes of workspace the RelGCN encoder needs on the tensor-core path (weight images, adjacency masks, per-layer temporaries at the
// padded width); 0 = shape not covered.  The size is the same for training and inference.
extern "C" size_t bmp_relgcn_x3_workspace_bytes(int mb, int n_atoms, int ch_max, int n_layers, int inference) {
    (void)inference;
    if (!relgcn_shape_ok(mb, n_atoms, ch_max, n_layers)) return 0;
    return RLayout(mb, n_atoms, relgcn_cpad(ch_max), n_layers).total;
}

// "" when the call can take the tensor-core path, else why not (n_atoms and the channel count named)
const char *bmp_relgcn_x3_refusal(int mb, int N, int E, int L, const int *ch, int act, const void *ws, size_t ws_bytes) {
    static thread_local char why[256];
    const int cmax = L > 0 && L <= BMP_MAX_STEPS ? relgcn_cmax(ch, L) : 0;
    if (!relgcn_shape_ok(mb, N, cmax, L) || E != 4) {
        snprintf(why, sizeof(why), "n_atoms=%d with %d channels and %d bond types: above %d atoms only 4 bond types, n_atoms <= %d and "
                 "n_atoms * channels (rounded up to 64/128/256) * 4 bytes <= 160 KB are covered", N, cmax, E, BMP_MAX_ATOMS, BMP_X3_MAX_ATOMS);
        return why;
    }
    if (act != BMP_ACT_IDENTITY && act != BMP_ACT_TANH) {
        snprintf(why, sizeof(why), "n_atoms=%d: above %d atoms the activation must be identity or tanh", N, BMP_MAX_ATOMS);
        return why;
    }
    const size_t need = RLayout(mb, N, relgcn_cpad(cmax), L).total;
    if (!ws || ws_bytes < need) {
        snprintf(why, sizeof(why), "n_atoms=%d (> %d) needs tc_workspace of bmp_relgcn_x3_workspace_bytes() = %zu bytes (got %zu)", N,
                 BMP_MAX_ATOMS, need, ws ? ws_bytes : (size_t)0);
        return why;
    }
    return "";
}

int bmp_relgcn_forward_x3(const bmp_relgcn_fwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int N = a->n_atoms, L = a->n_layers, Cp = relgcn_cpad(relgcn_cmax(a->ch, L)), kb = Cp / 64, hc = (Cp + 127) / 128;
    const long rows = (long)a->mb * N;
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 1023) & ~(uintptr_t)1023);
    const RLayout R(a->mb, N, Cp, L);
    const long rg = R.rg;
    int rc;
    if ((rc = relgcn_pack(a->self_W, a->self_b, a->edge_W, a->edge_b, a->ch, L, Cp, false, ws, R, st))) return rc;
    if ((rc = relgcn_adjacency(a->adj, a->mb, N, a->scale_adj != 0, ws, R, st))) return rc;
    float *deg = reinterpret_cast<float *>(ws + R.deg_off), *AH = reinterpret_cast<float *>(ws + R.ah_off);
    float *X[2] = {reinterpret_cast<float *>(ws + R.x_off), reinterpret_cast<float *>(ws + R.x_off) + (size_t)rg * Cp};
    cudaMemsetAsync(deg, 0, (size_t)rg * 64 * sizeof(float), st);
    if (rg > rows) {       // rows of the padded tile: zero inputs (their outputs are never read)
        cudaMemsetAsync(X[0] + (size_t)rows * Cp, 0, (size_t)(rg - rows) * Cp * sizeof(float), st);
        cudaMemsetAsync(AH + (size_t)rows * 4 * Cp, 0, (size_t)(rg - rows) * 4 * Cp * sizeof(float), st);
    }
    relgcn_input_kernel<<<pointwise_grid(rows * Cp), 256, 0, st>>>(a->atoms, a->embed_W, a->n_atom_types, a->h_in, X[0], rows, a->ch[0], Cp);
    count_launch();
    if ((rc = check_launch("relgcn_input_kernel"))) return rc;
    if (a->Hs && (rc = copy_cols(a->Hs, a->ch[0], X[0], Cp, rows, st))) return rc;
    const size_t agg_smem = (size_t)N * Cp * sizeof(float);
    cudaFuncSetAttribute(agg_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)agg_smem);
    const int agg_grid = a->mb < 8 * sm_count() ? a->mb : 8 * sm_count();
    const int *flag = reinterpret_cast<const int *>(ws + R.mask_off);
    const unsigned long long *masks = reinterpret_cast<const unsigned long long *>(ws + R.mask_off + 256);
    const float *cs = a->scale_adj ? reinterpret_cast<const float *>(ws + R.cs_off) : nullptr;
    size_t hs_off = (size_t)rows * a->ch[0];
    for (int l = 0; l < L; ++l) {
        float *h = X[l & 1], *hn = X[(l + 1) & 1];
        agg_kernel<false><<<agg_grid, 256, agg_smem, st>>>(masks, flag, a->adj, h, AH, l == 0 ? deg : nullptr, a->mb, N, Cp, cs);
        count_launch();
        if ((rc = check_launch("agg_kernel"))) return rc;
        const uint8_t *img = ws + (size_t)l * R.layer_img;
        const float *bias = reinterpret_cast<const float *>(ws + R.bias_off) + (size_t)l * Cp;
        Args ga;
        memset(&ga, 0, sizeof(ga));
        ga.rows = rg; ga.NC = Cp < 128 ? Cp : 128; ga.njobs = hc;
        for (int nc = 0; nc < hc; ++nc) {
            Job &J = ga.job[nc];
            J.nblk = 6;
            J.A[0] = h; J.lda[0] = Cp; J.kt[0] = kb;
            for (int e = 0; e < 4; ++e) { J.A[1 + e] = AH + (size_t)e * Cp; J.lda[1 + e] = 4 * Cp; J.kt[1 + e] = kb; }
            J.A[5] = deg; J.lda[5] = 64; J.kt[5] = 1;
            J.wimg = img + (size_t)nc * (5 * kb + 1) * WSLOT;
            J.epi = a->act == BMP_ACT_TANH ? EPI_TANH : EPI_LIN;
            J.bias = bias + nc * 128;
            J.out0 = hn + nc * 128; J.lo0 = Cp;
        }
        if ((rc = launch_gemm(ga, st))) return rc;
        const int Cout = a->ch[l + 1];
        if (a->Hs && (rc = copy_cols(a->Hs + hs_off, Cout, hn, Cp, rows, st))) return rc;
        if (l == L - 1 && a->h_out && (rc = copy_cols(a->h_out, Cout, hn, Cp, rows, st))) return rc;
        hs_off += (size_t)rows * Cout;
    }
    return BMP_OK;
}

int bmp_relgcn_backward_x3(const bmp_relgcn_bwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int N = a->n_atoms, L = a->n_layers, E = a->n_edge, Cp = relgcn_cpad(relgcn_cmax(a->ch, L)), kb = Cp / 64, hc = (Cp + 127) / 128;
    const long rows = (long)a->mb * N;
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 1023) & ~(uintptr_t)1023);
    const RLayout R(a->mb, N, Cp, L);
    const long rg = R.rg;
    int rc;
    if ((rc = relgcn_pack(a->self_W, nullptr, a->edge_W, nullptr, a->ch, L, Cp, true, ws, R, st))) return rc;
    if ((rc = relgcn_adjacency(a->adj, a->mb, N, a->scale_adj != 0, ws, R, st))) return rc;
    float *P = reinterpret_cast<float *>(ws + R.ah_off);
    float *D = reinterpret_cast<float *>(ws + R.x_off), *G = D + (size_t)rg * Cp;     // delta, gradient w.r.t. the layer input
    if (rg > rows) {
        cudaMemsetAsync(D + (size_t)rows * Cp, 0, (size_t)(rg - rows) * Cp * sizeof(float), st);
        cudaMemsetAsync(P + (size_t)rows * 4 * Cp, 0, (size_t)(rg - rows) * 4 * Cp * sizeof(float), st);
    }
    const size_t agg_smem = (size_t)N * Cp * sizeof(float);
    cudaFuncSetAttribute(agg_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)agg_smem);
    const int agg_grid = a->mb < 8 * sm_count() ? a->mb : 8 * sm_count();
    const int *flag = reinterpret_cast<const int *>(ws + R.mask_off);
    const unsigned long long *masks = reinterpret_cast<const unsigned long long *>(ws + R.mask_off + 256);
    const float *cs = a->scale_adj ? reinterpret_cast<const float *>(ws + R.cs_off) : nullptr;
    size_t hs_off[BMP_MAX_STEPS + 2];
    hs_off[0] = 0;
    for (int l = 0; l < L; ++l) hs_off[l + 1] = hs_off[l] + (size_t)rows * a->ch[l];
    // C (Cout, Cin; ldc) += A[:, :Cout]^T h_l, dbias += column sums of A[:, :Cout]
    auto WG = [&](const float *A_, int lda, const float *Hl, int Cin, int Cout, float *C_, int ldc, float *db, int dbs) -> int {
        if (C_ && (Cin == 64 || Cin == 128 || Cin == 256)) return bmp_wgrad_tc3(A_, lda, Hl, Cin, C_, ldc, rows, Cout, Cin, db, dbs, stream);
        int e_ = C_ ? bmp_wgrad(A_, lda, Hl, Cin, C_, ldc, rows, Cout, Cin, stream) : BMP_OK;
        if (!e_ && db) e_ = bmp_colsum(A_, lda, db, dbs, rows, Cout, stream);
        return e_;
    };
    for (int l = L - 1; l >= 0; --l) {
        const int Cin = a->ch[l], Cout = a->ch[l + 1];
        const float *g = l == L - 1 ? a->d_h_out : G;
        relgcn_delta_kernel<<<pointwise_grid(rows * (Cp / 4)), 256, 0, st>>>(g, l == L - 1 ? Cout : Cp, a->Hs + hs_off[l + 1], D, rows, Cout,
                                                                             Cp, a->act);
        count_launch();
        if ((rc = check_launch("relgcn_delta_kernel"))) return rc;
        agg_kernel<true><<<agg_grid, 256, agg_smem, st>>>(masks, flag, a->adj, D, P, nullptr, a->mb, N, Cp, cs);
        count_launch();
        if ((rc = check_launch("agg_kernel"))) return rc;
        const float *Hl = a->Hs + hs_off[l];
        if ((rc = WG(D, Cp, Hl, Cin, Cout, a->d_self_W[l], Cin, a->d_self_b[l], 1))) return rc;
        for (int e = 0; e < E; ++e)
            if ((rc = WG(P + (size_t)e * Cp, 4 * Cp, Hl, Cin, Cout, a->d_edge_W[l] ? a->d_edge_W[l] + (size_t)e * Cin : nullptr, E * Cin,
                         a->d_edge_b[l] ? a->d_edge_b[l] + e : nullptr, E)))
                return rc;
        if (l == 0 && !a->d_h0) break;
        const uint8_t *img = ws + (size_t)l * R.layer_img + (size_t)relgcn_ftiles(Cp) * WSLOT;
        Args ga;
        memset(&ga, 0, sizeof(ga));
        ga.rows = rg; ga.NC = Cp < 128 ? Cp : 128; ga.njobs = hc;
        for (int nc = 0; nc < hc; ++nc) {
            Job &J = ga.job[nc];
            J.nblk = 5;
            J.A[0] = D; J.lda[0] = Cp; J.kt[0] = kb;
            for (int e = 0; e < 4; ++e) { J.A[1 + e] = P + (size_t)e * Cp; J.lda[1 + e] = 4 * Cp; J.kt[1 + e] = kb; }
            J.wimg = img + (size_t)nc * 5 * kb * WSLOT;
            J.epi = EPI_LIN;
            J.out0 = G + nc * 128; J.lo0 = Cp;
        }
        if ((rc = launch_gemm(ga, st))) return rc;
        if (l == 0 && (rc = copy_cols(a->d_h0, Cin, G, Cp, rows, st))) return rc;
    }
    return BMP_OK;
}
