// ggnn_tc_bwd.cu -- backward (data part) of the fused GGNN encoder on tcgen05 (BMP_MODE_BF16).
//
// Mirror of ggnn_tc.cu: persistent CTA per SM, a tile = two padded molecules = 128 rows, steps walked in
// reverse over the forward's bf16 panel stash.  The running gradient dL/dh_{t+1} lives in fp32 registers of the
// epilogue threads; per step (SURVEY.md Appendix B, state == step input so U_r/U_z fold into W_r/W_z):
//   phase A   dz, dhbar -> delta_z, delta_h (bf16 operand panels, dumped to the stash for the wgrad contractions)
//   MMA-q     q = delta_h U                      -> phase B: delta_r = q*s*r(1-r), ds += q*r
//   MMA-dx    [dh_x | dm] = [delta_r|delta_z|delta_h] [W_r+U_r ; W_z+U_z ; W]       K = 3H, N = 2H
//   MMA-P     P[(e,j), c] = sum_i A_e[i,j] dm[i,c]   per (molecule, bond-type pair); A read MN-major
//   MMA-dh    dh_x += Pcat Wcat                       K = 4H
//   phase E   dh_t = dh_x + ds + external dHs[t]
// Parameter gradients are C += A^T B contractions streamed from the stash panels (bmp_wgrad_panels_multi).
#include "tc_common.cuh"

namespace bmp {
namespace tcb {
using namespace tc;

template <int H>
struct Cfg {
    static constexpr int KP = H / 64;
    static constexpr int TILE_BYTES = H * 128;
    static constexpr int STAGES = 4;
    static constexpr int TILES_STATEFUL = 11 * KP;     // q: KP, dx: 6KP, dh: 4KP
    static constexpr int TILES_STATELESS = 8 * KP;     // dx (z, hbar): 4KP, dh: 4KP
    static constexpr int TMEM_COLS = 4 * H;
    static constexpr int OFF_D = 0;                                // delta panels [dr | dz | dh] : 3KP panels
    static constexpr int OFF_ADJ = OFF_D + 3 * KP * PANEL_BYTES;   //   later: Pcat half (2KP panels) + dm (KP panels)
    static constexpr int OFF_W = OFF_ADJ + 8 * ADJ_TILE_BYTES;
    static constexpr int OFF_BAR = OFF_W + STAGES * TILE_BYTES;
    static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;
};

struct Args {
    int mb, N, T;
    const void *adj;             // fp32 (mb,E,N,N), or bytes when adj_u8
    int adj_u8;
    float *dHs;
    int every_step;              // dHs: (T+1) slices, an external gradient for every h_t; else two, [0] <-> h_0, [1] <-> h_T
    const uint8_t *img[BMP_MAX_STEPS];
    int stateful[BMP_MAX_STEPS];
    const int *ext_flags;        // [T+1]: != 0 where dHs[t] holds a non-zero external gradient
    long long *dbg;              // optional phase timestamps of CTA 0 (tools/tc_timeline.py)
    Stash2 st;                   // bf16 panel stash: gate values in, delta / P panels out
    const int32_t *midx;         // optional (mb,): adj is a drug table, molecule b = table row midx[b]
};

// flags[t] |= 1 when dHs[t] has any non-zero entry (the intermediate states normally receive no external gradient)
__global__ void nonzero_flags_kernel(const float *__restrict__ x, long n_per_t, int *flags) {
    const int t = blockIdx.y;
    const float4 *p = reinterpret_cast<const float4 *>(x + (long)t * n_per_t);
    bool nz = false;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n_per_t / 4; i += (long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(p + i);
        nz |= (v.x != 0.f) | (v.y != 0.f) | (v.z != 0.f) | (v.w != 0.f);
    }
    if (__syncthreads_or(nz) && threadIdx.x == 0) atomicOr(flags + t, 1);
}

template <int H>
__global__ void __launch_bounds__(32 * (H / 8 + 2), 1) ggnn_tc_bwd_kernel(const Args a) {
    using C = Cfg<H>;
    constexpr int KP = C::KP;
    constexpr int EPW = H / 8;          // epilogue warps: 4 TMEM lane quarters x (H / 32) column groups
    constexpr int NE = 32 * EPW;
    constexpr int NC = 32;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_d = sbase + C::OFF_D, s_adj = sbase + C::OFF_ADJ, s_w = sbase + C::OFF_W, s_bar = sbase + C::OFF_BAR;
    const uint32_t s_dm = s_d + 2 * KP * PANEL_BYTES;     // dm panels alias the delta_h panels (dead after MMA-dx)
    auto BAR = [&](int i) { return s_bar + 8u * i; };
    constexpr int B_FULL = 0, B_EMPTY = 4, B_DRDY = 8, B_Q = 9, B_DRRDY = 10, B_DX = 11, B_DMRDY = 12, B_P = 13,
                  B_PRDY = 17, B_PFREE = 19, B_DH = 20, NBAR = 21;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::OFF_BAR + 8 * NBAR + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (a.mb + 1) / 2;
    const long rows_total = (long)a.mb * a.N;

    if (tid == 0) {
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(BAR(B_FULL + s), 1); mbar_init(BAR(B_EMPTY + s), 1); }
        mbar_init(BAR(B_DRDY), EPW);
        mbar_init(BAR(B_Q), 1);
        mbar_init(BAR(B_DRRDY), EPW);
        mbar_init(BAR(B_DX), 1);
        mbar_init(BAR(B_DMRDY), EPW);
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
    // TMEM columns: [0,H) q, then P(0,0) and P(1,1) ; [H,2H) dh_x (+ dh_msg) ; [2H,3H) dm, then P(1,0) ; [3H,4H) P(0,1)
    constexpr uint32_t COL_Q = 0, COL_DHX = H, COL_DM = 2 * H;

    if (warp == EPW) {
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int t = a.T - 1; t >= 0; --t) {
                    const int ntiles = a.stateful[t] ? C::TILES_STATEFUL : C::TILES_STATELESS;
                    const uint8_t *src = a.img[t];
                    for (int s = 0; s < ntiles; ++s) {
                        mbar_wait(BAR(B_EMPTY + stage), phase ^ 1);
                        mbar_expect_tx(BAR(B_FULL + stage), C::TILE_BYTES);
                        tma_bulk_g2s(s_w + stage * C::TILE_BYTES, src + (size_t)s * C::TILE_BYTES, C::TILE_BYTES, BAR(B_FULL + stage));
                        if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                    }
                }
        }
    } else if (warp == EPW + 1) {
        if (lane == 0) {
            constexpr uint32_t ID_KK = idesc2(H, 0, 0), ID_MNMN = idesc2(H, 1, 1);
            uint32_t stage = 0, phase = 0, it = 0;
            auto mma_wtile = [&](uint32_t a_addr, uint32_t dcol, bool first) {
                mbar_wait(BAR(B_FULL + stage), phase);
                tc_fence_after();
                const uint32_t b_addr = s_w + stage * C::TILE_BYTES;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem + dcol, desc_kmajor(a_addr + k * 32), desc_kmajor(b_addr + k * 32), ID_KK, (first && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_EMPTY + stage));
                if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            };
            // P(mol,p) = [A_2p^T ; A_2p+1^T](mol) x dm(mol): both operands MN-major
            auto mma_p = [&](int mol, int p, uint32_t dcol, int bar) {
                const uint32_t a_addr = s_adj + (mol * 4 + 2 * p) * ADJ_TILE_BYTES;
                const uint32_t b_addr = s_dm + mol * 64 * 128;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem + dcol, desc_mnmajor_adj(a_addr + k * 16 * 128), desc_mnmajor(b_addr + k * 16 * 128), ID_MNMN, k ? 1u : 0u);
                tc_commit(BAR(bar));
            };
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int t = a.T - 1; t >= 0; --t, ++it) {
                    const uint32_t par = it & 1;
                    const bool stateful = a.stateful[t] != 0;
                    mbar_wait(BAR(B_DRDY), par);
                    tc_fence_after();
                    uint8_t *Dt = a.st.Dp + ((size_t)t * n_tiles + tile) * 3 * KP * PANEL_BYTES;
                    uint8_t *Pt2 = a.st.Pp + ((size_t)t * n_tiles + tile) * 4 * KP * PANEL_BYTES;
                    {   // delta_z | delta_h panels (and the zeroed delta_r of a stateless step)
                        const uint32_t from = stateful ? KP : 0;
                        tma_bulk_s2g(Dt + (size_t)from * PANEL_BYTES, s_d + from * PANEL_BYTES, (3 * KP - from) * PANEL_BYTES);
                        bulk_commit();
                    }
                    if (stateful)
                        for (int kp = 0; kp < KP; ++kp) mma_wtile(s_d + (2 * KP + kp) * PANEL_BYTES, COL_Q, kp == 0);
                    tc_commit(BAR(B_Q));
                    // dx over the delta_z and delta_h panels (K blocks 1, 2), both N blocks
                    for (int kb = 1; kb <= 2; ++kb)
                        for (int nb = 0; nb < 2; ++nb)
                            for (int kp = 0; kp < KP; ++kp)
                                mma_wtile(s_d + (kb * KP + kp) * PANEL_BYTES, nb ? COL_DM : COL_DHX, kb == 1 && kp == 0);
                    mbar_wait(BAR(B_DRRDY), par);
                    tc_fence_after();
                    if (stateful) {
                        tma_bulk_s2g(Dt, s_d, KP * PANEL_BYTES);      // delta_r panels
                        bulk_commit();
                    }
                    if (stateful)
                        for (int nb = 0; nb < 2; ++nb)
                            for (int kp = 0; kp < KP; ++kp) mma_wtile(s_d + kp * PANEL_BYTES, nb ? COL_DM : COL_DHX, false);
                    bulk_wait_read();      // the delta panels are about to be reused (dm, Pcat)
                    tc_commit(BAR(B_DX));
                    mbar_wait(BAR(B_DMRDY), par);
                    tc_fence_after();
                    mma_p(0, 0, 0 * H, B_P + 0);
                    mma_p(1, 0, 2 * H, B_P + 1);
                    mma_p(0, 1, 3 * H, B_P + 2);
                    mbar_wait(BAR(B_PRDY + 0), par);          // P(0,0) has left columns [0,H); Pcat half 0 is ready
                    tc_fence_after();
                    tma_bulk_s2g(Pt2, s_d, 2 * KP * PANEL_BYTES);
                    bulk_commit();
                    mma_p(1, 1, 0 * H, B_P + 3);
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_d + kp * PANEL_BYTES, COL_DHX, false);
                    bulk_wait_read();
                    tc_commit(BAR(B_PFREE));
                    mbar_wait(BAR(B_PRDY + 1), par);
                    tc_fence_after();
                    tma_bulk_s2g(Pt2 + (size_t)2 * KP * PANEL_BYTES, s_d, 2 * KP * PANEL_BYTES);
                    bulk_commit();
                    for (int kp = 0; kp < 2 * KP; ++kp) mma_wtile(s_d + kp * PANEL_BYTES, COL_DHX, false);
                    bulk_wait_read();
                    tc_commit(BAR(B_DH));
                }
        }
    } else {
        const int q = warp & 3, hf = warp >> 2;
        const int row = 32 * q + lane;
        const int colbase = hf * NC;
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
        const int molslot = row >> 6, atom = row & 63;
        float acc[NC];       // dL/dh_{t+1}, then ds, then dL/dh_t
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int molg = tile * 2 + molslot;
            const bool live = molg < a.mb && atom < a.N;
            const long grow = (long)molg * a.N + atom;
            stage_adjacency<NE>(smem + C::OFF_ADJ, a.adj, a.adj_u8, tile, a.mb, a.N, tid, a.midx);
            {
                const float *src = live ? a.dHs + ((long)(a.every_step ? a.T : 1) * rows_total + grow) * H + colbase : nullptr;
#pragma unroll
                for (int c = 0; c < NC; c += 4) {
                    float4 v = src ? *reinterpret_cast<const float4 *>(src + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                    acc[c] = v.x; acc[c + 1] = v.y; acc[c + 2] = v.z; acc[c + 3] = v.w;
                }
            }
            for (int t = a.T - 1; t >= 0; --t, ++it) {
                const uint32_t par = it & 1;
                const bool stateful = a.stateful[t] != 0;
                uint32_t v[32];
#define TS(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0 && it < 64) a.dbg[it * 16 + (i)] = clock64(); } while (0)
                TS(0);
                if (t == 0 && tile + (int)gridDim.x < n_tiles) prefetch_adjacency_l2<NE>(a.adj, a.adj_u8, tile + gridDim.x, a.mb, a.N, tid, a.midx);
                // ---- phase A: gate derivatives ----
                // gate values of the step: coalesced 16-byte loads in the thread-native bf16 order, two 16-column halves
                // (L2-resident: prefetched during the previous step) so the live set stays under the 96-register budget
                const uint8_t *bz = a.st.zn(t, tile, 0, H), *bh = a.st.zn(t, tile, 1, H), *bs = a.st.zn(t, tile, 3, H);
#pragma unroll
                for (int half = 0; half < NC / 16; ++half) {
                    uint4 zp[2], hp[2], sp[2];
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const size_t o = ((size_t)(2 * half + g) * NE + tid) * 16;
                        zp[g] = __ldg(reinterpret_cast<const uint4 *>(bz + o));
                        hp[g] = __ldg(reinterpret_cast<const uint4 *>(bh + o));
                        sp[g] = stateful ? __ldg(reinterpret_cast<const uint4 *>(bs + o)) : make_uint4(0, 0, 0, 0);
                    }
#pragma unroll
                    for (int g = 0; g < 2; ++g) {
                        const int j = 2 * half + g;
                        const __nv_bfloat162 *z2 = reinterpret_cast<const __nv_bfloat162 *>(&zp[g]);
                        const __nv_bfloat162 *h2 = reinterpret_cast<const __nv_bfloat162 *>(&hp[g]);
                        const __nv_bfloat162 *s2 = reinterpret_cast<const __nv_bfloat162 *>(&sp[g]);
                        float dz[8], dh[8];
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            const float2 zz = __bfloat1622float2(z2[x]), hh = __bfloat1622float2(h2[x]), ss = __bfloat1622float2(s2[x]);
                            const float g0 = live ? acc[8 * j + 2 * x] : 0.f, g1 = live ? acc[8 * j + 2 * x + 1] : 0.f;
                            dz[2 * x] = g0 * (hh.x - ss.x) * zz.x * (1.f - zz.x);
                            dz[2 * x + 1] = g1 * (hh.y - ss.y) * zz.y * (1.f - zz.y);
                            dh[2 * x] = g0 * zz.x * (1.f - hh.x * hh.x);
                            dh[2 * x + 1] = g1 * zz.y * (1.f - hh.y * hh.y);
                            acc[8 * j + 2 * x] = stateful ? g0 * (1.f - zz.x) : 0.f;
                            acc[8 * j + 2 * x + 1] = stateful ? g1 * (1.f - zz.y) : 0.f;
                        }
                        const int kk = colbase + 8 * j;
                        uint4 pz = make_uint4(pack_bf16(dz[0], dz[1]), pack_bf16(dz[2], dz[3]), pack_bf16(dz[4], dz[5]), pack_bf16(dz[6], dz[7]));
                        uint4 ph = make_uint4(pack_bf16(dh[0], dh[1]), pack_bf16(dh[2], dh[3]), pack_bf16(dh[4], dh[5]), pack_bf16(dh[6], dh[7]));
                        *reinterpret_cast<uint4 *>(smem + C::OFF_D + (KP + (kk >> 6)) * PANEL_BYTES + sw128(row, kk & 63)) = pz;
                        *reinterpret_cast<uint4 *>(smem + C::OFF_D + (2 * KP + (kk >> 6)) * PANEL_BYTES + sw128(row, kk & 63)) = ph;
                        if (!stateful)   // delta_r panel of a stateless step: zeros (the merged W_r contraction reads it)
                            *reinterpret_cast<uint4 *>(smem + C::OFF_D + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = make_uint4(0, 0, 0, 0);
                    }
                }
                warp_arrive(BAR(B_DRDY), lane);
                TS(1);
                // ---- phase B: through U and the reset gate ----
                // 16-column halves keep the live set under the 96-register budget: r and (again, L2-resident) the state of
                // the first half are requested before waiting for q (the latency overlaps MMA-q), the second half's while
                // the first is consumed
                const uint8_t *br = a.st.zn(t, tile, 2, H);
                uint4 rp[2], sp[2];
                auto load_rs = [&](int half) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        rp[j] = __ldg(reinterpret_cast<const uint4 *>(br + ((size_t)(2 * half + j) * NE + tid) * 16));
                        sp[j] = __ldg(reinterpret_cast<const uint4 *>(bs + ((size_t)(2 * half + j) * NE + tid) * 16));
                    }
                };
                if (stateful) load_rs(0);
                mbar_wait(BAR(B_Q), par);
                tc_fence_after();
                TS(2);
                if (stateful) {
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
                        uint32_t w[16];
                        tc_ld16(t_lane + COL_Q + colbase + 16 * half, w);
                        tc_wait_ld();
                        float dr[16];
#pragma unroll
                        for (int g = 0; g < 2; ++g) {
                            const int j = 2 * half + g;
                            const __nv_bfloat162 *r2 = reinterpret_cast<const __nv_bfloat162 *>(&rp[g]);
                            const __nv_bfloat162 *s2 = reinterpret_cast<const __nv_bfloat162 *>(&sp[g]);
#pragma unroll
                            for (int x = 0; x < 4; ++x) {
                                const float2 rr = __bfloat1622float2(r2[x]), ss = __bfloat1622float2(s2[x]);
                                const float q0 = live ? __uint_as_float(w[8 * g + 2 * x]) : 0.f, q1 = live ? __uint_as_float(w[8 * g + 2 * x + 1]) : 0.f;
                                acc[8 * j + 2 * x] += q0 * rr.x;
                                acc[8 * j + 2 * x + 1] += q1 * rr.y;
                                dr[8 * g + 2 * x] = q0 * ss.x * rr.x * (1.f - rr.x);
                                dr[8 * g + 2 * x + 1] = q1 * ss.y * rr.y * (1.f - rr.y);
                            }
                        }
                        if (half == 0) load_rs(1);
#pragma unroll
                        for (int g = 0; g < 2; ++g) {
                            const int kk = colbase + 8 * (2 * half + g);
                            uint4 pr = make_uint4(pack_bf16(dr[8 * g], dr[8 * g + 1]), pack_bf16(dr[8 * g + 2], dr[8 * g + 3]),
                                                  pack_bf16(dr[8 * g + 4], dr[8 * g + 5]), pack_bf16(dr[8 * g + 6], dr[8 * g + 7]));
                            *reinterpret_cast<uint4 *>(smem + C::OFF_D + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pr;
                        }
                    }
                }
                warp_arrive(BAR(B_DRRDY), lane);
                TS(3);
                // ---- phase C: dm -> bf16 operand panels (B of MMA-P) ----
                mbar_wait(BAR(B_DX), par);
                tc_fence_after();
                TS(4);
#pragma unroll
                for (int cc = 0; cc < NC; cc += 32) {
                    tc_ld32(t_lane + COL_DM + colbase + cc, v);
                    tc_wait_ld();
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const int kk = colbase + cc + 8 * g;
                        uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])),
                                              pack_bf16(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3])),
                                              pack_bf16(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5])),
                                              pack_bf16(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
                        *reinterpret_cast<uint4 *>(smem + C::OFF_D + (2 * KP + (kk >> 6)) * PANEL_BYTES + sw128(row, kk & 63)) = pk;
                    }
                }
                warp_arrive(BAR(B_DMRDY), lane);
                TS(5);
                if (t > 0) {      // while MMA-P runs: gate values of the NEXT step (t-1) towards L2 (four 128 x H bf16 blocks)
                    const char *nx = reinterpret_cast<const char *>(a.st.zn(t - 1, tile, 0, H));
                    for (int off = tid * 128; off < 4 * 128 * H * 2; off += NE * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + off));
                }
                // ---- phase D: P accumulators -> bf16 A-operand panels (two K halves) ----
                for (int p = 0; p < 2; ++p) {
                    if (p == 1) mbar_wait(BAR(B_PFREE), par);
                    for (int mol = 0; mol < 2; ++mol) {
                        const int pi = 2 * p + mol;                         // (0,0)->0 (1,0)->1 (0,1)->2 (1,1)->3
                        const uint32_t pcol = (pi == 0 || pi == 3) ? 0u : (pi == 1 ? 2u * H : 3u * H);
                        mbar_wait(BAR(B_P + pi), par);
                        tc_fence_after();
                        TS(6 + pi);
                        const int orow = mol * 64 + atom;                   // row of (mol, atom j) in the tile
                        const int kbase = molslot * H + colbase;            // TMEM lane half = bond type within the pair
#pragma unroll
                        for (int cc = 0; cc < NC; cc += 32) {
                            tc_ld32(t_lane + pcol + colbase + cc, v);
                            tc_wait_ld();
#pragma unroll
                            for (int g = 0; g < 4; ++g) {
                                const int kk = kbase + cc + 8 * g;
                                uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])),
                                                      pack_bf16(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3])),
                                                      pack_bf16(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5])),
                                                      pack_bf16(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
                                *reinterpret_cast<uint4 *>(smem + C::OFF_D + (kk >> 6) * PANEL_BYTES + sw128(orow, kk & 63)) = pk;
                            }
                        }
                    }
                    warp_arrive(BAR(B_PRDY + p), lane);         // one hand-off per K half (both molecules written)
                }
                TS(10);
                // ---- phase E: dh_t = dh_x (+ dh_msg) + ds + external gradient ----
                {
                    const float *ext = a.dHs + ((long)(a.every_step ? t : 0) * rows_total + grow) * H + colbase;
                    const bool has_ext = live && (a.every_step ? a.ext_flags[t] != 0 : t == 0);
                    if (has_ext) {      // requested and folded in before waiting for the accumulator: the latency overlaps MMA-dh
#pragma unroll
                        for (int x = 0; x < NC; x += 4) {
                            const float4 e = __ldg(reinterpret_cast<const float4 *>(ext + x));
                            acc[x] += e.x; acc[x + 1] += e.y; acc[x + 2] += e.z; acc[x + 3] += e.w;
                        }
                    }
                    mbar_wait(BAR(B_DH), par);
                    tc_fence_after();
                    TS(11);
#pragma unroll
                    for (int cc = 0; cc < NC; cc += 32) {
                        tc_ld32(t_lane + COL_DHX + colbase + cc, v);
                        tc_wait_ld();
#pragma unroll
                        for (int x = 0; x < 32; ++x) acc[cc + x] += __uint_as_float(v[x]);
                    }
                    if (t == 0) {
                        // dL/dh_0 of the tile: coalesced rows through a transposition block (the delta panels are idle:
                        // every MMA of the tile has completed)
                        float *stg = reinterpret_cast<float *>(smem + C::OFF_D + warp * 2048);
                        float *out = a.dHs + colbase;      // slice 0 in both dHs layouts
#pragma unroll
                        for (int h2 = 0; h2 < 2; ++h2)
                            warp_store_rows<16>(stg, acc + 16 * h2, lane, [&](int r) -> float * {
                                const int tr = 32 * q + r, mg = tile * 2 + (tr >> 6), at = tr & 63;
                                return (mg < a.mb && at < a.N) ? out + ((long)mg * a.N + at) * H + 16 * h2 : nullptr;
                            });
                    }
                }
                TS(12);
                tc_fence_before();
                if (t == 0) asm volatile("bar.sync 1, %0;" ::"n"(NE));   // tile finished: smem/TMEM may be re-staged
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

// ---- weight images for the backward: tiles [H n][64 k] bf16, SW128, in consumption order
//   stateful : [q: KP] [z: dhx KP, dm KP] [hbar: dhx KP, dm KP] [r: dhx KP, dm KP] [dh: 4KP]
//   stateless:         [z: dhx KP, dm KP] [hbar: dhx KP, dm KP]                     [dh: 4KP]
struct PackArgs {
    int H, stateful;
    const float *msg_W;
    bmp_gru_t g;
    uint8_t *img;
};

__global__ void pack_bwd_kernel(const PackArgs p) {
    const int H = p.H, KP = H / 64;
    const int nq = p.stateful ? KP : 0, ndx = p.stateful ? 6 * KP : 4 * KP;
    const int ntiles = nq + ndx + 4 * KP;
    const long total = (long)ntiles * H * 64;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int k = idx & 63, n = (idx >> 6) % H, tile = (int)(idx / (64L * H));
        float w;
        if (tile < nq) {                                   // q[row][n] = sum_c delta_h[row][c] U[c][n]
            const int c = tile * 64 + k;
            w = p.g.U[(long)c * H + n];
        } else if (tile < nq + ndx) {
            const int u = tile - nq, kb = u / (2 * KP), nb = (u / KP) & 1, kp = u % KP;
            const int gate = kb == 0 ? 1 : (kb == 1 ? 2 : 0);                 // z, hbar, r
            const int c = kp * 64 + k;
            const float *W = gate == 0 ? p.g.W_r : (gate == 1 ? p.g.W_z : p.g.W);
            w = W[(long)c * 2 * H + nb * H + n];
            if (p.stateful && nb == 0 && gate < 2) w += (gate == 0 ? p.g.U_r : p.g.U_z)[(long)c * H + n];
        } else {                                           // dh[row][n] = sum_{e,c} P_e[row][c] W_e[c][n]
            const int K = (tile - nq - ndx) * 64 + k, e = K / H, c = K % H;
            w = p.msg_W[((long)c * 4 + e) * H + n];
        }
        __nv_bfloat16 b = __float2bfloat16_rn(w);
        const uint32_t off = (uint32_t)n * 128u + ((((uint32_t)(k >> 3) ^ ((uint32_t)n & 7u)) << 4) | (((uint32_t)k & 7u) << 1));
        *reinterpret_cast<__nv_bfloat16 *>(p.img + (size_t)tile * H * 128 + off) = b;
    }
}

static size_t image_bytes(int H) { return (size_t)(11 * (H / 64)) * H * 128 + 256; }

}  // namespace tcb
}  // namespace bmp

using namespace bmp;

static long long *g_tc_dbg = nullptr;
extern "C" void bmp_debug_set_buffer(void *p) { g_tc_dbg = (long long *)p; }

int bmp_wgrad_panels_multi(bmp::w2::Args *list, int n, void *stream);   // wgrad_tc2.cu

// BMP_MODE_BF16 backward over the bf16 panel stash; called by bmp_ggnn_backward.  The data kernel, then every parameter
// gradient as a C += A^T B contraction whose operands are streamed straight from the dumped panels.
int bmp_ggnn_backward_tc(const bmp_ggnn_bwd_t *a, void *stream) {
    const int H = a->hidden, T = a->n_steps, KP = H / 64;
    if (!a->tc_workspace || a->tc_workspace_bytes < bmp_ggnn_tc_workspace_bytes(H, T)) {
        set_error("BMP_MODE_BF16 backward: tc_workspace of >= %zu bytes required", bmp_ggnn_tc_workspace_bytes(H, T));
        return BMP_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    tcb::Args k = {};
    k.mb = a->mb; k.N = a->n_atoms; k.T = T; k.adj = a->adj; k.adj_u8 = a->adj_u8; k.dHs = a->dHs; k.every_step = a->dHs_every_step != 0;
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 255) & ~(uintptr_t)255);
    int *flags = reinterpret_cast<int *>(ws);      // first 256 B of the workspace: per-step external-gradient flags
    ws += 256;
    if (k.every_step) {
        cudaMemsetAsync(flags, 0, (T + 1) * sizeof(int), st);
        tcb::nonzero_flags_kernel<<<dim3(64, T + 1), 256, 0, st>>>(a->dHs, (long)a->mb * a->n_atoms * H, flags);
        count_launch();
    }
    k.ext_flags = flags;
    k.dbg = g_tc_dbg;
    k.midx = a->mol_index;
    const int n_tiles = (a->mb + 1) / 2;
    k.st.carve(a->stash2, n_tiles, H, T);
    const size_t ib = tcb::image_bytes(H);
    int n_img = 0;
    for (int t = 0; t < T; ++t) {
        int found = -1;
        for (int u = 0; u < t; ++u)
            if (a->msg_W[u] == a->msg_W[t] && same_gru(a->gru[u], a->gru[t]) &&
                (a->stateful[u] != 0) == (a->stateful[t] != 0)) { found = u; break; }
        k.stateful[t] = a->stateful[t] != 0;
        if (found >= 0) { k.img[t] = k.img[found]; continue; }
        tcb::PackArgs p;
        p.H = H; p.stateful = k.stateful[t]; p.msg_W = a->msg_W[t]; p.g = a->gru[t]; p.img = ws + (size_t)n_img * ib;
        if (!a->tc_images_ready) {
            tcb::pack_bwd_kernel<<<64, 256, 0, st>>>(p);
            count_launch();
        }
        k.img[t] = p.img;
        ++n_img;
    }
    int rc = check_launch("pack_bwd_kernel");
    if (rc) return rc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = n_tiles < sms ? n_tiles : sms;
#define LAUNCH_BWD(HH)                                                                                                     \
    do {                                                                                                                   \
        cudaFuncSetAttribute(tcb::ggnn_tc_bwd_kernel<HH>, cudaFuncAttributeMaxDynamicSharedMemorySize, tcb::Cfg<HH>::SMEM_BYTES); \
        tcb::ggnn_tc_bwd_kernel<HH><<<grid, 32 * (HH / 8 + 2), tcb::Cfg<HH>::SMEM_BYTES, st>>>(k);                              \
    } while (0)
    {
        ProfScope prof(BMP_PROF_GGNN_BWD, st);
        if (H == 64) LAUNCH_BWD(64);
        else LAUNCH_BWD(128);
    }
#undef LAUNCH_BWD
    count_launch();
    if ((rc = check_launch("ggnn_tc_bwd_kernel"))) return rc;
    const tc::Stash2 &S = k.st;
    // Grouped contractions: every launch reads its A blocks and B blocks once (the kernel is HBM-bound), so the
    // launches are arranged for the fewest operand reads:
    //   per gate g and run of equal statefulness:  delta_g^T [h | m | r*h]  -> W_g (both halves) and U_g together
    //   per pair of bond types:                    [P_e ; P_e']^T h         -> two row groups of W_msg
    // One launch per run of equal statefulness: its gate classes and its message classes walk the same (step, tile) units in
    // lockstep, so the h / m panels all of them read come from HBM once (w2::Multi).
    w2::Args cls[w2::MAX_CLASSES];
    int ncls = 0;
    auto flush = [&]() -> int {
        int e = ncls ? bmp_wgrad_panels_multi(cls, ncls, stream) : BMP_OK;
        ncls = 0;
        return e;
    };
    auto push = [&](const w2::Args &k) -> int {
        if (ncls && (cls[0].t0 != k.t0 || cls[0].t1 != k.t1)) { int e = flush(); if (e) return e; }
        cls[ncls++] = k;
        return ncls == w2::MAX_CLASSES ? flush() : BMP_OK;
    };
    auto gate_launch = [&](int g, int ta, int tb, bool stateful, const bmp_gru_grad_t &D) -> int {
        float *Wg = g == 0 ? D.W_r : (g == 1 ? D.W_z : D.W), *bW = g == 0 ? D.b_Wr : (g == 1 ? D.b_Wz : D.b_W);
        float *Ug = !stateful ? nullptr : (g == 0 ? D.U_r : (g == 1 ? D.U_z : D.U));
        float *bU = !stateful ? nullptr : (g == 0 ? D.b_Ur : (g == 1 ? D.b_Uz : D.b_U));
        if (!Wg && !Ug) return BMP_OK;
        for (int mt = 0; mt < KP; mt += 2) {          // 128 rows of the gradient per class
            w2::Args k = {};
            k.A = S.Dp; k.a_ppt = 3 * KP; k.n_mt = 1;
            k.a_panel[0][0] = g * KP + mt; k.a_panel[0][1] = mt + 1 < KP ? g * KP + mt + 1 : -1;
            k.a_panel[1][0] = k.a_panel[1][1] = -1;
            int nb = 0;
            for (int j = 0; j < KP; ++j, ++nb) { k.B[nb] = S.Xp; k.b_ppt[nb] = KP; k.b_panel[nb] = j; }
            for (int j = 0; j < KP; ++j, ++nb) { k.B[nb] = S.Mp; k.b_ppt[nb] = KP; k.b_panel[nb] = j; }
            if (g == 2 && Ug)
                for (int j = 0; j < KP; ++j, ++nb) { k.B[nb] = S.RSp; k.b_ppt[nb] = KP; k.b_panel[nb] = j; }
            k.nb = nb;
            for (int bl = 0; bl < 2; ++bl) {
                if (k.a_panel[0][bl] < 0) continue;
                const long row0 = (long)(mt + bl) * 64;
                for (int j = 0; j < nb; ++j) {
                    if (j < 2 * KP) {                  // W_g[:, j*64 ...] ; U_r / U_z see the h product as well
                        k.C[0][bl][j] = Wg ? Wg + row0 * 2 * H + j * 64 : nullptr;
                        k.ldc[j] = 2 * H;
                        if (g < 2 && Ug && j < KP) { k.C2[0][bl][j] = Ug + row0 * H + j * 64; k.ldc2[j] = H; }
                    } else {                           // U[:, ...] from the r*h panels
                        k.C[0][bl][j] = Ug + row0 * H + (j - 2 * KP) * 64;
                        k.ldc[j] = H;
                    }
                }
                k.bias[0][bl] = bW ? bW + row0 : nullptr;
                k.bias2[0][bl] = bU ? bU + row0 : nullptr;
            }
            k.bias_stride = 1;
            k.t0 = ta; k.t1 = tb; k.n_tiles = n_tiles;
            int e = push(k);
            if (e) return e;
        }
        return BMP_OK;
    };
    auto msg_launch = [&](int tw, int ta, int tb) -> int {
        // dW_m[c*E+e][:] += P_e^T h_t : C rows c with stride E*H, offset e*H; bias d_msg_b[c*E+e]
        const bool pair_up = KP <= 3;              // two bond types (M tiles) per class while N = 64 KP fits 192 columns
        for (int e = 0; e < 4; e += pair_up ? 2 : 1)
            for (int mt = 0; mt < KP; mt += 2) {
                w2::Args k = {};
                k.A = S.Pp; k.a_ppt = 4 * KP; k.n_mt = pair_up ? 2 : 1;
                for (int m = 0; m < 2; ++m) {
                    const bool on = m < k.n_mt;
                    k.a_panel[m][0] = on ? (e + m) * KP + mt : -1;
                    k.a_panel[m][1] = on && mt + 1 < KP ? (e + m) * KP + mt + 1 : -1;
                }
                k.nb = KP;
                for (int j = 0; j < KP; ++j) { k.B[j] = S.Xp; k.b_ppt[j] = KP; k.b_panel[j] = j; k.ldc[j] = 4 * H; }
                for (int m = 0; m < k.n_mt; ++m)
                    for (int bl = 0; bl < 2; ++bl) {
                        if (k.a_panel[m][bl] < 0) continue;
                        const long c0 = (long)(mt + bl) * 64;          // first channel c of this block
                        for (int j = 0; j < KP; ++j) k.C[m][bl][j] = a->d_msg_W[tw] + (c0 * 4 + (e + m)) * H + j * 64;
                        k.bias[m][bl] = a->d_msg_b[tw] ? a->d_msg_b[tw] + c0 * 4 + (e + m) : nullptr;
                    }
                k.bias_stride = 4;
                k.t0 = ta; k.t1 = tb; k.n_tiles = n_tiles;
                int e2 = push(k);
                if (e2) return e2;
            }
        return BMP_OK;
    };
    int t0 = 0;
    while (t0 < T) {
        int t1 = t0;
        while (t1 + 1 < T && a->d_msg_W[t1 + 1] == a->d_msg_W[t0] && a->d_gru[t1 + 1].W == a->d_gru[t0].W &&
               a->d_gru[t1 + 1].U == a->d_gru[t0].U)
            ++t1;
        const bmp_gru_grad_t &D = a->d_gru[t0];
        int s0 = t0;
        while (s0 <= t1) {       // runs of equal statefulness (U-type gradients only over stateful steps)
            const bool st = a->stateful[s0] != 0;
            int s1 = s0;
            while (s1 + 1 <= t1 && (a->stateful[s1 + 1] != 0) == st) ++s1;
            for (int g = st ? 0 : 1; g < 3; ++g)       // delta_r of a stateless step is identically zero
                if ((rc = gate_launch(g, s0, s1, st, D))) return rc;
            if (a->d_msg_W[t0] && (rc = msg_launch(t0, s0, s1))) return rc;
            if ((rc = flush())) return rc;
            s0 = s1 + 1;
        }
        t0 = t1 + 1;
    }
    return BMP_OK;
}
