// ggnn_tc.cu -- fused GGNN encoder on the 5th-gen tensor cores (BMP_MODE_BF16).
//
// One persistent CTA per SM; a work item is a TILE of two padded molecules (2 x 64 atoms =
// 128 rows = one UMMA M).  For all T message-passing steps the tile's adjacency (bf16, exact
// for 0/1 bonds), its hidden state (bf16 operand copy in smem + fp32 master copy in the
// epilogue threads' registers) and every intermediate stay on chip; accumulators live in
// TMEM; the (pre-packed, pre-swizzled bf16) weights stream from L2 with cp.async.bulk (TMA)
// through an mbarrier ring.  Per step (H = hidden):
//   MMA-1  AH[(e,i), c]   = sum_j A_e[i,j] h[j,c]        per molecule, two bond types stacked
//                           on M (128 x 64) x (64 x H); B = the h buffer read MN-major
//   MMA-2  m[(mol,i), c]  = sum_{e,c'} AH_e[i,c'] W_e[c,c']      K = 4H  (+ deg_e b_e in the epilogue)
//   MMA-3  [r|z|hbar]     = [h | m] [W_r+U_r | W_z+U_z | W]^T    K = 2H, N = 3H (U folded: state == h)
//   MMA-4  hbar          += (r*h) U^T                            K = H
//   epilogue: sigmoid/tanh, h <- z*hbar + (1-z)*h  (fp32), new bf16 operand copy
// Warp roles: H/8 epilogue warps (TMEM lane quarter = warp%4, 32-column group = warp/4),
// then one TMA producer warp and one MMA issuer warp (one elected lane each).
// Replaces models/update/ggnn_update.py:31-63 / models/models/ggnn.py:72-106 like ggnn.cu.
#include "tc_common.cuh"

namespace bmp {
namespace tc {

template <int H>
struct Cfg {
    static constexpr int KP = H / 64;
    static constexpr int TILE_BYTES = H * 128;            // weight tile: H rows (n) x 64 bf16 (k)
    static constexpr int STAGES = 4;
    static constexpr int T_MSG = 4 * KP, T_GATE = 2 * KP, T_U = KP;
    static constexpr int TILES_STATEFUL = T_MSG + 3 * T_GATE + T_U;
    static constexpr int TILES_STATELESS = T_MSG + 2 * T_GATE;
    static constexpr int TMEM_COLS = 4 * H;               // 256 or 512 (power of two)
    static constexpr int OFF_H = 0;
    static constexpr int OFF_ADJ = OFF_H + KP * PANEL_BYTES;
    static constexpr int OFF_AH = OFF_ADJ + 8 * ADJ_TILE_BYTES;
    static constexpr int OFF_W = OFF_AH + 2 * KP * PANEL_BYTES;
    static constexpr int OFF_BAR = OFF_W + STAGES * TILE_BYTES;
    static constexpr int SMEM_BYTES = OFF_BAR + 256 + 1024;   // + alignment slack
};

struct Args {
    int mb, N, T, n_types;
    const int32_t *atoms;
    const float *embed_W, *h_in;
    const void *adj;             // fp32 (mb,E,N,N), or bytes when adj_u8
    int adj_u8;
    const uint8_t *img[BMP_MAX_STEPS];     // packed weight tiles of step t
    const float *bias3[BMP_MAX_STEPS];     // [b_r | b_z | b_h] (U biases folded for stateful steps)
    const float *msg_b[BMP_MAX_STEPS];     // (H*4) as in the reference: b[c*4+e]
    int stateful[BMP_MAX_STEPS];
    float *h_out, *h0_out;
    float *Hs;                   // optional (T+1, mb*N, H): h_t of every step (an output, not read back by the backward)
    long long *dbg;              // optional phase timestamps of CTA 0 (tools/tc_timeline.py)
    Stash2 st;                   // bf16 panel stash of the training forward (V2)
    const int32_t *midx;         // optional (mb,): atoms / adj are a drug table, molecule b = table row midx[b]
};

// V2: training, dumps the bf16 panel stash; otherwise inference
template <int H, bool V2>
__global__ void __launch_bounds__(32 * (H / 8 + 2), 1) ggnn_tc_kernel(const Args a) {
    using C = Cfg<H>;
    constexpr int KP = C::KP;
    constexpr int EPW = H / 8;          // epilogue warps: 4 TMEM lane quarters x (H / 32) column groups
    constexpr int NE = 32 * EPW;
    constexpr int NC = 32;              // columns per epilogue thread
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_h = sbase + C::OFF_H, s_adj = sbase + C::OFF_ADJ, s_ah = sbase + C::OFF_AH, s_w = sbase + C::OFF_W;
    const uint32_t s_bar = sbase + C::OFF_BAR;
    // barriers (8 bytes each)
    auto BAR = [&](int i) { return s_bar + 8u * i; };
    // AH slots: the AH buffer (one bond-type pair = 2KP panels) is handed over in KP slots of two panels (both bond types of
    // a 64-column block), so the conversion of the next slot overlaps the UMMAs on the previous one
    constexpr int B_FULL = 0, B_EMPTY = 4, B_HREADY = 8, B_D1 = 9, B_AHREADY = 13, B_AHFREE = 15, B_M = 17,
                  B_XREADY = 18, B_R = 19, B_RSREADY = 20, B_ZH = 21, NBAR = 22;
    // TMEM columns: [0,H) m ; [H,2H) r ; [2H,3H) z ; [3H,4H) hbar.  The two AH accumulators of a bond-type pair (one per
    // molecule) use [2H,4H) -- z / hbar of the previous step are consumed by then -- for p = 0 and again for p = 1, so the
    // message accumulator m never overlaps an AH accumulator that is still being read.
    static_assert(KP <= 2, "two AH slots");
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::OFF_BAR + 8 * NBAR + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (a.mb + 1) / 2;
    const long rows_total = (long)a.mb * a.N;

    if (tid == 0) {
        for (int s = 0; s < C::STAGES; ++s) { mbar_init(BAR(B_FULL + s), 1); mbar_init(BAR(B_EMPTY + s), 1); }
        mbar_init(BAR(B_HREADY), EPW);
        for (int i = 0; i < 2; ++i) mbar_init(BAR(B_D1 + i), 1);
        mbar_init(BAR(B_AHREADY), EPW);
        mbar_init(BAR(B_AHREADY + 1), EPW);
        mbar_init(BAR(B_AHFREE), 1);
        mbar_init(BAR(B_AHFREE + 1), 1);
        mbar_init(BAR(B_M), 1);
        mbar_init(BAR(B_XREADY), EPW);
        mbar_init(BAR(B_R), 1);
        mbar_init(BAR(B_RSREADY), EPW);
        mbar_init(BAR(B_ZH), 1);
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
        // ===================== TMA producer: stream the weight tiles in consumption order
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int t = 0; t < a.T; ++t) {
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
        // ===================== MMA issuer
        if (lane == 0) {
            constexpr uint32_t ID_KK = idesc(H, 0), ID_KMN = idesc(H, 1);
            uint32_t stage = 0, phase = 0, it = 0;
            // one weight tile: 4 k-steps of 16; A panel base `a_addr` (K-major), D columns `dcol`
            long long wsum = 0;          // cycles this lane spent waiting for weight tiles (timeline slot 15)
            auto mma_wtile = [&](uint32_t a_addr, uint32_t dcol, bool first) {
                const long long w0 = a.dbg ? clock64() : 0;
                mbar_wait(BAR(B_FULL + stage), phase);
                if (a.dbg) wsum += clock64() - w0;
                tc_fence_after();
                const uint32_t b_addr = s_w + stage * C::TILE_BYTES;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc_mma(tmem + dcol, desc_kmajor(a_addr + k * 32), desc_kmajor(b_addr + k * 32), ID_KK, (first && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_EMPTY + stage));
                if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            };
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int t = 0; t < a.T; ++t, ++it) {
                    const uint32_t par = it & 1;
                    const bool stateful = a.stateful[t] != 0;
                    mbar_wait(BAR(B_HREADY), par);
                    tc_fence_after();
                    if (V2) {   // every earlier panel dump has left shared memory; dump h_t (the step input)
                        bulk_wait_read();
                        tma_bulk_s2g(a.st.Xp + ((size_t)t * n_tiles + tile) * KP * PANEL_BYTES, s_h, KP * PANEL_BYTES);
                        bulk_commit();
                    }
                    // MMA-1: D1[mol] = [A_2p ; A_2p+1](mol) x h(mol)   (B MN-major from the h panels), p = 0 now, p = 1 as soon as
                    // the epilogue has read the p = 0 accumulators
                    auto mma1 = [&](int p) {
                        for (int mol = 0; mol < 2; ++mol) {
                            const uint32_t a_addr = s_adj + (mol * 4 + 2 * p) * ADJ_TILE_BYTES;
                            const uint32_t b_addr = s_h + mol * 64 * 128;
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                tc_mma(tmem + (2 + mol) * H, desc_kmajor(a_addr + k * 32),
                                       desc_mnmajor(b_addr + k * 16 * 128), ID_KMN, k ? 1u : 0u);
                            tc_commit(BAR(B_D1 + mol));
                        }
                    };
                    mma1(0);
                    // MMA-2: m = AHcat Wcat^T, slot by slot: (bond-type pair p, 64-column block cp) = two K blocks of 64
                    for (int p = 0; p < 2; ++p)
                        for (int cp = 0; cp < KP; ++cp) {
                            mbar_wait(BAR(B_AHREADY + cp), p);          // every slot barrier completes twice per step
                            tc_fence_after();
                            if (p == 0 && cp == KP - 1) mma1(1);        // both p = 0 accumulators have been read completely
                            for (int ein = 0; ein < 2; ++ein) mma_wtile(s_ah + (ein * KP + cp) * PANEL_BYTES, 0, p == 0 && cp == 0 && ein == 0);
                            tc_commit(BAR(B_AHFREE + cp));
                            if (p == 1 && cp == KP - 1) tc_commit(BAR(B_M));
                        }
                    // MMA-3: gates over x = [h | m]
                    mbar_wait(BAR(B_XREADY), par);
                    tc_fence_after();
                    if (V2) {
                        tma_bulk_s2g(a.st.Mp + ((size_t)t * n_tiles + tile) * KP * PANEL_BYTES, s_ah, KP * PANEL_BYTES);
                        bulk_commit();
                    }
                    auto gate_block = [&](uint32_t dcol) {
                        for (int kp = 0; kp < 2 * KP; ++kp)
                            mma_wtile(kp < KP ? s_h + kp * PANEL_BYTES : s_ah + (kp - KP) * PANEL_BYTES, dcol, kp == 0);
                    };
                    if (stateful) gate_block(1 * H);
                    tc_commit(BAR(B_R));
                    gate_block(2 * H);
                    gate_block(3 * H);
                    // MMA-4: hbar += (r*h) U^T
                    mbar_wait(BAR(B_RSREADY), par);
                    tc_fence_after();
                    if (V2 && stateful) {
                        tma_bulk_s2g(a.st.RSp + ((size_t)t * n_tiles + tile) * KP * PANEL_BYTES, s_ah + KP * PANEL_BYTES, KP * PANEL_BYTES);
                        bulk_commit();
                    }
                    if (stateful)
                        for (int kp = 0; kp < KP; ++kp) mma_wtile(s_ah + (KP + kp) * PANEL_BYTES, 3 * H, false);
                    if (V2) bulk_wait_read();      // h_t / m_t / r*h_t dumps are out before E4 rewrites the h panels
                    tc_commit(BAR(B_ZH));
                    if (a.dbg && blockIdx.x == 0 && it < 64) { a.dbg[it * 16 + 15] = wsum; wsum = 0; }
                }
        }
    } else {
        // ===================== epilogue warps 0..7
        const int q = warp & 3, hf = warp >> 2;
        const int row = 32 * q + lane;            // TMEM lane == tile row
        const int colbase = hf * NC;
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
        const int molslot = row >> 6, atom = row & 63;
        float hreg[NC];
        // transposition staging for coalesced fp32 stores: the AH buffer, idle at the only moments anything is stored -- tile
        // start (h_0) and E4 (the new state): after B_ZH every MMA of the step has read AH and its panel dumps have left it
        // (bulk_wait_read), and no warp writes it again before all of them have arrived on B_HREADY
        float *stg = reinterpret_cast<float *>(smem + C::OFF_AH + warp * 2048);
        uint32_t it = 0;
#define TSP(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0 && it < 64) a.dbg[it * 16 + 8 + (i)] = clock64(); } while (0)
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            TSP(0);
            const int molg = tile * 2 + molslot;
            const bool live = molg < a.mb && atom < a.N;
            const long grow = (long)molg * a.N + atom;       // global row of this thread (if live)
            // global row of warp row r (0..31), or -1: used by the coalesced (transposed) stash stores
            auto wrow = [&](int r) -> long {
                const int tr = 32 * q + r, mg = tile * 2 + (tr >> 6), at = tr & 63;
                return (mg < a.mb && at < a.N) ? (long)mg * a.N + at : -1L;
            };
            // store 32 columns [col0, col0+32) of every live row of this warp to base[(grow*ld) + col0 ..]
            auto store_rows = [&](float *base, long ld, int col0, const float *vals) {
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2)      // two 16-column passes: 2 KB of staging per warp
                    warp_store_rows<16>(stg, vals + 16 * h2, lane, [&](int r) -> float * {
                        const long g = wrow(r);
                        return g >= 0 ? base + g * ld + col0 + 16 * h2 : nullptr;
                    });
            };
            // bf16 gate values in the thread-native order [16-byte chunk j][thread]: coalesced 512 B per warp store
            auto store_native16 = [&](int t, int arr, int cc, const float *vals) {
                uint8_t *base = a.st.zn(t, tile, arr, H);
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    uint4 pk = make_uint4(pack_bf16(vals[8 * g], vals[8 * g + 1]), pack_bf16(vals[8 * g + 2], vals[8 * g + 3]),
                                          pack_bf16(vals[8 * g + 4], vals[8 * g + 5]), pack_bf16(vals[8 * g + 6], vals[8 * g + 7]));
                    *reinterpret_cast<uint4 *>(base + ((size_t)((cc >> 3) + g) * NE + tid) * 16) = pk;
                }
            };
            // ---- h_0: embedding gather (or h_in) -> fp32 registers (requested first: the latency overlaps the staging)
            {
                const float *src = nullptr;
                if (live) {
                    if (a.atoms) {
                        int id = __ldg(a.atoms + (a.midx ? (long)__ldg(a.midx + molg) * a.N + atom : grow));
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
            // ---- stage the adjacency (fp32 global -> bf16 SW128 tiles [mol][e][i][j]) ----
            TSP(1);
            stage_adjacency<NE>(smem + C::OFF_ADJ, a.adj, a.adj_u8, tile, a.mb, a.N, tid, a.midx);
            TSP(2);
            {
#pragma unroll
                for (int cc = 0; cc < NC; cc += 32) {
                    if (a.h0_out) store_rows(a.h0_out, H, colbase + cc, &hreg[cc]);
                    if (V2 && a.Hs) store_rows(a.Hs, H, colbase + cc, &hreg[cc]);
                }
            }
            auto store_h_operand = [&](int t_next) {
                if (V2 && t_next < a.T) {
#pragma unroll
                    for (int cc = 0; cc < NC; cc += 16) store_native16(t_next, 3, cc, &hreg[cc]);
                }
#pragma unroll
                for (int g = 0; g < NC / 8; ++g) {
                    const int kk = colbase + 8 * g;
                    uint4 pk = make_uint4(pack_bf16(hreg[8 * g], hreg[8 * g + 1]), pack_bf16(hreg[8 * g + 2], hreg[8 * g + 3]),
                                          pack_bf16(hreg[8 * g + 4], hreg[8 * g + 5]), pack_bf16(hreg[8 * g + 6], hreg[8 * g + 7]));
                    *reinterpret_cast<uint4 *>(smem + C::OFF_H + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pk;
                }
            };
            TSP(3);
            store_h_operand(0);
            TSP(4);
            // degrees deg_e[atom] = sum_j A_e[atom][j]  (from the staged bf16 tile; needs the staging complete)
            asm volatile("bar.sync 1, %0;" ::"n"(NE));
            TSP(5);
            // each column group sums ONE bond type for its 128 rows (H = 128: four groups; H = 64: two groups x two types),
            // the four values per row are exchanged through the (idle) AH buffer
            float deg[4];
            {
                float *dsh = reinterpret_cast<float *>(smem + C::OFF_AH);       // [4][128]
                for (int e = hf; e < 4; e += EPW / 4) {
                    float s0 = 0.f, s1 = 0.f;
                    const uint8_t *rowp = smem + C::OFF_ADJ + (molslot * 4 + e) * ADJ_TILE_BYTES + atom * 128;
#pragma unroll
                    for (int ch = 0; ch < 8; ++ch) {
                        uint4 u = *reinterpret_cast<const uint4 *>(rowp + ((ch ^ (atom & 7)) << 4));     // any chunk order; rotated: conflict-free
                        const __nv_bfloat162 *b2 = reinterpret_cast<const __nv_bfloat162 *>(&u);
#pragma unroll
                        for (int x = 0; x < 4; ++x) { float2 f = __bfloat1622float2(b2[x]); s0 += f.x; s1 += f.y; }
                    }
                    dsh[e * 128 + row] = s0 + s1;
                }
                asm volatile("bar.sync 1, %0;" ::"n"(NE));
#pragma unroll
                for (int e = 0; e < 4; ++e) deg[e] = dsh[e * 128 + row];
                asm volatile("bar.sync 1, %0;" ::"n"(NE));      // AH is handed to the epilogue / staging again
            }
            TSP(6);
            warp_arrive(BAR(B_HREADY), lane);

            for (int t = 0; t < a.T; ++t, ++it) {
                const uint32_t par = it & 1;
                const bool stateful = a.stateful[t] != 0;
                const float *b3 = a.bias3[t];
#define TSF(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0 && it < 64) a.dbg[it * 16 + (i)] = clock64(); } while (0)
                TSF(0);
                if (t == a.T - 1 && tile + (int)gridDim.x < n_tiles) {      // next tile of this CTA: adjacency and atom ids towards L2
                    prefetch_adjacency_l2<NE>(a.adj, a.adj_u8, tile + gridDim.x, a.mb, a.N, tid, a.midx);
                    if (a.atoms && !a.midx && tid < 8) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.atoms + (long)(tile + gridDim.x) * 2 * a.N + tid * 32));
                }
                uint32_t v[32];
                // ---- E1: AH accumulators -> bf16 A-operand panels, one slot (64-column block of both bond types) at a time ----
                {
                    constexpr int W1 = 2048 / H;                   // columns per warp within a 64-column slot: 16 (H = 128) or 32 (H = 64)
                    const int cg = hf;                             // column group of this warp inside the slot
                    for (int p = 0; p < 2; ++p)
                        for (int cp = 0; cp < KP; ++cp) {
                            // the slot's previous use (same step, p - 1; or the previous step's p = 1) has been consumed by MMA-2
                            if (it > 0 || p > 0) mbar_wait(BAR(B_AHFREE + cp), p ^ 1u);
                            for (int mol = 0; mol < 2; ++mol) {
                                if (cp == 0) mbar_wait(BAR(B_D1 + mol), p);
                                tc_fence_after();
                                const int orow = mol * 64 + atom;  // row of (mol, atom) in the 128-row tile; TMEM lane half = bond type
                                uint8_t *pan = smem + C::OFF_AH + (molslot * KP + cp) * PANEL_BYTES;
                                const uint32_t tcol = t_lane + (2 + mol) * H + 64 * cp + cg * W1;
                                if (W1 == 16) {
                                    uint32_t w[16];
                                    tc_ld16(tcol, w);
                                    tc_wait_ld();
#pragma unroll
                                    for (int g = 0; g < 2; ++g) {
                                        uint4 pk = make_uint4(pack_bf16(__uint_as_float(w[8 * g]), __uint_as_float(w[8 * g + 1])),
                                                              pack_bf16(__uint_as_float(w[8 * g + 2]), __uint_as_float(w[8 * g + 3])),
                                                              pack_bf16(__uint_as_float(w[8 * g + 4]), __uint_as_float(w[8 * g + 5])),
                                                              pack_bf16(__uint_as_float(w[8 * g + 6]), __uint_as_float(w[8 * g + 7])));
                                        *reinterpret_cast<uint4 *>(pan + sw128(orow, cg * W1 + 8 * g)) = pk;
                                    }
                                } else {
                                    tc_ld32(tcol, v);
                                    tc_wait_ld();
#pragma unroll
                                    for (int g = 0; g < 4; ++g) {
                                        uint4 pk = make_uint4(pack_bf16(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])),
                                                              pack_bf16(__uint_as_float(v[8 * g + 2]), __uint_as_float(v[8 * g + 3])),
                                                              pack_bf16(__uint_as_float(v[8 * g + 4]), __uint_as_float(v[8 * g + 5])),
                                                              pack_bf16(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
                                        *reinterpret_cast<uint4 *>(pan + sw128(orow, cg * W1 + 8 * g)) = pk;
                                    }
                                }
                            }
                            warp_arrive(BAR(B_AHREADY + cp), lane);
                        }
                }
                // ---- E2: message m (+ bias through the degrees) -> bf16 operand (AH panels [0,KP)) ----
                TSF(1);
                mbar_wait(BAR(B_M), par);
                TSF(2);
                tc_fence_after();
                {
                    const float *mb_ = a.msg_b[t];
#pragma unroll
                    for (int cc = 0; cc < NC; cc += 32) {
                        tc_ld32(t_lane + 0 * H + colbase + cc, v);
                        tc_wait_ld();
                        float m[32];
#pragma unroll
                        for (int x = 0; x < 32; ++x) {
                            float4 b4 = __ldg(reinterpret_cast<const float4 *>(mb_) + colbase + cc + x);
                            m[x] = __uint_as_float(v[x]) + deg[0] * b4.x + deg[1] * b4.y + deg[2] * b4.z + deg[3] * b4.w;
                        }
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            const int kk = colbase + cc + 8 * g;
                            uint4 pk = make_uint4(pack_bf16(m[8 * g], m[8 * g + 1]), pack_bf16(m[8 * g + 2], m[8 * g + 3]),
                                                  pack_bf16(m[8 * g + 4], m[8 * g + 5]), pack_bf16(m[8 * g + 6], m[8 * g + 7]));
                            *reinterpret_cast<uint4 *>(smem + C::OFF_AH + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pk;
                        }
                    }
                }
                warp_arrive(BAR(B_XREADY), lane);
                TSF(3);
                // ---- E3: reset gate, r*h -> bf16 operand (AH panels [KP,2KP)) ----
                mbar_wait(BAR(B_R), par);
                TSF(4);
                tc_fence_after();
                if (stateful) {
#pragma unroll
                    for (int cc = 0; cc < NC; cc += 16) {
                        uint32_t w[16];
                        tc_ld16(t_lane + 1 * H + colbase + cc, w);
                        tc_wait_ld();
                        float r[16], rs[16];
#pragma unroll
                        for (int x = 0; x < 16; x += 4) {
                            const float4 b4 = __ldg(reinterpret_cast<const float4 *>(b3 + colbase + cc + x));
                            const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                            for (int y = 0; y < 4; ++y) {
                                r[x + y] = sigmoid_fast(__uint_as_float(w[x + y]) + bb[y]);
                                rs[x + y] = r[x + y] * hreg[cc + x + y];
                            }
                        }
                        if (V2) store_native16(t, 2, cc, r);
#pragma unroll
                        for (int g = 0; g < 2; ++g) {
                            const int kk = colbase + cc + 8 * g;
                            uint4 pk = make_uint4(pack_bf16(rs[8 * g], rs[8 * g + 1]), pack_bf16(rs[8 * g + 2], rs[8 * g + 3]),
                                                  pack_bf16(rs[8 * g + 4], rs[8 * g + 5]), pack_bf16(rs[8 * g + 6], rs[8 * g + 7]));
                            *reinterpret_cast<uint4 *>(smem + C::OFF_AH + (KP + (kk >> 6)) * PANEL_BYTES + sw128(row, kk & 63)) = pk;
                        }
                    }
                }
                warp_arrive(BAR(B_RSREADY), lane);
                TSF(5);
                // ---- E4: update gate + candidate -> new state ----
                mbar_wait(BAR(B_ZH), par);
                TSF(6);
                tc_fence_after();
#pragma unroll
                for (int cc = 0; cc < NC; cc += 16) {
                    uint32_t wz[16], wh[16];
                    tc_ld16(t_lane + 2 * H + colbase + cc, wz);
                    tc_ld16(t_lane + 3 * H + colbase + cc, wh);
                    tc_wait_ld();
                    float z[16], hb[16];
#pragma unroll
                    for (int x = 0; x < 16; x += 4) {
                        const float4 bz4 = __ldg(reinterpret_cast<const float4 *>(b3 + H + colbase + cc + x));
                        const float4 bh4 = __ldg(reinterpret_cast<const float4 *>(b3 + 2 * H + colbase + cc + x));
                        const float bz[4] = {bz4.x, bz4.y, bz4.z, bz4.w}, bh[4] = {bh4.x, bh4.y, bh4.z, bh4.w};
#pragma unroll
                        for (int y = 0; y < 4; ++y) {
                            z[x + y] = sigmoid_fast(__uint_as_float(wz[x + y]) + bz[y]);
                            hb[x + y] = tanh_fast(__uint_as_float(wh[x + y]) + bh[y]);
                            hreg[cc + x + y] = stateful ? fmaf(z[x + y], hb[x + y] - hreg[cc + x + y], hreg[cc + x + y]) : z[x + y] * hb[x + y];
                        }
                    }
                    if (V2) {
                        store_native16(t, 0, cc, z);
                        store_native16(t, 1, cc, hb);
                    }
                }
#pragma unroll
                for (int cc = 0; cc < NC; cc += 32) {
                    if (V2 && a.Hs) store_rows(a.Hs + (long)(t + 1) * rows_total * H, H, colbase + cc, &hreg[cc]);
                    if (t == a.T - 1 && a.h_out) store_rows(a.h_out, H, colbase + cc, &hreg[cc]);
                }
                TSF(7);
                if (t + 1 < a.T) {
                    store_h_operand(t + 1);
                    warp_arrive(BAR(B_HREADY), lane);
                } else {
                    tc_fence_before();
                    asm volatile("bar.sync 1, %0;" ::"n"(NE));   // everyone done with this tile's smem/TMEM
                }
            }
        }
    }
    // teardown
    tc_fence_before();
    __syncthreads();
    if (warp == EPW + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(C::TMEM_COLS));
    }
}

// ---------------------------------------------------------------- weight packing
// Builds the bf16, SW128-swizzled B-operand tiles ([H n][64 k]) of one step in consumption order:
//   [MMA-2: 4KP tiles, K = e*H + c'] [r: 2KP] [z: 2KP] [hbar: 2KP] [U: KP]   (stateless: no r, no U)
// and bias3 = [b_Wr+b_Ur | b_Wz(+b_Uz) | b_W(+b_U)].
struct PackArgs {
    int H, stateful;
    const float *msg_W;
    bmp_gru_t g;
    uint8_t *img;
    float *bias3;
};

__global__ void pack_kernel(const PackArgs p) {
    const int H = p.H, KP = H / 64;
    const int t_msg = 4 * KP, t_gate = 2 * KP;
    const int ntiles = p.stateful ? t_msg + 3 * t_gate + KP : t_msg + 2 * t_gate;
    const long total = (long)ntiles * H * 64;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int k = idx & 63, n = (idx >> 6) % H, tile = (int)(idx / (64L * H));
        float w;
        if (tile < t_msg) {                       // consumption order (pair p, 64-column block cb, bond type in the pair): K = e*H + c'
            const int pr = tile / (2 * KP), rem = tile % (2 * KP), cb = rem / 2, e = 2 * pr + (rem & 1), cp = cb * 64 + k;
            w = p.msg_W[((long)n * 4 + e) * H + cp];
        } else {
            int g = (tile - t_msg) / t_gate, kp = (tile - t_msg) % t_gate;
            if (!p.stateful) g += 1;              // stateless images start at the z block
            if (g < 3) {
                const int K = kp * 64 + k;        // column of the (H, 2H) gate matrix
                const float *W = g == 0 ? p.g.W_r : (g == 1 ? p.g.W_z : p.g.W);
                w = W[(long)n * 2 * H + K];
                if (p.stateful && K < H && g < 2) w += (g == 0 ? p.g.U_r : p.g.U_z)[(long)n * H + K];   // state == h: fold U
            } else {                              // U tiles (tile index past the three gate blocks)
                const int K = (tile - t_msg - 3 * t_gate) * 64 + k;
                w = p.g.U[(long)n * H + K];
            }
        }
        __nv_bfloat16 b = __float2bfloat16_rn(w);
        const uint32_t off = (uint32_t)n * 128u + ((((uint32_t)(k >> 3) ^ ((uint32_t)n & 7u)) << 4) | (((uint32_t)k & 7u) << 1));
        *reinterpret_cast<__nv_bfloat16 *>(p.img + (size_t)tile * H * 128 + off) = b;
    }
    if (blockIdx.x == 0)
        for (int c = threadIdx.x; c < H; c += blockDim.x) {
            p.bias3[c] = p.stateful ? p.g.b_Wr[c] + p.g.b_Ur[c] : 0.f;
            p.bias3[H + c] = p.g.b_Wz[c] + (p.stateful ? p.g.b_Uz[c] : 0.f);
            p.bias3[2 * H + c] = p.g.b_W[c] + (p.stateful ? p.g.b_U[c] : 0.f);
        }
}

static size_t image_bytes(int H) { return (size_t)(11 * (H / 64)) * H * 128 + 3 * H * sizeof(float) + 256; }

}  // namespace tc
}  // namespace bmp

using namespace bmp;

extern "C" size_t bmp_ggnn_stash2_bytes(int mb, int hidden, int n_steps) {
    if (hidden != 64 && hidden != 128) return 0;
    return tc::Stash2::bytes((mb + 1) / 2, hidden, n_steps);
}

size_t bmp_ggnn_tc256_workspace_bytes(int n_steps);                   // ggnn_tc256.cu (hidden 256, forward only)
int bmp_ggnn_forward_tc256(const bmp_ggnn_fwd_t *a, void *stream);

extern "C" size_t bmp_ggnn_tc_workspace_bytes(int hidden, int n_steps) {
    if (hidden == 256) return bmp_ggnn_tc256_workspace_bytes(n_steps);
    if (hidden != 64 && hidden != 128) return 0;
    return tc::image_bytes(hidden) * (size_t)n_steps + 2048;
}

extern long long *g_tc_dbg_fwd;
long long *g_tc_dbg_fwd = nullptr;
extern "C" void bmp_debug_set_buffer_fwd(void *p) { g_tc_dbg_fwd = (long long *)p; }

int bmp_ggnn_forward_tc(const bmp_ggnn_fwd_t *a, void *stream) {
    const int H = a->hidden, T = a->n_steps;
    if (H == 256) return bmp_ggnn_forward_tc256(a, stream);
    if (H != 64 && H != 128) { set_error("BMP_MODE_BF16: hidden=%d not supported (64, 128; 256 forward-only)", H); return BMP_ESHAPE; }
    if (a->n_edge != 4) { set_error("BMP_MODE_BF16: n_edge=%d not supported (4)", a->n_edge); return BMP_ESHAPE; }
    if (a->mb <= 0 || T <= 0 || T > BMP_MAX_STEPS || a->n_atoms <= 0 || a->n_atoms > BMP_MAX_ATOMS) {
        set_error("BMP_MODE_BF16: bad shape mb=%d T=%d N=%d", a->mb, T, a->n_atoms);
        return BMP_ESHAPE;
    }
    if (a->state_in) { set_error("BMP_MODE_BF16: an external GRU state is not supported (state must equal h)"); return BMP_ESHAPE; }
    if (a->Ms || a->Gs || a->RSs || (a->Hs && !a->stash2)) {
        set_error("BMP_MODE_BF16: the training tape is the bf16 panel stash (stash2); Ms / Gs / RSs must be NULL and Hs needs stash2");
        return BMP_EINVAL;
    }
    if (!a->tc_workspace || a->tc_workspace_bytes < bmp_ggnn_tc_workspace_bytes(H, T)) {
        set_error("BMP_MODE_BF16: tc_workspace of >= %zu bytes required", bmp_ggnn_tc_workspace_bytes(H, T));
        return BMP_EINVAL;
    }
    if (!aligned16({a->h_in, a->embed_W, a->adj, a->h_out, a->h0_out, a->Hs, a->tc_workspace})) {
        set_error("BMP_MODE_BF16: buffers must be 16-byte aligned");
        return BMP_EINVAL;
    }
    cudaStream_t st = (cudaStream_t)stream;
    tc::Args k = {};
    k.mb = a->mb; k.N = a->n_atoms; k.T = T; k.n_types = a->n_atom_types;
    k.atoms = a->atoms; k.embed_W = a->embed_W; k.h_in = a->h_in; k.adj = a->adj; k.adj_u8 = a->adj_u8;
    k.h_out = a->h_out; k.h0_out = a->h0_out; k.Hs = a->Hs;
    k.dbg = g_tc_dbg_fwd;
    k.midx = a->mol_index;
    if (a->mol_index && !a->atoms) { set_error("BMP_MODE_BF16: mol_index needs atom ids (a drug table), not h_in"); return BMP_EINVAL; }
    if (a->stash2) k.st.carve(a->stash2, (a->mb + 1) / 2, H, T);
    uint8_t *ws = (uint8_t *)(((uintptr_t)a->tc_workspace + 255) & ~(uintptr_t)255);
    const size_t ib = tc::image_bytes(H);
    int n_img = 0;
    for (int t = 0; t < T; ++t) {
        if (!a->msg_W[t] || !a->msg_b[t] || !a->gru[t].W_z || !a->gru[t].W) { set_error("BMP_MODE_BF16: null parameter at step %d", t); return BMP_EINVAL; }
        if (((uintptr_t)a->msg_b[t]) & 15) { set_error("BMP_MODE_BF16: msg_b must be 16-byte aligned"); return BMP_EINVAL; }
        int found = -1;
        for (int u = 0; u < t; ++u)
            if (a->msg_W[u] == a->msg_W[t] && same_gru(a->gru[u], a->gru[t]) &&
                (a->stateful[u] != 0) == (a->stateful[t] != 0)) { found = u; break; }
        k.stateful[t] = a->stateful[t] != 0;
        k.msg_b[t] = a->msg_b[t];
        if (found >= 0) { k.img[t] = k.img[found]; k.bias3[t] = k.bias3[found]; continue; }
        uint8_t *img = ws + (size_t)n_img * ib;
        float *bias3 = reinterpret_cast<float *>(img + (size_t)(11 * (H / 64)) * H * 128);
        tc::PackArgs p;
        p.H = H; p.stateful = k.stateful[t]; p.msg_W = a->msg_W[t]; p.g = a->gru[t]; p.img = img; p.bias3 = bias3;
        if (!a->tc_images_ready) {
            tc::pack_kernel<<<64, 256, 0, st>>>(p);
            count_launch();
        }
        k.img[t] = img; k.bias3[t] = bias3;
        ++n_img;
    }
    int rc = check_launch("pack_kernel");
    if (rc) return rc;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int n_tiles = (a->mb + 1) / 2;
    const int grid = n_tiles < sms ? n_tiles : sms;
#define LAUNCH_FWD(HH, VV)                                                                                               \
    do {                                                                                                                 \
        cudaFuncSetAttribute(tc::ggnn_tc_kernel<HH, VV>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Cfg<HH>::SMEM_BYTES); \
        tc::ggnn_tc_kernel<HH, VV><<<grid, 32 * (HH / 8 + 2), tc::Cfg<HH>::SMEM_BYTES, st>>>(k);                          \
    } while (0)
    ProfScope prof(BMP_PROF_GGNN_FWD, st);
    if (H == 64) { if (a->stash2) LAUNCH_FWD(64, true); else LAUNCH_FWD(64, false); }
    else { if (a->stash2) LAUNCH_FWD(128, true); else LAUNCH_FWD(128, false); }
#undef LAUNCH_FWD
    count_launch();
    return check_launch("ggnn_tc_kernel");
}
