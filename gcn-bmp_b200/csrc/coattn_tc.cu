// coattn_tc.cu -- fine-grained co-attention with its contractions on tcgen05 (BMP_MODE_BF16).
//
// Same math as coattn.cu (nie_coattention.py:335-396 / vqa_parallel_coattention.py:42-103); one persistent CTA
// per SM, a work item = one drug pair.  The pair's atom states form ONE bf16 operand tile
//   X = [a1 ; a2]  (rows 0-63: atoms_1, rows 64-127: atoms_2, K = hidden, 128-byte swizzle)
// and every (64 x H x H)-sized contraction becomes a single M = 128 UMMA group with fp32 accumulation in TMEM:
//   G1    [X W^T | X lt_1^T | X V1 | X lt_2^T | X V2]     N = H + 32: Q = a2 W^T, head projections, V terms
//   G2    C^T = a1 Q^T                                     N = 64
//   S     S  = a1 W                (backward)              N = H
//   R     R  = dC^T a2             (backward, B = X rows 64.. read MN-major)
//   A2    d a2 = [dC | dlt_2 | rsum] [S ; lt_2 ; V2]       (K = 64 + 16: the rank-hd and rank-1 terms ride along)
//   A1    d a1 = [R | dlt_1 | cs] [W | lt_1 | V1]^T        (K = H + 16)
// The softmaxes, head non-linearity and pooling between them are the scalar phases of coattn.cu on 16 warps.
// Weights stream from L2 as pre-packed bf16 tiles (cp.async.bulk + mbarrier ring); warp 16 produces, warp 17
// issues the MMAs, warps 0-15 own TMEM lane quarter (warp % 4) and column group (warp / 4).
#include "tc_common.cuh"
#include "det.cuh"

namespace bmp {
namespace ctc {
using namespace tc;

constexpr int EPW = 16, NE = 32 * EPW, NT = NE + 64;
constexpr int CLD = 68;       // ld of the C^T map (float4 rows, conflict-free lane-per-row stores)
constexpr int PLD = 65;       // ld of the scalar-accessed probability maps
constexpr int MAXHD = 15;     // head projections share a 16-column group with the V term (column 15)
constexpr int STAGES = 2;

#define EPI_SYNC() asm volatile("bar.sync 1, %0;" ::"n"(NE) : "memory")
#define CTS(i) do { if (a.dbg && blockIdx.x == 0 && tid == 0 && it == 1) a.dbg[i] = clock64(); } while (0)

struct Args {
    int mb, n1, n2, O, head, act, pool;      // pool: PoolingFineCoattention (scores = means of C, no head path; head = 0)
    const float *atoms_1, *atoms_2, *b, *wa_1, *wa_2, *W_j, *b_j, *lt_2, *V2;
    const uint8_t *img1, *img2, *img1x;      // packed weight tiles
    float *c1, *c2;                          // forward outputs
    // backward
    const float *dc1, *dc2;
    float *R, *P1, *P2, *DL1, *DL2, *d_a1, *d_a2;
    float *d_W, *d_lt_1, *d_lt_2, *d_V1, *d_V2, *d_b, *d_wa_1, *d_wa_2;
    CoDet det;                   // deterministic mode: this CTA's slot takes the flush below instead of the atomics
    long long *dbg;              // optional phase timestamps of CTA 0, second pair (tools/co_timeline.py)
};

template <int H, bool BWD>
struct Cfg {
    static constexpr int KP = H / 64;
    static constexpr int W1_TILE = (H + 32) * 128;        // k-tile of img1: H + 32 rows (n) x 64 bf16 (k)
    static constexpr int WH_TILE = H * 128;
    static constexpr int OFF_XP = 0;                                   // X panels
    static constexpr int OFF_QP = OFF_XP + KP * PANEL_BYTES;           // Q blocks [KP][64 i][64 h]; backward: R extension panel
    static constexpr int OFF_W = OFF_QP + PANEL_BYTES;
    static constexpr int OFF_SP = OFF_W + STAGES * W1_TILE;            // S panels (+ static rows 64..79: lt_2, V2), then R panels (rows 0-63)
    static constexpr int OFF_DP = OFF_SP + (BWD ? KP * PANEL_BYTES : 0);   // [dC^T ; dC] panel + extension panel; then store staging
    static constexpr int OFF_F = OFF_DP + (BWD ? 2 * PANEL_BYTES : 0);     // fp32 area (carved at run time: depends on head)
    static constexpr int TMEM_COLS = BWD ? 512 : 256;
    // TMEM columns.  Per pair: D1 [0, H+32) -> R [0, H) -> d a1 [0, H) ; C^T [192, 256) ; S [256, 256+H) -> d a2 [256, 256+H).
    // Persistent over the CTA's pairs: [d lt_1 | d V1] [160, 176), [d lt_2 | d V2] [176, 192), d W [384, 384+H).
    static constexpr uint32_t COL_D1 = 0, COL_D2 = 192, COL_R = 0, COL_A1 = 0, COL_S = 256, COL_A2 = 256, COL_X1 = 160, COL_X2 = 176, COL_DW = 384;
};

__host__ __device__ inline int f32_floats(int H, int hd, bool bwd) {
    hd = hd <= 8 ? 8 : 16;                          // padded head count HP
    int n = AT * CLD + 2 * AT * PLD + 4;            // Cs, L1t, L2p
    n += 4 * hd * AT;                               // lt1, lt2, H1, H2
    n += 4 * AT + 2 * H;                            // attn1, attn2, v1, v2, p1, p2
    n += 4 * AT + 16 * AT;                          // m2/is2/m1/is1 (later t1,t2,cs,rsum), partial stats
    if (bwd) n += 2 * H + 2 * hd * AT + 2 * 16 + 4;   // dp1, dp2, dpre1, dpre2, gwa1, gwa2, gb
    return (n + 3) & ~3;
}
template <int H, bool BWD>
__host__ __device__ inline size_t smem_bytes(int hd) {
    return (size_t)Cfg<H, BWD>::OFF_F + (size_t)f32_floats(H, hd, BWD) * 4 + 256 + 1024;
}

__device__ __forceinline__ float warp_sum(float v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float bf16_at(const uint8_t *panels, int row, int col) {
    return __bfloat162float(*reinterpret_cast<const __nv_bfloat16 *>(panels + (col >> 6) * PANEL_BYTES + sw128(row, col & 63)));
}
__device__ __forceinline__ uint4 pack8(const float *v) {
    return make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
}

// HP = padded head count (8 or 16): the head arrays are atom-major [64][HP] with the heads contiguous, so every
// rank-head product is a few 16-byte loads per atom (mostly warp-wide broadcasts).
template <int H, bool BWD, int HP>
__global__ void __launch_bounds__(NT, 1) coattn_tc_kernel(const Args a) {
    using C = Cfg<H, BWD>;
    constexpr int HS = HP, HQ = HP / 4;
    constexpr int KP = C::KP;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_xp = sbase + C::OFF_XP, s_qp = sbase + C::OFF_QP, s_w = sbase + C::OFF_W, s_sp = sbase + C::OFF_SP,
                   s_dp = sbase + C::OFF_DP;
    uint8_t *XP = smem + C::OFF_XP, *QP = smem + C::OFF_QP, *SP = smem + C::OFF_SP, *DP = smem + C::OFF_DP;
    const int hd = a.head, N1 = a.n1, N2 = a.n2, O = a.O;
    const bool pool = a.pool != 0;
    // ---- fp32 area
    float *fp = reinterpret_cast<float *>(smem + C::OFF_F);
    float *Cs = fp; fp += AT * CLD;
    float *L1t = fp; fp += AT * PLD;
    float *L2p = fp; fp += AT * PLD + 4;
    float *lt1 = fp; fp += HS * AT;
    float *lt2 = fp; fp += HS * AT;
    float *H1 = fp; fp += HS * AT;
    float *H2 = fp; fp += HS * AT;
    float *attn1 = fp; fp += AT;
    float *attn2 = fp; fp += AT;
    float *v1 = fp; fp += AT;
    float *v2 = fp; fp += AT;
    float *p1 = fp; fp += H;
    float *p2 = fp; fp += H;
    float *st4 = fp; fp += 4 * AT;          // forward: m2 | 1/s2 | m1 | 1/s1 ; backward: t1 | t2 | cs | rsum
    float *part = fp; fp += 16 * AT;        // partial column statistics [2][8][64]
    float *dp1 = fp, *dp2 = fp + H, *dpre1 = fp + 2 * H, *dpre2 = dpre1 + HS * AT;
    float *gwa1 = dpre2 + HS * AT, *gwa2 = gwa1 + 16, *gb = gwa2 + 16;
    const int f32n = f32_floats(H, hd, BWD);
    const uint32_t s_bar = sbase + C::OFF_F + f32n * 4;
    auto BAR = [&](int i) { return s_bar + 8u * i; };
    constexpr int B_FULL = 0, B_EMPTY = 2, B_XRDY = 4, B_G1 = 5, B_S = 6, B_QRDY = 7, B_G2 = 8, B_DRDY = 9, B_R = 10,
                  B_A2 = 11, B_RRDY = 12, B_A1 = 13, NBAR = 14;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + C::OFF_F + f32n * 4 + 8 * NBAR + 8);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(BAR(B_FULL + s), 1); mbar_init(BAR(B_EMPTY + s), 1); }
        mbar_init(BAR(B_XRDY), EPW);
        mbar_init(BAR(B_G1), 1);
        mbar_init(BAR(B_S), 1);
        mbar_init(BAR(B_QRDY), EPW);
        mbar_init(BAR(B_G2), 1);
        mbar_init(BAR(B_DRDY), EPW);
        mbar_init(BAR(B_R), 1);
        mbar_init(BAR(B_A2), 1);
        mbar_init(BAR(B_RRDY), EPW);
        mbar_init(BAR(B_A1), 1);
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
        // ===================== TMA producer: weight tiles in consumption order
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            auto put = [&](const uint8_t *src, uint32_t bytes) {
                mbar_wait(BAR(B_EMPTY + stage), phase ^ 1);
                mbar_expect_tx(BAR(B_FULL + stage), bytes);
                tma_bulk_g2s(s_w + stage * C::W1_TILE, src, bytes, BAR(B_FULL + stage));
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            };
            for (int pair = blockIdx.x; pair < a.mb; pair += gridDim.x) {
                for (int kt = 0; kt < KP; ++kt) put(a.img1 + (size_t)kt * C::W1_TILE, C::W1_TILE);
                if (BWD) {
                    for (int kt = 0; kt < KP; ++kt) put(a.img2 + (size_t)kt * C::WH_TILE, C::WH_TILE);
                    for (int kt = 0; kt < KP; ++kt) put(a.img1 + (size_t)kt * C::W1_TILE, C::WH_TILE);   // rows [0, H): W
                    put(a.img1x, C::WH_TILE);
                }
            }
        }
    } else if (warp == EPW + 1) {
        // ===================== MMA issuer
        if (lane == 0) {
            constexpr uint32_t ID_G1 = idesc2(H + 32, 0, 0), ID_H = idesc2(H, 0, 0), ID_64 = idesc2(64, 0, 0), ID_HMN = idesc2(H, 0, 1),
                               ID_WMN = idesc2(H, 1, 1), ID_X = idesc2(16, 1, 1);
            uint32_t stage = 0, phase = 0, it = 0;
            // one weight tile against the K-major A panel at a_addr: ksteps k-steps of 16
            auto mma_wtile = [&](uint32_t a_addr, uint32_t dcol, uint32_t id, bool first, int ksteps) {
                mbar_wait(BAR(B_FULL + stage), phase);
                tc_fence_after();
                const uint32_t b_addr = s_w + stage * C::W1_TILE;
                for (int k = 0; k < ksteps; ++k)
                    tc_mma(tmem + dcol, desc_kmajor(a_addr + k * 32), desc_kmajor(b_addr + k * 32), id, (first && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_EMPTY + stage));
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            };
            for (int pair = blockIdx.x; pair < a.mb; pair += gridDim.x, ++it) {
                const uint32_t par = it & 1;
                mbar_wait(BAR(B_XRDY), par);
                tc_fence_after();
                for (int kp = 0; kp < KP; ++kp) mma_wtile(s_xp + kp * PANEL_BYTES, C::COL_D1, ID_G1, kp == 0, 4);
                tc_commit(BAR(B_G1));
                if (BWD) {
                    for (int kp = 0; kp < KP; ++kp) mma_wtile(s_xp + kp * PANEL_BYTES, C::COL_S, ID_H, kp == 0, 4);
                    tc_commit(BAR(B_S));
                }
                mbar_wait(BAR(B_QRDY), par);
                tc_fence_after();
                for (int kp = 0; kp < KP; ++kp)
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        tc_mma(tmem + C::COL_D2, desc_kmajor(s_xp + kp * PANEL_BYTES + k * 32), desc_kmajor(s_qp + kp * 8192 + k * 32), ID_64,
                               (kp == 0 && k == 0) ? 0u : 1u);
                tc_commit(BAR(B_G2));
                if (BWD) {
                    const uint32_t acc = it ? 1u : 0u;            // persistent parameter-gradient accumulators
                    mbar_wait(BAR(B_DRDY), par);
                    tc_fence_after();
#pragma unroll
                    for (int k = 0; k < 4; ++k)       // R = dC^T a2: B = rows 64.. of the X panels, MN-major
                        tc_mma(tmem + C::COL_R, desc_kmajor(s_dp + k * 32), desc_mnmajor(s_xp + 64 * 128 + k * 16 * 128), ID_HMN, k ? 1u : 0u);
                    tc_commit(BAR(B_R));
#pragma unroll
                    for (int k = 0; k < 5; ++k)       // d a2 = [dC | ext] [S ; ext rows]
                        tc_mma(tmem + C::COL_A2, desc_kmajor(k < 4 ? s_dp + k * 32 : s_dp + PANEL_BYTES), desc_mnmajor(s_sp + k * 16 * 128), ID_HMN,
                               k ? 1u : 0u);
#pragma unroll
                    for (int k = 0; k < 4; ++k)       // [d lt_2 | d V2]^T += a2^T [dlt_2 | rsum]   (both operands MN-major)
                        tc_mma(tmem + C::COL_X2, desc_mnmajor(s_xp + 64 * 128 + k * 16 * 128), desc_mnmajor(s_dp + PANEL_BYTES + 64 * 128 + k * 16 * 128),
                               ID_X, (acc || k) ? 1u : 0u);
                    tc_commit(BAR(B_A2));
                    mbar_wait(BAR(B_RRDY), par);
                    tc_fence_after();
                    for (int kp = 0; kp < KP; ++kp) mma_wtile(s_sp + kp * PANEL_BYTES, C::COL_A1, ID_H, kp == 0, 4);
                    mma_wtile(s_qp, C::COL_A1, ID_H, false, 1);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {     // d W += a1^T R ; [d lt_1 | d V1]^T += a1^T [dlt_1 | cs]
                        tc_mma(tmem + C::COL_DW, desc_mnmajor(s_xp + k * 16 * 128), desc_mnmajor(s_sp + k * 16 * 128), ID_WMN, (acc || k) ? 1u : 0u);
                        tc_mma(tmem + C::COL_X1, desc_mnmajor(s_xp + k * 16 * 128), desc_mnmajor(s_qp + k * 16 * 128), ID_X, (acc || k) ? 1u : 0u);
                    }
                    tc_commit(BAR(B_A1));
                }
            }
        }
    } else {
        // ===================== 16 epilogue / scalar warps
        const int q = warp & 3, cg = warp >> 2;
        const int row = 32 * q + lane;
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
        uint32_t it = 0;
        if (BWD) {
            for (int i = tid; i < 36; i += NE) gwa1[i] = 0.f;
            // static part of the operands: rows 64..79 of the S panels = [lt_2 ; 0 ; V2], extension panel rows 0-63 = 0
            for (int idx = tid; idx < 16 * (H / 8); idx += NE) {
                const int e = idx / (H / 8), c8 = idx % (H / 8);
                float v[8];
#pragma unroll
                for (int x = 0; x < 8; ++x) {
                    const int k = c8 * 8 + x;
                    v[x] = e < hd ? a.lt_2[(long)e * H + k] : (e == 15 ? a.V2[k] : 0.f);
                }
                *reinterpret_cast<uint4 *>(SP + (c8 >> 3) * PANEL_BYTES + sw128(64 + e, (c8 & 7) * 8)) = pack8(v);
            }
            for (int idx = tid; idx < 128 * 8; idx += NE)
                *reinterpret_cast<uint4 *>(DP + PANEL_BYTES + idx * 16) = make_uint4(0, 0, 0, 0);
        }
        for (int pair = blockIdx.x; pair < a.mb; pair += gridDim.x, ++it) {
            const uint32_t par = it & 1;
            const long r1 = (long)pair * N1, r2 = (long)pair * N2;
            EPI_SYNC();
            CTS(0);
            // ---- X = [a1 ; a2] -> bf16 operand panels
            {
                constexpr int PER = 128 * (H / 8) / NE;         // 16-byte operand chunks per thread
                float4 x0[PER], x1[PER];
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int idx = tid + u * NE, r = idx / (H / 8), c8 = idx % (H / 8), n = r & 63;
                    const bool live = r < 64 ? n < N1 : n < N2;
                    x0[u] = x1[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (live) {
                        const float4 *src = reinterpret_cast<const float4 *>((r < 64 ? a.atoms_1 + (r1 + n) * H : a.atoms_2 + (r2 + n) * H) + c8 * 8);
                        x0[u] = __ldg(src);
                        x1[u] = __ldg(src + 1);
                    }
                }
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int idx = tid + u * NE, r = idx / (H / 8), c8 = idx % (H / 8);
                    *reinterpret_cast<uint4 *>(XP + (c8 >> 3) * PANEL_BYTES + sw128(r, (c8 & 7) * 8)) =
                        make_uint4(pack_bf16(x0[u].x, x0[u].y), pack_bf16(x0[u].z, x0[u].w), pack_bf16(x1[u].x, x1[u].y), pack_bf16(x1[u].z, x1[u].w));
                }
            }
            warp_arrive(BAR(B_XRDY), lane);
            CTS(1);
            if (pair + (int)gridDim.x < a.mb) {       // next pair of this CTA: its atom states towards L2
                const long np = pair + gridDim.x;
                const char *b1 = reinterpret_cast<const char *>(a.atoms_1 + np * N1 * H), *b2 = reinterpret_cast<const char *>(a.atoms_2 + np * N2 * H);
                for (int off = tid * 128; off < N1 * H * 4; off += NE * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(b1 + off));
                for (int off = tid * 128; off < N2 * H * 4; off += NE * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(b2 + off));
            }
            // ---- G1 epilogue: Q (rows of a2) -> bf16 B-operand blocks; head projections and V terms -> fp32
            mbar_wait(BAR(B_G1), par);
            tc_fence_after();
            CTS(2);
            if (q >= 2 && cg * 32 < H) {
                uint32_t v[32];
                tc_ld32(t_lane + C::COL_D1 + cg * 32, v);
                tc_wait_ld();
                const int i = row - 64;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const int kk = cg * 32 + 8 * g;
                    float f[8];
#pragma unroll
                    for (int x = 0; x < 8; ++x) f[x] = __uint_as_float(v[8 * g + x]);
                    *reinterpret_cast<uint4 *>(QP + (kk >> 6) * 8192 + sw128(i, kk & 63)) = pack8(f);
                }
            }
            if (cg == (H == 128 ? 0 : 3)) {
                uint32_t w[16];
                tc_ld16(t_lane + C::COL_D1 + H + (q >= 2 ? 16 : 0), w);
                tc_wait_ld();
                const int n = row & 63;
                float *lt = (q >= 2 ? lt2 : lt1) + n * HS;      // columns >= head are zero (zero weight rows); 15 is the V term
#pragma unroll
                for (int d4 = 0; d4 < HQ; ++d4)
                    *reinterpret_cast<float4 *>(lt + 4 * d4) = make_float4(__uint_as_float(w[4 * d4]), __uint_as_float(w[4 * d4 + 1]), __uint_as_float(w[4 * d4 + 2]),
                                                                           4 * d4 + 3 == 15 ? 0.f : __uint_as_float(w[4 * d4 + 3]));
                (q >= 2 ? v2 : v1)[n] = __uint_as_float(w[15]);
            }
            if (BWD) {
                // ---- S = a1 W -> bf16 panel (B operand of the d a2 contraction, read MN-major)
                mbar_wait(BAR(B_S), par);
                tc_fence_after();
                if (q < 2 && cg * 32 < H) {
                    uint32_t v[32];
                    tc_ld32(t_lane + C::COL_S + cg * 32, v);
                    tc_wait_ld();
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const int kk = cg * 32 + 8 * g;
                        float f[8];
#pragma unroll
                        for (int x = 0; x < 8; ++x) f[x] = __uint_as_float(v[8 * g + x]);
                        *reinterpret_cast<uint4 *>(SP + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pack8(f);
                    }
                }
            }
            warp_arrive(BAR(B_QRDY), lane);
            EPI_SYNC();
            CTS(3);                       // v1 / v2 / lt visible to every warp
            // ---- G2 epilogue: C^T[j][i] = act(a1_j . Q_i + v1[j] + v2[i] + b)
            mbar_wait(BAR(B_G2), par);
            tc_fence_after();
            CTS(4);
            if (q < 2) {
                uint32_t w[16];
                tc_ld16(t_lane + C::COL_D2 + cg * 16, w);
                tc_wait_ld();
                const float base = v1[row] + a.b[0];
#pragma unroll
                for (int x = 0; x < 16; x += 4) {
                    const float4 vv = *reinterpret_cast<const float4 *>(v2 + cg * 16 + x);
                    float4 o;
                    o.x = act_fast(a.act, __uint_as_float(w[x]) + base + vv.x);
                    o.y = act_fast(a.act, __uint_as_float(w[x + 1]) + base + vv.y);
                    o.z = act_fast(a.act, __uint_as_float(w[x + 2]) + base + vv.z);
                    o.w = act_fast(a.act, __uint_as_float(w[x + 3]) + base + vv.w);
                    *reinterpret_cast<float4 *>(Cs + row * CLD + cg * 16 + x) = o;
                }
            }
            tc_fence_before();
            EPI_SYNC();
            CTS(5);
            if (pool) {
                // PoolingFineCoattention: attn_1 = softmax_j(mean_i C), attn_2 = softmax_i(mean_j C)
                if (tid < AT) {
                    float sm = 0.f;
                    for (int j = 0; j < N1; ++j) sm += Cs[j * CLD + tid];
                    attn2[tid] = sm / (float)N1;
                }
                for (int j = warp; j < AT; j += EPW) {
                    const float sm = warp_sum((lane < N2 ? Cs[j * CLD + lane] : 0.f) + (lane + 32 < N2 ? Cs[j * CLD + lane + 32] : 0.f));
                    if (lane == 0) attn1[j] = sm / (float)N2;
                }
            } else {
            // ---- softmax statistics: over i for every j (rows of C^T, one warp each), over j for every i (8 partials)
            float *m2 = st4, *is2 = st4 + AT, *m1 = st4 + 2 * AT, *is1 = st4 + 3 * AT;
            {
                const int i = tid & 63, pt = tid >> 6;
                float m = -INFINITY, s = 0.f;
                if (i < N2) {
                    float c[8];
#pragma unroll
                    for (int x = 0; x < 8; ++x) c[x] = (8 * pt + x < N1) ? Cs[(8 * pt + x) * CLD + i] : -INFINITY;
#pragma unroll
                    for (int x = 0; x < 8; ++x) m = fmaxf(m, c[x]);
#pragma unroll
                    for (int x = 0; x < 8; ++x) s += c[x] > -INFINITY ? __expf(c[x] - m) : 0.f;
                }
                part[pt * AT + i] = m;
                part[8 * AT + pt * AT + i] = s;
                {   // rows j = warp + 16 k: the four reductions run in lockstep (independent shuffle chains)
                    float x0[4], x1[4], mx[4], sm[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int j = warp + EPW * k;
                        x0[k] = (j < N1 && lane < N2) ? Cs[j * CLD + lane] : -INFINITY;
                        x1[k] = (j < N1 && lane + 32 < N2) ? Cs[j * CLD + lane + 32] : -INFINITY;
                        mx[k] = fmaxf(x0[k], x1[k]);
                    }
#pragma unroll
                    for (int o = 16; o; o >>= 1)
#pragma unroll
                        for (int k = 0; k < 4; ++k) mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        sm[k] = (x0[k] > -INFINITY ? __expf(x0[k] - mx[k]) : 0.f) + (x1[k] > -INFINITY ? __expf(x1[k] - mx[k]) : 0.f);
#pragma unroll
                    for (int o = 16; o; o >>= 1)
#pragma unroll
                        for (int k = 0; k < 4; ++k) sm[k] += __shfl_xor_sync(0xffffffffu, sm[k], o);
                    if (lane < 4) {
                        const float mm = lane == 0 ? mx[0] : (lane == 1 ? mx[1] : (lane == 2 ? mx[2] : mx[3]));
                        const float ss = lane == 0 ? sm[0] : (lane == 1 ? sm[1] : (lane == 2 ? sm[2] : sm[3]));
                        m2[warp + EPW * lane] = mm;
                        is2[warp + EPW * lane] = ss > 0.f ? 1.f / ss : 0.f;
                    }
                }
            }
            EPI_SYNC();
            if (tid < AT) {
                float m = -INFINITY, s = 0.f;
#pragma unroll
                for (int pt = 0; pt < 8; ++pt) m = fmaxf(m, part[pt * AT + tid]);
#pragma unroll
                for (int pt = 0; pt < 8; ++pt) {
                    const float pm = part[pt * AT + tid];
                    s += pm > -INFINITY ? part[8 * AT + pt * AT + tid] * __expf(pm - m) : 0.f;
                }
                m1[tid] = m;
                is1[tid] = s > 0.f ? 1.f / s : 0.f;
            }
            EPI_SYNC();
            for (int idx = tid; idx < AT * AT; idx += NE) {
                const int j = idx >> 6, i = idx & 63;
                const bool live = j < N1 && i < N2;
                const float c = Cs[j * CLD + i];
                L2p[j * PLD + i] = live ? __expf(c - m2[j]) * is2[j] : 0.f;
                L1t[i * PLD + j] = live ? __expf(c - m1[i]) * is1[i] : 0.f;
            }
            EPI_SYNC();
            CTS(6);
            // ---- H_1[j][:] = tanh(lt_1[j][:] + sum_i L_1[j][i] lt_2[i][:]) ; H_2 likewise.  Four threads per atom, each a
            // quarter of the inner index (interleaved), all heads in registers; quad shuffle reduction.
            {
                const int which = tid >> 8, n = (tid >> 2) & 63, pt = tid & 3;
                const float *Lw = which ? L2p : L1t, *other = which ? lt1 : lt2;
                float acc[HP];
#pragma unroll
                for (int d = 0; d < HP; ++d) acc[d] = 0.f;
#pragma unroll 4
                for (int mm = 0; mm < 16; ++mm) {
                    const int m = 4 * mm + pt;
                    const float l = Lw[m * PLD + n];
#pragma unroll
                    for (int d4 = 0; d4 < HQ; ++d4) {
                        const float4 r4 = *reinterpret_cast<const float4 *>(other + m * HS + 4 * d4);
                        acc[4 * d4] = fmaf(l, r4.x, acc[4 * d4]); acc[4 * d4 + 1] = fmaf(l, r4.y, acc[4 * d4 + 1]);
                        acc[4 * d4 + 2] = fmaf(l, r4.z, acc[4 * d4 + 2]); acc[4 * d4 + 3] = fmaf(l, r4.w, acc[4 * d4 + 3]);
                    }
                }
#pragma unroll
                for (int d = 0; d < HP; ++d) {
                    acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], 1);
                    acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], 2);
                }
                const float *self = (which ? lt2 : lt1) + n * HS;
                float *Hk = (which ? H2 : H1) + n * HS;
#pragma unroll
                for (int d4 = 0; d4 < HQ; ++d4) {       // lane pt finishes head 4*d4 + pt
                    const float v = pt == 0 ? acc[4 * d4] : (pt == 1 ? acc[4 * d4 + 1] : (pt == 2 ? acc[4 * d4 + 2] : acc[4 * d4 + 3]));
                    Hk[4 * d4 + pt] = tanh_fast(self[4 * d4 + pt] + v);
                }
            }
            EPI_SYNC();
            CTS(7);
            if (tid < 2 * AT) {
                const int n = tid & 63;
                const float *Hk = (tid < AT ? H1 : H2) + n * HS, *wa = tid < AT ? a.wa_1 : a.wa_2;
                float sc = 0.f;
#pragma unroll
                for (int d = 0; d < HP; ++d) sc += d < hd ? __ldg(wa + d) * Hk[d] : 0.f;
                (tid < AT ? attn1 : attn2)[n] = sc;
            }
            }
            EPI_SYNC();
            if (warp < 2) {
                float *x = warp ? attn2 : attn1;
                const int n = warp ? N2 : N1;
                const float x0 = lane < n ? x[lane] : -INFINITY, x1 = lane + 32 < n ? x[lane + 32] : -INFINITY;
                const float m = warp_max(fmaxf(x0, x1));
                const float e0 = lane < n ? __expf(x0 - m) : 0.f, e1 = lane + 32 < n ? __expf(x1 - m) : 0.f;
                const float s = warp_sum(e0 + e1);
                x[lane] = e0 / s;
                x[lane + 32] = e1 / s;
            }
            EPI_SYNC();
            CTS(8);
            // ---- pooled atoms p_k[h] = sum_n attn_k[n] a_k[n][h]
            if (tid < 2 * H) {
                const int which = tid >= H, h = which ? tid - H : tid;
                const float *at = which ? attn2 : attn1;
                const int n = which ? N2 : N1;
                float s = 0.f;
                for (int r = 0; r < n; ++r) s += at[r] * bf16_at(XP, 64 * which + r, h);
                (which ? p2 : p1)[h] = s;
            }
            EPI_SYNC();
            CTS(9);
            if (!BWD) {
                // compact_k[o] = W_j[o] . p_k + b_j[o]: four lanes per output, interleaved 16-byte weight loads all in flight
                for (int r = tid >> 2; r < 2 * O; r += NE / 4) {
                    const int which = r >= O, o = which ? r - O : r, pt = tid & 3;
                    const float *p = which ? p2 : p1;
                    const float4 *w = reinterpret_cast<const float4 *>(a.W_j + (long)o * H);
                    float4 ww[H / 16];
#pragma unroll
                    for (int u = 0; u < H / 16; ++u) ww[u] = __ldg(w + 4 * u + pt);
                    float s0 = 0.f, s1 = 0.f;
#pragma unroll
                    for (int u = 0; u < H / 16; ++u) {
                        const float4 pp = *reinterpret_cast<const float4 *>(p + 4 * (4 * u + pt));
                        s0 = fmaf(ww[u].x, pp.x, fmaf(ww[u].y, pp.y, s0));
                        s1 = fmaf(ww[u].z, pp.z, fmaf(ww[u].w, pp.w, s1));
                    }
                    float sum = s0 + s1;
                    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                    if (pt == 0) (which ? a.c2 : a.c1)[(long)pair * O + o] = sum + a.b_j[o];
                }
                CTS(10);
                continue;
            }
            // ======================================================== backward
            float *t1 = st4, *t2 = st4 + AT, *cs = st4 + 2 * AT, *rsum = st4 + 3 * AT;
            // pooled atoms for d W_j ; dp_k[h] = sum_o W_j[o][h] dc_k[o]: thread pair (two halves of the o range), eight
            // coalesced weight rows in flight each, combined through shared memory
            {
                const int oh = tid >> 8, e = tid & 255;
                const int which = e >= H, h = which ? e - H : e;
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
                if (e < 2 * H) {
                    if (oh == 0) (which ? a.P2 : a.P1)[(long)pair * H + h] = (which ? p2 : p1)[h];
                    const float *dc = (which ? a.dc2 : a.dc1) + (long)pair * O;
                    const int ob = ((O + 1) / 2 + 7) & ~7, o_end = oh ? O : (ob < O ? ob : O);
                    int o = oh ? (ob < O ? ob : O) : 0;
                    for (; o + 8 <= o_end; o += 8) {
                        float w[8];
#pragma unroll
                        for (int x = 0; x < 8; ++x) w[x] = __ldg(a.W_j + (long)(o + x) * H + h);
                        const float4 d0 = __ldg(reinterpret_cast<const float4 *>(dc + o)), d1 = __ldg(reinterpret_cast<const float4 *>(dc + o) + 1);
                        s0 = fmaf(w[0], d0.x, s0); s1 = fmaf(w[1], d0.y, s1); s2 = fmaf(w[2], d0.z, s2); s3 = fmaf(w[3], d0.w, s3);
                        s0 = fmaf(w[4], d1.x, s0); s1 = fmaf(w[5], d1.y, s1); s2 = fmaf(w[6], d1.z, s2); s3 = fmaf(w[7], d1.w, s3);
                    }
                    for (; o < o_end; ++o) s0 = fmaf(__ldg(a.W_j + (long)o * H + h), __ldg(dc + o), s0);
                }
                if (oh == 1 && e < 2 * H) part[e] = (s0 + s1) + (s2 + s3);
                EPI_SYNC();
                if (oh == 0 && e < 2 * H) (which ? dp2 : dp1)[h] = (s0 + s1) + (s2 + s3) + part[e];
            }
            EPI_SYNC();
            CTS(10);
            // d attn_k[n] = dp_k . a_k[n]: four threads per atom, 16-byte operand chunks
            {
                const int which = tid >> 8, n = (tid >> 2) & 63, hp = tid & 3;
                const float *dp = which ? dp2 : dp1;
                float s = 0.f;
                for (int c8 = hp; c8 < H / 8; c8 += 4) {
                    const uint4 u = *reinterpret_cast<const uint4 *>(XP + (c8 >> 3) * PANEL_BYTES + sw128(64 * which + n, (c8 & 7) * 8));
                    const __nv_bfloat162 *b2 = reinterpret_cast<const __nv_bfloat162 *>(&u);
#pragma unroll
                    for (int x = 0; x < 4; ++x) {
                        const float2 f = __bfloat1622float2(b2[x]);
                        s += f.x * dp[c8 * 8 + 2 * x] + f.y * dp[c8 * 8 + 2 * x + 1];
                    }
                }
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                if (hp == 0) (which ? t2 : t1)[n] = s;
            }
            EPI_SYNC();
            if (warp < 2) {     // softmax backward -> gradient of the pre-softmax scores
                const float *at = warp ? attn2 : attn1;
                float *da = warp ? t2 : t1;
                const int n = warp ? N2 : N1;
                const float x0 = lane < n ? at[lane] * da[lane] : 0.f, x1 = lane + 32 < n ? at[lane + 32] * da[lane + 32] : 0.f;
                const float dot = warp_sum(x0 + x1);
                da[lane] = lane < n ? at[lane] * (da[lane] - dot) : 0.f;
                da[lane + 32] = lane + 32 < n ? at[lane + 32] * (da[lane + 32] - dot) : 0.f;
            }
            EPI_SYNC();
            CTS(11);
            if (pool) {
                // scores are means of C: dC[i][j] = ds_1[j] / N2 + ds_2[i] / N1 ; no head path (d lt = 0)
                for (int idx = tid; idx < 2 * AT * HP; idx += NE) (idx < AT * HP ? H1 : H2 - AT * HP)[idx] = 0.f;
                for (int idx = tid; idx < AT * AT; idx += NE) {
                    const int j = idx >> 6, i = idx & 63;
                    const float c = Cs[j * CLD + i];
                    const float g = (j < N1 && i < N2) ? t1[j] / (float)N2 + t2[i] / (float)N1 : 0.f;
                    Cs[j * CLD + i] = g * act_bwd(a.act, c, c);
                }
                EPI_SYNC();
            } else {
            // dpre_k[n][:] = ds_k[n] wa_k[:] (1 - H_k^2) ; d wa_k[d] += sum_n ds_k[n] H_k[n][d]
            for (int idx = tid; idx < 2 * AT * HQ; idx += NE) {
                const int which = idx / (AT * HQ), r = idx % (AT * HQ), n = r / HQ, d4 = r % HQ;
                const float4 hv = *reinterpret_cast<const float4 *>((which ? H2 : H1) + n * HS + 4 * d4);
                const float *wa = which ? a.wa_2 : a.wa_1;
                const float ds = (which ? t2 : t1)[n];
                float4 o;
                o.x = 4 * d4 + 0 < hd ? ds * __ldg(wa + 4 * d4 + 0) * (1.f - hv.x * hv.x) : 0.f;
                o.y = 4 * d4 + 1 < hd ? ds * __ldg(wa + 4 * d4 + 1) * (1.f - hv.y * hv.y) : 0.f;
                o.z = 4 * d4 + 2 < hd ? ds * __ldg(wa + 4 * d4 + 2) * (1.f - hv.z * hv.z) : 0.f;
                o.w = 4 * d4 + 3 < hd ? ds * __ldg(wa + 4 * d4 + 3) * (1.f - hv.w * hv.w) : 0.f;
                *reinterpret_cast<float4 *>((which ? dpre2 : dpre1) + n * HS + 4 * d4) = o;
            }
            for (int r = warp; r < 2 * hd; r += EPW) {
                const int which = r >= hd, d = which ? r - hd : r;
                const float *Hk = (which ? H2 : H1) + d, *ds = which ? t2 : t1;
                const float sw = warp_sum(ds[lane] * Hk[lane * HS] + ds[lane + 32] * Hk[(lane + 32) * HS]);
                if (lane == 0) (which ? gwa2 : gwa1)[d] += sw;
            }
            EPI_SYNC();
            CTS(12);
            // u1[i] = sum_j L_1[j][i] dL_1[j][i], dL_1[j][i] = dpre1[j] . lt2[i] ; u2[j] = sum_i L_2[i][j] (dpre2[i] . lt1[j])
            // four threads per output (a quarter of the inner index each), the output's own head row in registers
            {
                const int out = tid >> 2, pt = tid & 3, which = out >= AT, n = out & 63;
                const float *Lw = which ? L2p : L1t;            // L_1[j][i] at L1t[i*PLD + j] ; L_2[i][j] at L2p[j*PLD + i]
                const float *other = which ? dpre2 : dpre1;
                float own[HP];
#pragma unroll
                for (int d4 = 0; d4 < HQ; ++d4) {
                    const float4 r4 = *reinterpret_cast<const float4 *>((which ? lt1 : lt2) + n * HS + 4 * d4);
                    own[4 * d4] = r4.x; own[4 * d4 + 1] = r4.y; own[4 * d4 + 2] = r4.z; own[4 * d4 + 3] = r4.w;
                }
                float u = 0.f;
#pragma unroll 4
                for (int mm = 0; mm < 16; ++mm) {
                    const int m = 4 * mm + pt;
                    float dl = 0.f;
#pragma unroll
                    for (int d4 = 0; d4 < HQ; ++d4) {
                        const float4 r4 = *reinterpret_cast<const float4 *>(other + m * HS + 4 * d4);
                        dl = fmaf(r4.x, own[4 * d4], fmaf(r4.y, own[4 * d4 + 1], fmaf(r4.z, own[4 * d4 + 2], fmaf(r4.w, own[4 * d4 + 3], dl))));
                    }
                    u = fmaf(Lw[n * PLD + m], dl, u);
                }
                u += __shfl_xor_sync(0xffffffffu, u, 1);
                u += __shfl_xor_sync(0xffffffffu, u, 2);
                if (pt == 0) part[out] = u;          // u1 at [0,64), u2 at [64,128)
            }
            // total d lt_k (direct + through the other molecule's H) -> over H_k:
            //   d lt_1[j][:] = dpre1[j][:] + sum_i L_2[i][j] dpre2[i][:] ; d lt_2[i][:] = dpre2[i][:] + sum_j L_1[j][i] dpre1[j][:]
            {
                const int which = tid >> 8, n = (tid >> 2) & 63, pt = tid & 3;
                const float *Lw = which ? L1t : L2p, *other = which ? dpre1 : dpre2;
                float acc[HP];
#pragma unroll
                for (int d = 0; d < HP; ++d) acc[d] = 0.f;
#pragma unroll 4
                for (int mm = 0; mm < 16; ++mm) {
                    const int m = 4 * mm + pt;
                    const float l = Lw[n * PLD + m];
#pragma unroll
                    for (int d4 = 0; d4 < HQ; ++d4) {
                        const float4 r4 = *reinterpret_cast<const float4 *>(other + m * HS + 4 * d4);
                        acc[4 * d4] = fmaf(l, r4.x, acc[4 * d4]); acc[4 * d4 + 1] = fmaf(l, r4.y, acc[4 * d4 + 1]);
                        acc[4 * d4 + 2] = fmaf(l, r4.z, acc[4 * d4 + 2]); acc[4 * d4 + 3] = fmaf(l, r4.w, acc[4 * d4 + 3]);
                    }
                }
#pragma unroll
                for (int d = 0; d < HP; ++d) {
                    acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], 1);
                    acc[d] += __shfl_xor_sync(0xffffffffu, acc[d], 2);
                }
                const float *self = (which ? dpre2 : dpre1) + n * HS;
                float *dst = (which ? H2 : H1) + n * HS;       // H_k is dead: it becomes d lt_k
#pragma unroll
                for (int d4 = 0; d4 < HQ; ++d4) {
                    const float v = pt == 0 ? acc[4 * d4] : (pt == 1 ? acc[4 * d4 + 1] : (pt == 2 ? acc[4 * d4 + 2] : acc[4 * d4 + 3]));
                    dst[4 * d4 + pt] = self[4 * d4 + pt] + v;
                }
            }
            EPI_SYNC();
            CTS(13);
            // dC^T[j][i] (pre-activation) in place of C^T: a thread keeps ITS column i (lt2[i], dpre2[i] in registers) and
            // walks eight rows j whose head rows are warp-wide broadcasts
            {
                const int i = tid & 63;
                float l2[HP], p2[HP];
#pragma unroll
                for (int d4 = 0; d4 < HQ; ++d4) {
                    const float4 x4 = *reinterpret_cast<const float4 *>(lt2 + i * HS + 4 * d4), y4 = *reinterpret_cast<const float4 *>(dpre2 + i * HS + 4 * d4);
                    l2[4 * d4] = x4.x; l2[4 * d4 + 1] = x4.y; l2[4 * d4 + 2] = x4.z; l2[4 * d4 + 3] = x4.w;
                    p2[4 * d4] = y4.x; p2[4 * d4 + 1] = y4.y; p2[4 * d4 + 2] = y4.z; p2[4 * d4 + 3] = y4.w;
                }
                const float u1i = part[i];
#pragma unroll 2
                for (int u8 = 0; u8 < AT * AT / NE; ++u8) {
                    const int j = (tid >> 6) + u8 * (NE / 64);
                    float dl1 = 0.f, dl2 = 0.f;
#pragma unroll
                    for (int d4 = 0; d4 < HQ; ++d4) {
                        const float4 x4 = *reinterpret_cast<const float4 *>(dpre1 + j * HS + 4 * d4), y4 = *reinterpret_cast<const float4 *>(lt1 + j * HS + 4 * d4);
                        dl1 = fmaf(x4.x, l2[4 * d4], fmaf(x4.y, l2[4 * d4 + 1], fmaf(x4.z, l2[4 * d4 + 2], fmaf(x4.w, l2[4 * d4 + 3], dl1))));
                        dl2 = fmaf(y4.x, p2[4 * d4], fmaf(y4.y, p2[4 * d4 + 1], fmaf(y4.z, p2[4 * d4 + 2], fmaf(y4.w, p2[4 * d4 + 3], dl2))));
                    }
                    const float c = Cs[j * CLD + i];
                    const float g = L1t[i * PLD + j] * (dl1 - u1i) + L2p[j * PLD + i] * (dl2 - part[AT + j]);
                    Cs[j * CLD + i] = g * act_bwd(a.act, c, c);
                }
            }
            EPI_SYNC();
            CTS(14);
            }
            // rsum[i] = sum_j dC[i][j] ; cs[j] = sum_i dC[i][j]
            if (tid < AT) {
                float s = 0.f;
                for (int j = 0; j < AT; ++j) s += Cs[j * CLD + tid];
                rsum[tid] = s;
            }
            for (int j = warp; j < AT; j += EPW) {
                const float s = warp_sum(Cs[j * CLD + lane] + Cs[j * CLD + lane + 32]);
                if (lane == 0) cs[j] = s;
            }
            EPI_SYNC();
            CTS(15);
            if (warp == EPW - 1) {
                const float s = warp_sum(rsum[lane] + rsum[lane + 32]);
                if (lane == 0) gb[0] += s;
            }
            // operand panel [dC^T ; dC] (+ extension columns [dlt_2 | rsum] of the a2 rows)
            for (int idx = tid; idx < 2 * AT * 8; idx += NE) {
                float v[8];
                if (idx < AT * 8) {
                    const int j = idx >> 3, c8 = idx & 7;
                    const float4 x0 = *reinterpret_cast<const float4 *>(Cs + j * CLD + c8 * 8), x1 = *reinterpret_cast<const float4 *>(Cs + j * CLD + c8 * 8 + 4);
                    v[0] = x0.x; v[1] = x0.y; v[2] = x0.z; v[3] = x0.w; v[4] = x1.x; v[5] = x1.y; v[6] = x1.z; v[7] = x1.w;
                    *reinterpret_cast<uint4 *>(DP + sw128(j, c8 * 8)) = pack8(v);
                } else {
                    const int i = idx & 63, c8 = (idx - AT * 8) >> 6;
#pragma unroll
                    for (int x = 0; x < 8; ++x) v[x] = Cs[(c8 * 8 + x) * CLD + i];
                    *reinterpret_cast<uint4 *>(DP + sw128(64 + i, c8 * 8)) = pack8(v);
                }
            }
            if (tid < 2 * AT) {       // extension chunks: a2 rows of the dC panel (tid < 64), a1 rows of the R panel (tid >= 64)
                const int which = tid < AT, n = tid & 63;
                const float *dl = (which ? H2 : H1) + n * HS;
                float v[16];
#pragma unroll
                for (int d = 0; d < 16; ++d) v[d] = d < HP ? dl[d] : 0.f;      // heads >= head are zero by construction
                v[15] = which ? rsum[n] : cs[n];
                uint8_t *dst = which ? DP + PANEL_BYTES : QP;
                const int r = which ? 64 + n : n;
                *reinterpret_cast<uint4 *>(dst + sw128(r, 0)) = pack8(v);
                *reinterpret_cast<uint4 *>(dst + sw128(r, 8)) = pack8(v + 8);
            }
            warp_arrive(BAR(B_DRDY), lane);
            CTS(16);
            // ---- both contractions of the dC panel are done: S is dead, the R panels take its place
            mbar_wait(BAR(B_R), par);
            mbar_wait(BAR(B_A2), par);
            tc_fence_after();
            CTS(17);
            float *stg = reinterpret_cast<float *>(DP + warp * 2048);      // the dC panels are dead too: store staging
            if (cg * 32 < H) {
                uint32_t v[32];
                if (q < 2) {
                    // R = dC^T a2 -> bf16 panels: A operand of d a1 = R W^T, B operand of d W += a1^T R
                    tc_ld32(t_lane + C::COL_R + cg * 32, v);
                    tc_wait_ld();
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const int kk = cg * 32 + 8 * g;
                        float f[8];
#pragma unroll
                        for (int x = 0; x < 8; ++x) f[x] = __uint_as_float(v[8 * g + x]);
                        *reinterpret_cast<uint4 *>(SP + (kk >> 6) * PANEL_BYTES + sw128(row, kk & 63)) = pack8(f);
                    }
                } else {
                    // d a2 = dC S + dlt_2 lt_2 + rsum V2^T (all in the accumulator) + attn_2[i] dp2[k]
                    tc_ld32(t_lane + C::COL_A2 + cg * 32, v);
                    tc_wait_ld();
                    const float at = attn2[row - 64];
                    float f[32];
#pragma unroll
                    for (int x = 0; x < 32; x += 4) {
                        const float4 d4 = *reinterpret_cast<const float4 *>(dp2 + cg * 32 + x);
                        f[x] = fmaf(at, d4.x, __uint_as_float(v[x])); f[x + 1] = fmaf(at, d4.y, __uint_as_float(v[x + 1]));
                        f[x + 2] = fmaf(at, d4.z, __uint_as_float(v[x + 2])); f[x + 3] = fmaf(at, d4.w, __uint_as_float(v[x + 3]));
                    }
#pragma unroll
                    for (int h2 = 0; h2 < 2; ++h2)
                        warp_store_rows<16>(stg, f + 16 * h2, lane, [&](int r) -> float * {
                            const int i = 32 * (q - 2) + r;
                            return i < N2 ? a.d_a2 + (r2 + i) * H + cg * 32 + 16 * h2 : nullptr;
                        });
                }
            }
            warp_arrive(BAR(B_RRDY), lane);
            CTS(18);
            // ---- d a1 = R W^T + dlt_1 lt_1 + cs V1^T + attn_1[j] dp1[h]
            mbar_wait(BAR(B_A1), par);
            tc_fence_after();
            CTS(19);
            if (q < 2 && cg * 32 < H) {
                uint32_t v[32];
                tc_ld32(t_lane + C::COL_A1 + cg * 32, v);
                tc_wait_ld();
                const float at = attn1[row];
                float f[32];
#pragma unroll
                for (int x = 0; x < 32; x += 4) {
                    const float4 d4 = *reinterpret_cast<const float4 *>(dp1 + cg * 32 + x);
                    f[x] = fmaf(at, d4.x, __uint_as_float(v[x])); f[x + 1] = fmaf(at, d4.y, __uint_as_float(v[x + 1]));
                    f[x + 2] = fmaf(at, d4.z, __uint_as_float(v[x + 2])); f[x + 3] = fmaf(at, d4.w, __uint_as_float(v[x + 3]));
                }
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2)
                    warp_store_rows<16>(stg, f + 16 * h2, lane, [&](int r) -> float * {
                        const int j = 32 * q + r;
                        return j < N1 ? a.d_a1 + (r1 + j) * H + cg * 32 + 16 * h2 : nullptr;
                    });
            }
            CTS(20);
            CTS(21);
            tc_fence_before();
        }
        if (BWD && it > 0) {
            // every MMA of the last pair has completed (B_A1): flush the persistent parameter-gradient accumulators
            tc_fence_after();
            if (row < H && cg * 32 < H && a.d_W) {            // TMEM lane = row h of d W
                uint32_t v[32];
                tc_ld32(t_lane + C::COL_DW + cg * 32, v);
                tc_wait_ld();
                float *dst = a.d_W + (long)row * H + cg * 32, *sp = a.det.slot(a.det.w() + (long)row * H + cg * 32);
#pragma unroll
                for (int x = 0; x < 32; x += 4)
                    det_put4(dst + x, sp ? sp + x : nullptr,
                             make_float4(__uint_as_float(v[x]), __uint_as_float(v[x + 1]), __uint_as_float(v[x + 2]), __uint_as_float(v[x + 3])));
            }
            if (row < H && cg >= 2) {                         // [d lt_k | d V_k]^T: lane = feature, column = head (15: V)
                const int k2 = cg - 2;
                uint32_t w[16];
                tc_ld16(t_lane + (k2 ? C::COL_X2 : C::COL_X1), w);
                tc_wait_ld();
                float *dlt = k2 ? a.d_lt_2 : a.d_lt_1, *dV = k2 ? a.d_V2 : a.d_V1;
#pragma unroll
                for (int d = 0; d < MAXHD; ++d)
                    if (d < hd && dlt) det_put(dlt + (long)d * H + row, a.det.slot(a.det.lt(k2) + (long)d * H + row), __uint_as_float(w[d]));
                if (dV) det_put(dV + row, a.det.slot(a.det.v(k2) + row), __uint_as_float(w[15]));
            }
            tc_fence_before();
            EPI_SYNC();
            if (tid < hd) {
                if (a.d_wa_1) det_put(a.d_wa_1 + tid, a.det.slot(a.det.wa(0) + tid), gwa1[tid]);
                if (a.d_wa_2) det_put(a.d_wa_2 + tid, a.det.slot(a.det.wa(1) + tid), gwa2[tid]);
            }
            if (tid == 0 && a.d_b) det_put(a.d_b, a.det.slot(a.det.b()), gb[0]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPW + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(C::TMEM_COLS));
    }
}

// ---- weight images: bf16, SW128 K-major tiles
//   img1 [KP k-tiles][H + 32 rows n][64 k]: n < H: W[n][k] ; H+e (e < 16): lt_1[e] (e < head), V1 (e = 15) ;
//                                          H+16+e: lt_2[e], V2 (e = 15)
//   img2 [KP k-tiles][H rows n][64 k]     : W[k][n]                        (S = a1 W)
//   img1x [H rows n][64 k]                : k < head: lt_1[k][n] ; k = 15: V1[n]   (extension k-step of d a1)
struct PackArgs {
    int H, head;
    const float *W, *V1, *V2, *lt_1, *lt_2;
    uint8_t *img1, *img2, *img1x;
};
__global__ void pack_coattn_kernel(const PackArgs p) {
    const int H = p.H, KP = H / 64, hd = p.head;
    const long n1 = (long)KP * (H + 32) * 64, n2 = (long)KP * H * 64, n3 = (long)H * 64;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < n1 + n2 + n3; idx += (long)gridDim.x * blockDim.x) {
        float w = 0.f;
        uint8_t *dst;
        int n, kk;
        if (idx < n1) {
            kk = idx & 63; n = (idx >> 6) % (H + 32);
            const int kt = (int)(idx / (64L * (H + 32))), K = kt * 64 + kk;
            if (n < H) w = p.W[(long)n * H + K];
            else {
                const int e = n - H, which = e >> 4, d = e & 15;
                if (d < hd) w = (which ? p.lt_2 : p.lt_1)[(long)d * H + K];
                else if (d == 15) w = (which ? p.V2 : p.V1)[K];
            }
            dst = p.img1 + (size_t)kt * (H + 32) * 128;
        } else if (idx < n1 + n2) {
            const long r = idx - n1;
            kk = r & 63; n = (r >> 6) % H;
            const int kt = (int)(r / (64L * H));
            w = p.W[(long)(kt * 64 + kk) * H + n];
            dst = p.img2 + (size_t)kt * H * 128;
        } else {
            const long r = idx - n1 - n2;
            kk = r & 63; n = (int)(r >> 6);
            if (kk < hd) w = p.lt_1[(long)kk * H + n];
            else if (kk == 15) w = p.V1[n];
            dst = p.img1x;
        }
        const uint32_t off = (uint32_t)n * 128u + ((((uint32_t)(kk >> 3) ^ ((uint32_t)n & 7u)) << 4) | (((uint32_t)kk & 7u) << 1));
        *reinterpret_cast<__nv_bfloat16 *>(dst + off) = __float2bfloat16_rn(w);
    }
}

static size_t img_bytes(int H) { return (size_t)(H / 64) * (H + 32) * 128 + (size_t)(H / 64) * H * 128 + (size_t)H * 128; }

}  // namespace ctc
}  // namespace bmp

using namespace bmp;

static long long *g_ctc_dbg = nullptr;
extern "C" void bmp_debug_set_buffer_ctc(void *p) { g_ctc_dbg = (long long *)p; }

extern "C" size_t bmp_coattn_tc_workspace_bytes(int hidden) {
    if (hidden != 64 && hidden != 128) return 0;
    return ctc::img_bytes(hidden) + 1024;
}

// whether the tcgen05 kernel covers this problem (otherwise the fp32 kernel of coattn.cu runs)
bool bmp_coattn_tc_supported(int H, int head, int variant, bool bwd) {
    if (H != 64 && H != 128) return false;
    if (variant == BMP_COATTN_FINE ? (head < 1 || head > ctc::MAXHD) : variant != BMP_COATTN_POOL) return false;
    if (variant == BMP_COATTN_POOL) head = 0;
    const size_t need = H == 64 ? (bwd ? ctc::smem_bytes<64, true>(head) : ctc::smem_bytes<64, false>(head))
                                : (bwd ? ctc::smem_bytes<128, true>(head) : ctc::smem_bytes<128, false>(head));
    return need <= 227 * 1024;
}

template <int H, bool BWD, int HP>
static int launch_ctc_hp(const ctc::Args &k, int head, cudaStream_t st) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = k.mb < sms ? k.mb : sms;
    const size_t smem = ctc::smem_bytes<H, BWD>(head);
    Partials pt(st);
    ctc::Args kk = k;
    if (BWD && co_det_begin(pt, kk.det, H, grid)) return BMP_EINVAL;
    cudaFuncSetAttribute(ctc::coattn_tc_kernel<H, BWD, HP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    {
        ProfScope prof(BWD ? BMP_PROF_COATTN_BWD : BMP_PROF_COATTN_FWD, st);
        ctc::coattn_tc_kernel<H, BWD, HP><<<grid, ctc::NT, smem, st>>>(kk);
    }
    count_launch();
    int rc = check_launch("coattn_tc_kernel");
    if (rc || !BWD) return rc;
    return co_det_end(pt, kk.det, grid, head, k.d_W, k.d_lt_1, k.d_lt_2, k.d_V1, k.d_V2, k.d_wa_1, k.d_wa_2, k.d_b, true,
                      "det_reduce_kernel (coattn_tc)");
}

template <int H, bool BWD>
static int launch_ctc(const ctc::Args &k, int head, cudaStream_t st) {
    return head <= 8 ? launch_ctc_hp<H, BWD, 8>(k, head, st) : launch_ctc_hp<H, BWD, 16>(k, head, st);
}

// Shared by forward and backward: pack the weight images into the workspace, fill the common arguments.
static int ctc_prepare(ctc::Args &k, int mb, int n1, int n2, int H, int O, int head, int act, const float *a1, const float *a2,
                       const float *W, const float *V1, const float *V2, const float *b, const float *lt1, const float *lt2,
                       const float *wa1, const float *wa2, const float *Wj, const float *bj, void *ws, size_t ws_bytes, bool images_ready,
                       cudaStream_t st) {
    if (!ws || ws_bytes < bmp_coattn_tc_workspace_bytes(H)) {
        set_error("BMP_MODE_BF16 co-attention: tc_workspace of >= %zu bytes required", bmp_coattn_tc_workspace_bytes(H));
        return BMP_EINVAL;
    }
    uint8_t *base = (uint8_t *)(((uintptr_t)ws + 255) & ~(uintptr_t)255);
    ctc::PackArgs p;
    p.H = H; p.head = head; p.W = W; p.V1 = V1; p.V2 = V2; p.lt_1 = lt1; p.lt_2 = lt2;
    p.img1 = base;
    p.img2 = p.img1 + (size_t)(H / 64) * (H + 32) * 128;
    p.img1x = p.img2 + (size_t)(H / 64) * H * 128;
    if (!images_ready) {
        ctc::pack_coattn_kernel<<<32, 256, 0, st>>>(p);
        count_launch();
        int rc = check_launch("pack_coattn_kernel");
        if (rc) return rc;
    }
    k = ctc::Args{};
    k.mb = mb; k.n1 = n1; k.n2 = n2; k.O = O; k.head = head; k.act = act;
    k.atoms_1 = a1; k.atoms_2 = a2; k.b = b; k.wa_1 = wa1; k.wa_2 = wa2; k.W_j = Wj; k.b_j = bj; k.lt_2 = lt2; k.V2 = V2;
    k.img1 = p.img1; k.img2 = p.img2; k.img1x = p.img1x;
    k.dbg = g_ctc_dbg;
    return BMP_OK;
}

int bmp_coattn_forward_tc(const bmp_coattn_fwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    ctc::Args k;
    const int head = a->variant == BMP_COATTN_POOL ? 0 : a->head;
    int rc = ctc_prepare(k, a->mb, a->n1, a->n2, a->hidden, a->out_dim, head, a->act, a->atoms_1, a->atoms_2, a->W, a->V1, a->V2, a->b,
                         a->lt_1, a->lt_2, a->wa_1, a->wa_2, a->W_j, a->b_j, a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, st);
    if (rc) return rc;
    k.c1 = a->compact_1; k.c2 = a->compact_2;
    k.pool = a->variant == BMP_COATTN_POOL;
    return a->hidden == 64 ? launch_ctc<64, false>(k, head, st) : launch_ctc<128, false>(k, head, st);
}

// data part of the backward; the parameter-gradient contractions stay with bmp_coattn_backward
int bmp_coattn_backward_tc(const bmp_coattn_bwd_t *a, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    ctc::Args k;
    const int head = a->variant == BMP_COATTN_POOL ? 0 : a->head;
    int rc = ctc_prepare(k, a->mb, a->n1, a->n2, a->hidden, a->out_dim, head, a->act, a->atoms_1, a->atoms_2, a->W, a->V1, a->V2, a->b,
                         a->lt_1, a->lt_2, a->wa_1, a->wa_2, a->W_j, a->b_j, a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, st);
    if (rc) return rc;
    k.dc1 = a->d_compact_1; k.dc2 = a->d_compact_2; k.R = a->R; k.P1 = a->P1; k.P2 = a->P2; k.DL1 = a->DL1; k.DL2 = a->DL2;
    k.d_a1 = a->d_atoms_1; k.d_a2 = a->d_atoms_2;
    k.d_W = a->d_W; k.d_lt_1 = a->d_lt_1; k.d_lt_2 = a->d_lt_2;
    k.d_V1 = a->d_V1; k.d_V2 = a->d_V2; k.d_b = a->d_b; k.d_wa_1 = a->d_wa_1; k.d_wa_2 = a->d_wa_2;
    k.pool = a->variant == BMP_COATTN_POOL;
    return a->hidden == 64 ? launch_ctc<64, true>(k, head, st) : launch_ctc<128, true>(k, head, st);
}
