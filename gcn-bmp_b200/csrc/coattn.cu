// coattn.cu -- fused fine-grained cross-graph co-attention, fp32.
// Replaces models/coattention/nie_coattention.py:335-396 (= vqa_parallel_coattention.py:42-103)
// and PoolingFineCoattention.py:31-83.  One CTA per drug pair:
//   C[i][j] = act(a1_j^T W a2_i + V1.a1_j + V2.a2_i + b)        i: atoms_2, j: atoms_1
// is built as Q = W a2^T (streamed W) then C^T = a1 Q, entirely in shared memory --
// the reference's two F.tile copies of (mb*N2*N1, H) never exist.  Row/column
// softmaxes, the head projections and the attended pooling follow in the same CTA.
// compact_k = j_layer(sum_n attn_k[n] atoms_k[n]) because sum_n attn_k[n] = 1.
#include "det.cuh"

namespace bmp {

constexpr int PLD = 65;     // padded ld for scalar-accessed 64x64 maps
constexpr int DLD = 68;     // ld of the i-major dC copy used as a GEMM Y operand
constexpr int MAXHEAD = 16;

struct CoSmem {
    float *a1s, *a2s, *Qs;          // [H][64] each
    float *Cs;                      // [64 j][64 i]  C^T (post-activation), later dC^T (pre-activation grad)
    float *L1t;                     // [64 i][PLD]   L_1[j][i] at [i*PLD + j];   later Ds [64 i][DLD]
    float *L2p;                     // [64 j][PLD]   L_2[i][j] at [j*PLD + i]
    float *lt1, *lt2;               // [head][64]
    float *H1, *H2;                 // [head][64]
    float *attn1, *attn2;           // [64]
    float *v1, *v2;                 // [64]  V1.a1_j, V2.a2_i
    float *p1, *p2;                 // [H]   pooled atoms
    float *tmp;                     // [4*64 + 2*H] scratch
    float *stage;
};

__host__ __device__ inline size_t co_smem_floats(int H, int head) {
    return (size_t)3 * H * AT + AT * AT + AT * DLD + AT * PLD + 4 * head * AT + 4 * AT + 2 * H + (4 * AT + 2 * H) +
           2 * head * AT /*dpre1,dpre2*/ + STAGE_FLOATS + 64;
}

__device__ __forceinline__ CoSmem co_carve(float *base, int H, int head) {
    CoSmem s;
    float *p = base;
    s.a1s = p; p += H * AT;
    s.a2s = p; p += H * AT;
    s.Qs = p; p += H * AT;
    s.Cs = p; p += AT * AT;
    s.L1t = p; p += AT * DLD;
    s.L2p = p; p += AT * PLD;
    p = (float *)(((uintptr_t)p + 15) & ~(uintptr_t)15);
    s.lt1 = p; p += head * AT;
    s.lt2 = p; p += head * AT;
    s.H1 = p; p += head * AT;
    s.H2 = p; p += head * AT;
    s.attn1 = p; p += AT;
    s.attn2 = p; p += AT;
    s.v1 = p; p += AT;
    s.v2 = p; p += AT;
    s.p1 = p; p += H;
    s.p2 = p; p += H;
    s.tmp = p; p += 4 * AT + 2 * H + 2 * head * AT;
    p = (float *)(((uintptr_t)p + 15) & ~(uintptr_t)15);
    s.stage = p;
    return s;
}

__device__ __forceinline__ float warp_sum(float v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

struct CoArgs {
    long long *dbg;
    int mb, n1, n2, H, O, head, variant, act;
    const float *atoms_1, *atoms_2, *W, *V1, *V2, *b, *lt_1, *lt_2, *wa_1, *wa_2, *W_j, *b_j;
};

// softmax over n entries of x (smem) by one warp; writes probabilities in place
__device__ __forceinline__ void warp_softmax(float *x, int n, int lane) {
    float a = lane < n ? x[lane] : -INFINITY, b = lane + 32 < n ? x[lane + 32] : -INFINITY;
    float m = warp_max(fmaxf(a, b));
    float ea = lane < n ? expf(a - m) : 0.f, eb = lane + 32 < n ? expf(b - m) : 0.f;
    float s = warp_sum(ea + eb);
    if (lane < n) x[lane] = ea / s;
    if (lane + 32 < n) x[lane + 32] = eb / s;
}

// Forward for one pair into shared memory.  On exit (after the trailing sync):
// Cs, L1t, L2p, lt*, H*, attn*, p* are valid.
#define CTS(i) do { if (A.dbg && blockIdx.x == 0 && threadIdx.x == 0 && pair == 0) A.dbg[i] = clock64(); } while (0)
__device__ void co_forward(const CoArgs &A, const CoSmem &S, int pair) {
    const int H = A.H, N1 = A.n1, N2 = A.n2, hd = A.head;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
    CTS(0);
    const float *a1 = A.atoms_1 + (long)pair * N1 * H, *a2 = A.atoms_2 + (long)pair * N2 * H;
    load_cm(S.a1s, a1, N1, H);
    load_cm(S.a2s, a2, N2, H);
    __syncthreads();
    CTS(1);
    // v1[j] = V1 . a1_j ; v2[i] = V2 . a2_i
    if (tid < 2 * AT) {
        const int n = tid & 63;
        const float *src = tid < AT ? S.a1s : S.a2s, *V = tid < AT ? A.V1 : A.V2;
        float s = 0.f;
        for (int h = 0; h < H; ++h) s += V[h] * src[h * AT + n];
        (tid < AT ? S.v1 : S.v2)[n] = s;
    }
    // Q[h][i] = sum_k W[h][k] a2[i][k]
    for (int oc = 0; oc * 64 < H; ++oc) {
        float acc[4][4];
        zero_acc(acc);
        gemm64_g<false>(acc, A.W, H, oc * 64, H, H, S.a2s, S.stage);
        if (oc * 64 + ty * 4 < H) tile_store_s(S.Qs, oc * 64, acc);
    }
    __syncthreads();
    CTS(2);
    // C^T[j][i] = act(sum_h a1[j][h] Q[h][i] + v1[j] + v2[i] + b)
    {
        float acc[4][4];
        zero_acc(acc);
        gemm64_g<false>(acc, a1, H, 0, N1 & ~3, H, S.Qs, S.stage);
        // rows j in the ragged tail (N1 % 4 != 0) are handled below with a scalar pass
        const float bias = A.b[0];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int b = 0; b < 4; ++b)
                acc[q][b] = act_fwd(A.act, acc[q][b] + S.v1[ty * 4 + q] + S.v2[tx * 4 + b] + bias);
        tile_store_s(S.Cs, 0, acc);
    }
    __syncthreads();
    if (N1 & 3) {   // ragged rows of a1: j in [N1&~3, N1)
        const int jb = N1 & ~3, nj = N1 - jb;
        for (int idx = tid; idx < nj * AT; idx += NTHREADS) {
            int j = jb + idx / AT, i = idx % AT;
            float s = 0.f;
            for (int h = 0; h < H; ++h) s += S.a1s[h * AT + j] * S.Qs[h * AT + i];
            S.Cs[j * AT + i] = act_fwd(A.act, s + S.v1[j] + S.v2[i] + A.b[0]);
        }
        __syncthreads();
    }
    CTS(3);
    if (A.variant == BMP_COATTN_FINE) {
        // column stats (softmax over i for each j) -> L2p ; row stats (over j for each i) -> L1t
        float *m2 = S.tmp, *s2 = S.tmp + AT, *m1 = S.tmp + 2 * AT, *s1 = S.tmp + 3 * AT;
        if (tid < AT) {            // thread = i : over j  (Cs[j*64+i], lanes over i: conflict-free)
            const int i = tid;
            float m = -INFINITY, s = 0.f;
            if (i < N2) {
                for (int j = 0; j < N1; ++j) m = fmaxf(m, S.Cs[j * AT + i]);
                for (int j = 0; j < N1; ++j) s += expf(S.Cs[j * AT + i] - m);
            }
            m1[i] = m; s1[i] = s;
        }
        for (int j = warp; j < AT; j += NTHREADS / 32) {   // warp = j : over i
            float a = (j < N1 && lane < N2) ? S.Cs[j * AT + lane] : -INFINITY;
            float b = (j < N1 && lane + 32 < N2) ? S.Cs[j * AT + lane + 32] : -INFINITY;
            float m = warp_max(fmaxf(a, b));
            float s = warp_sum((a > -INFINITY ? expf(a - m) : 0.f) + (b > -INFINITY ? expf(b - m) : 0.f));
            if (lane == 0) { m2[j] = m; s2[j] = s; }
        }
        __syncthreads();
        for (int idx = tid; idx < AT * AT; idx += NTHREADS) {
            const int j = idx >> 6, i = idx & 63;
            const bool live = j < N1 && i < N2;
            const float c = S.Cs[idx];
            S.L2p[j * PLD + i] = live ? expf(c - m2[j]) / s2[j] : 0.f;
            S.L1t[i * PLD + j] = live ? expf(c - m1[i]) / s1[i] : 0.f;
        }
        CTS(4);
        // lt_k[d][n] = sum_h lt_k[d][h] a_k[n][h]
        for (int idx = tid; idx < 2 * hd * AT; idx += NTHREADS) {
            const int which = idx / (hd * AT), r = idx % (hd * AT), d = r / AT, n = r % AT;
            const float *src = which ? S.a2s : S.a1s, *w = (which ? A.lt_2 : A.lt_1) + (long)d * H;
            float s = 0.f;
            for (int h = 0; h < H; ++h) s += w[h] * src[h * AT + n];
            (which ? S.lt2 : S.lt1)[d * AT + n] = s;
        }
        __syncthreads();
        CTS(5);
        // H_1[j][d] = tanh(lt_1[j][d] + sum_i L_1[j][i] lt_2[i][d]) ; H_2[i][d] likewise
        for (int idx = tid; idx < 2 * hd * AT; idx += NTHREADS) {
            const int which = idx / (hd * AT), r = idx % (hd * AT), d = r / AT, n = r % AT;
            float s;
            if (!which) {
                s = S.lt1[d * AT + n];
                for (int i = 0; i < N2; ++i) s += S.L1t[i * PLD + n] * S.lt2[d * AT + i];
                S.H1[d * AT + n] = tanhf(s);
            } else {
                s = S.lt2[d * AT + n];
                for (int j = 0; j < N1; ++j) s += S.L2p[j * PLD + n] * S.lt1[d * AT + j];
                S.H2[d * AT + n] = tanhf(s);
            }
        }
        __syncthreads();
        if (tid < 2 * AT) {
            const int n = tid & 63;
            const float *Hs = tid < AT ? S.H1 : S.H2, *wa = tid < AT ? A.wa_1 : A.wa_2;
            float s = 0.f;
            for (int d = 0; d < hd; ++d) s += wa[d] * Hs[d * AT + n];
            (tid < AT ? S.attn1 : S.attn2)[n] = s;
        }
    } else {   // POOL: attn_1 = softmax_j(mean_i C), attn_2 = softmax_i(mean_j C)
        if (tid < AT) {
            const int i = tid;
            float s = 0.f;
            for (int j = 0; j < N1; ++j) s += S.Cs[j * AT + i];
            S.attn2[i] = s / (float)N1;
        }
        for (int j = warp; j < AT; j += NTHREADS / 32) {
            float a = (lane < N2 ? S.Cs[j * AT + lane] : 0.f) + (lane + 32 < N2 ? S.Cs[j * AT + lane + 32] : 0.f);
            a = warp_sum(a);
            if (lane == 0) S.attn1[j] = a / (float)N2;
        }
    }
    __syncthreads();
    CTS(6);
    if (warp == 0) warp_softmax(S.attn1, N1, lane);
    if (warp == 1) warp_softmax(S.attn2, N2, lane);
    __syncthreads();
    CTS(7);
    // pooled atoms p_k[h] = sum_n attn_k[n] a_k[n][h]   (warp per channel)
    for (int r = warp; r < 2 * H; r += NTHREADS / 32) {
        const int which = r >= H, h = which ? r - H : r;
        const float *src = (which ? S.a2s : S.a1s) + h * AT, *at = which ? S.attn2 : S.attn1;
        const int n = which ? N2 : N1;
        float s = (lane < n ? at[lane] * src[lane] : 0.f) + (lane + 32 < n ? at[lane + 32] * src[lane + 32] : 0.f);
        s = warp_sum(s);
        if (lane == 0) (which ? S.p2 : S.p1)[h] = s;
    }
    __syncthreads();
    CTS(8);
}

__global__ void __launch_bounds__(NTHREADS, 1) coattn_fwd_kernel(const CoArgs A, float *__restrict__ c1, float *__restrict__ c2) {
    extern __shared__ __align__(16) float smem[];
    CoSmem S = co_carve(smem, A.H, A.head);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int pair = blockIdx.x; pair < A.mb; pair += gridDim.x) {
        __syncthreads();
        co_forward(A, S, pair);
        // compact_k[o] = W_j[o] . p_k + b_j[o]   (warp per output)
        for (int r = warp; r < 2 * A.O; r += NTHREADS / 32) {
            const int which = r >= A.O, o = which ? r - A.O : r;
            const float *p = which ? S.p2 : S.p1, *w = A.W_j + (long)o * A.H;
            float s = 0.f;
            for (int h = lane; h < A.H; h += 32) s += w[h] * p[h];
            s = warp_sum(s);
            if (lane == 0) (which ? c2 : c1)[(long)pair * A.O + o] = s + A.b_j[o];
        }
    }
}

struct CoBwd {
    const float *dc1, *dc2;
    float *R, *P1, *P2, *DL1, *DL2, *d_a1, *d_a2;
    float *d_V1, *d_V2, *d_b, *d_wa_1, *d_wa_2;
    CoDet det;          // deterministic mode: per-CTA slots of the vector gradients (det.cuh)
};

__global__ void __launch_bounds__(NTHREADS, 1) coattn_bwd_kernel(const CoArgs A, const CoBwd B) {
    extern __shared__ __align__(16) float smem[];
    const int H = A.H, N1 = A.n1, N2 = A.n2, hd = A.head, O = A.O;
    CoSmem S = co_carve(smem, H, hd);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
    // CTA-local accumulators of the small parameter gradients (flushed once at the end)
    __shared__ float acc_small[2 * BMP_MAX_HIDDEN + 2 * MAXHEAD + 4];
    float *gV1 = acc_small, *gV2 = gV1 + BMP_MAX_HIDDEN, *gwa1 = gV2 + BMP_MAX_HIDDEN, *gwa2 = gwa1 + MAXHEAD,
          *gb = gwa2 + MAXHEAD;
    for (int i = tid; i < 2 * BMP_MAX_HIDDEN + 2 * MAXHEAD + 4; i += NTHREADS) acc_small[i] = 0.f;
    float *dp1 = S.tmp + 4 * AT, *dp2 = dp1 + H;             // [H] each
    float *dpre1 = dp2 + H, *dpre2 = dpre1 + hd * AT;        // [hd][64] each
    float *t1 = S.tmp, *t2 = S.tmp + AT, *cs = S.tmp + 2 * AT, *rsum = S.tmp + 3 * AT;

    for (int pair = blockIdx.x; pair < A.mb; pair += gridDim.x) {
        __syncthreads();
        co_forward(A, S, pair);
        const long r1 = (long)pair * N1, r2 = (long)pair * N2;
        // stash pooled atoms for d_W_j ; dp_k[h] = sum_o W_j[o][h] dc_k[o]
        for (int h = tid; h < 2 * H; h += NTHREADS) {
            const int which = h >= H, hh = which ? h - H : h;
            (which ? B.P2 : B.P1)[(long)pair * H + hh] = (which ? S.p2 : S.p1)[hh];
            const float *dc = (which ? B.dc2 : B.dc1) + (long)pair * O;
            float s = 0.f;
            for (int o = 0; o < O; ++o) s += A.W_j[(long)o * H + hh] * dc[o];
            (which ? dp2 : dp1)[hh] = s;
        }
        __syncthreads();
        // d attn_k[n] = dp_k . a_k[n]  -> softmax backward -> ds_k[n]  (kept in t1/t2 temporarily)
        if (tid < 2 * AT) {
            const int which = tid >= AT, n = tid & 63;
            const float *src = which ? S.a2s : S.a1s, *dp = which ? dp2 : dp1;
            float s = 0.f;
            for (int h = 0; h < H; ++h) s += dp[h] * src[h * AT + n];
            (which ? t2 : t1)[n] = s;     // d attn
        }
        __syncthreads();
        if (warp < 2) {
            const float *at = warp ? S.attn2 : S.attn1;
            float *da = warp ? t2 : t1;
            const int n = warp ? N2 : N1;
            float a = lane < n ? at[lane] * da[lane] : 0.f, b = lane + 32 < n ? at[lane + 32] * da[lane + 32] : 0.f;
            float dot = warp_sum(a + b);
            if (lane < n) da[lane] = at[lane] * (da[lane] - dot);
            if (lane + 32 < n) da[lane + 32] = at[lane + 32] * (da[lane + 32] - dot);
            if (lane >= n) da[lane] = 0.f;
            if (lane + 32 >= n) da[lane + 32] = 0.f;
        }
        __syncthreads();
        // now t1 = ds_1[j], t2 = ds_2[i] (gradient of the pre-softmax scores)
        if (A.variant == BMP_COATTN_FINE) {
            // d wa_k[d] += sum_n ds_k[n] H_k[n][d] ; dpre_k[d][n] = ds_k[n] wa_k[d] (1 - H_k^2)
            for (int idx = tid; idx < 2 * hd * AT; idx += NTHREADS) {
                const int which = idx / (hd * AT), r = idx % (hd * AT), d = r / AT, n = r % AT;
                const float hv = (which ? S.H2 : S.H1)[d * AT + n];
                const float ds = (which ? t2 : t1)[n];
                (which ? dpre2 : dpre1)[d * AT + n] = ds * (which ? A.wa_2 : A.wa_1)[d] * (1.f - hv * hv);
            }
            if (warp < 2 * hd && warp < NTHREADS / 32) {
                for (int r = warp; r < 2 * hd; r += NTHREADS / 32) {
                    const int which = r >= hd, d = which ? r - hd : r;
                    const float *Hk = (which ? S.H2 : S.H1) + d * AT, *ds = which ? t2 : t1;
                    float s = warp_sum(ds[lane] * Hk[lane] + ds[lane + 32] * Hk[lane + 32]);
                    if (lane == 0) (which ? gwa2 : gwa1)[d] += s;
                }
            }
            __syncthreads();
            // softmax-backward inner products:
            //   u1[i] = sum_j L_1[j][i] dL_1[j][i],  dL_1[j][i] = sum_d dpre1[d][j] lt2[d][i]
            //   u2[j] = sum_i L_2[i][j] dL_2[i][j],  dL_2[i][j] = sum_d dpre2[d][i] lt1[d][j]
            float u = 0.f;
            if (tid < AT) {
                const int i = tid;
                for (int j = 0; j < N1; ++j) {
                    float dl = 0.f;
                    for (int d = 0; d < hd; ++d) dl += dpre1[d * AT + j] * S.lt2[d * AT + i];
                    u += S.L1t[i * PLD + j] * dl;
                }
            } else if (tid < 2 * AT) {
                const int j = tid - AT;
                for (int i = 0; i < N2; ++i) {
                    float dl = 0.f;
                    for (int d = 0; d < hd; ++d) dl += dpre2[d * AT + i] * S.lt1[d * AT + j];
                    u += S.L2p[j * PLD + i] * dl;
                }
            }
            // total d lt_k (direct + through the other molecule's H) -> DL_k (global, atom-major)
            for (int idx = tid; idx < 2 * hd * AT; idx += NTHREADS) {
                const int which = idx / (hd * AT), r = idx % (hd * AT), d = r / AT, n = r % AT;
                float s;
                if (!which) {     // d lt_1[j][d] = dpre1[j][d] + sum_i L_2[i][j] dpre2[i][d]
                    s = dpre1[d * AT + n];
                    for (int i = 0; i < N2; ++i) s += S.L2p[n * PLD + i] * dpre2[d * AT + i];
                    if (n < N1) B.DL1[(r1 + n) * hd + d] = s;
                    S.H1[d * AT + n] = s;     // H_k no longer needed: reuse as d lt_k
                } else {          // d lt_2[i][d] = dpre2[i][d] + sum_j L_1[j][i] dpre1[j][d]
                    s = dpre2[d * AT + n];
                    for (int j = 0; j < N1; ++j) s += S.L1t[n * PLD + j] * dpre1[d * AT + j];
                    if (n < N2) B.DL2[(r2 + n) * hd + d] = s;
                    S.H2[d * AT + n] = s;
                }
            }
            __syncthreads();
            if (tid < AT) cs[tid] = u;              // u1[i]  (borrow cs/rsum as u1/u2 for one phase)
            else if (tid < 2 * AT) rsum[tid - AT] = u;   // u2[j]
            __syncthreads();
            // dC^T[j][i] (pre-activation) in place of Cs
            for (int idx = tid; idx < AT * AT; idx += NTHREADS) {
                const int j = idx >> 6, i = idx & 63;
                float dl1 = 0.f, dl2 = 0.f;
                for (int d = 0; d < hd; ++d) {
                    dl1 += dpre1[d * AT + j] * S.lt2[d * AT + i];
                    dl2 += dpre2[d * AT + i] * S.lt1[d * AT + j];
                }
                const float c = S.Cs[idx];
                float g = S.L1t[i * PLD + j] * (dl1 - cs[i]) + S.L2p[j * PLD + i] * (dl2 - rsum[j]);
                S.Cs[idx] = g * act_bwd(A.act, c, c);
            }
        } else {
            // POOL: scores are means of C: dC[i][j] = ds_1[j]/N2 + ds_2[i]/N1
            for (int idx = tid; idx < AT * AT; idx += NTHREADS) {
                const int j = idx >> 6, i = idx & 63;
                const float c = S.Cs[idx];
                const bool live = j < N1 && i < N2;
                float g = live ? t1[j] / (float)N2 + t2[i] / (float)N1 : 0.f;
                S.Cs[idx] = g * act_bwd(A.act, c, c);
            }
        }
        __syncthreads();
        // Ds[i][j] = dC[i][j] (i-major copy, ld DLD, over the L1t region); row/col sums
        for (int idx = tid; idx < AT * AT; idx += NTHREADS) {
            const int j = idx >> 6, i = idx & 63;
            S.L1t[i * DLD + j] = S.Cs[idx];
        }
        __syncthreads();
        if (tid < AT) {             // rsum[i] = sum_j dC[i][j]
            float s = 0.f;
            for (int j = 0; j < N1; ++j) s += S.Cs[j * AT + tid];
            rsum[tid] = s;
        } else if (tid < 2 * AT) {  // cs[j] = sum_i dC[i][j]
            const int j = tid - AT;
            float s = 0.f;
            for (int i = 0; i < N2; ++i) s += S.L1t[i * DLD + j];
            cs[j] = s;
        }
        __syncthreads();
        if (warp == 0) {
            float s = warp_sum(rsum[lane] + rsum[lane + 32]);
            if (lane == 0) gb[0] += s;
        }
        // d V1[h] += sum_j a1[j][h] cs[j] ; d V2[k] += sum_i a2[i][k] rsum[i]   (warp per channel)
        for (int r = warp; r < 2 * H; r += NTHREADS / 32) {
            const int which = r >= H, h = which ? r - H : r;
            const float *src = (which ? S.a2s : S.a1s) + h * AT, *w = which ? rsum : cs;
            float s = warp_sum(src[lane] * w[lane] + src[lane + 32] * w[lane + 32]);
            if (lane == 0) (which ? gV2 : gV1)[h] += s;
        }
        // S^T[k][j] = sum_h W[h][k] a1[j][h]  -> Qs region
        for (int oc = 0; oc * 64 < H; ++oc) {
            float acc[4][4];
            zero_acc(acc);
            gemm64_g<true>(acc, A.W, H, oc * 64, H, H, S.a1s, S.stage);
            if (oc * 64 + ty * 4 < H) tile_store_s(S.Qs, oc * 64, acc);
        }
        __syncthreads();
        // d a2^T[k][i] = sum_j S^T[k][j] dC^T[j][i] + V2[k] rsum[i] + attn_2[i] dp2[k] + sum_d lt_2[d][k] dlt_2[i][d]
        for (int oc = 0; oc * 64 < H; ++oc) {
            const int k0 = oc * 64 + ty * 4;
            if (k0 >= H) continue;
            float acc[4][4];
            zero_acc(acc);
            gemm64_s(acc, S.Qs, AT, oc * 64, AT, S.Cs);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = k0 + q;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int i = tx * 4 + b;
                    float v = acc[q][b] + A.V2[k] * rsum[i] + S.attn2[i] * dp2[k];
                    if (A.variant == BMP_COATTN_FINE)
                        for (int d = 0; d < hd; ++d) v += A.lt_2[(long)d * H + k] * S.H2[d * AT + i];
                    acc[q][b] = v;
                }
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int i = tx * 4 + b;
                if (i >= N2) continue;
                *reinterpret_cast<float4 *>(B.d_a2 + (r2 + i) * H + k0) = make_float4(acc[0][b], acc[1][b], acc[2][b], acc[3][b]);
            }
        }
        __syncthreads();
        // R^T[k][j] = sum_i a2[i][k] dC[i][j]  -> Qs region + global R (atom-major)
        for (int oc = 0; oc * 64 < H; ++oc) {
            if (oc * 64 + ty * 4 >= H) continue;
            float acc[4][4];
            zero_acc(acc);
            // gemm64_s with a DLD-strided Y operand
            {
                const int o0 = oc * 64 + ty * 4, i0 = tx * 4;
                for (int kk = 0; kk < AT; kk += 4) {
                    float4 x[4], y[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) x[a] = *reinterpret_cast<const float4 *>(S.a2s + (o0 + a) * AT + kk);
#pragma unroll
                    for (int q = 0; q < 4; ++q) y[q] = *reinterpret_cast<const float4 *>(S.L1t + (kk + q) * DLD + i0);
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        acc[a][0] += x[a].x * y[0].x + x[a].y * y[1].x + x[a].z * y[2].x + x[a].w * y[3].x;
                        acc[a][1] += x[a].x * y[0].y + x[a].y * y[1].y + x[a].z * y[2].y + x[a].w * y[3].y;
                        acc[a][2] += x[a].x * y[0].z + x[a].y * y[1].z + x[a].z * y[2].z + x[a].w * y[3].z;
                        acc[a][3] += x[a].x * y[0].w + x[a].y * y[1].w + x[a].z * y[2].w + x[a].w * y[3].w;
                    }
                }
            }
            tile_store_g(B.R + r1 * H, H, oc * 64, H, N1, acc);
            // (stored below into Qs after all warps finished reading Qs: Qs is not read in this loop)
            tile_store_s(S.Qs, oc * 64, acc);
        }
        __syncthreads();
        // d a1^T[h][j] = sum_k W[h][k] R^T[k][j] + V1[h] cs[j] + attn_1[j] dp1[h] + sum_d lt_1[d][h] dlt_1[j][d]
        for (int oc = 0; oc * 64 < H; ++oc) {
            float acc[4][4];
            zero_acc(acc);
            gemm64_g<false>(acc, A.W, H, oc * 64, H, H, S.Qs, S.stage);
            const int h0 = oc * 64 + ty * 4;
            if (h0 >= H) continue;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int h = h0 + q;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int j = tx * 4 + b;
                    float v = acc[q][b] + A.V1[h] * cs[j] + S.attn1[j] * dp1[h];
                    if (A.variant == BMP_COATTN_FINE)
                        for (int d = 0; d < hd; ++d) v += A.lt_1[(long)d * H + h] * S.H1[d * AT + j];
                    acc[q][b] = v;
                }
            }
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int j = tx * 4 + b;
                if (j >= N1) continue;
                *reinterpret_cast<float4 *>(B.d_a1 + (r1 + j) * H + h0) = make_float4(acc[0][b], acc[1][b], acc[2][b], acc[3][b]);
            }
        }
    }
    __syncthreads();
    for (int h = tid; h < H; h += NTHREADS) {
        if (B.d_V1) det_put(B.d_V1 + h, B.det.slot(B.det.v(0) + h), gV1[h]);
        if (B.d_V2) det_put(B.d_V2 + h, B.det.slot(B.det.v(1) + h), gV2[h]);
    }
    if (tid < hd && A.variant == BMP_COATTN_FINE) {
        if (B.d_wa_1) det_put(B.d_wa_1 + tid, B.det.slot(B.det.wa(0) + tid), gwa1[tid]);
        if (B.d_wa_2) det_put(B.d_wa_2 + tid, B.det.slot(B.det.wa(1) + tid), gwa2[tid]);
    }
    if (tid == 0 && B.d_b) det_put(B.d_b, B.det.slot(B.det.b()), gb[0]);
}

static int co_check(int mb, int n1, int n2, int H, int O, int head, int variant, const void *ws, size_t ws_bytes) {
    if (mb <= 0) return BMP_ESHAPE;
    if (n1 <= 0 || n1 > BMP_X3_MAX_ATOMS || n2 <= 0 || n2 > BMP_X3_MAX_ATOMS) {
        set_error("coattn: n1=%d n2=%d outside 1..%d", n1, n2, BMP_X3_MAX_ATOMS);
        return BMP_ESHAPE;
    }
    if (H <= 0 || (H & 3) || O <= 0) { set_error("coattn: hidden=%d must be a positive multiple of 4, out_dim=%d > 0", H, O); return BMP_ESHAPE; }
    if (variant == BMP_COATTN_FINE && (head <= 0 || head > MAXHEAD)) { set_error("coattn: head=%d outside 1..%d", head, MAXHEAD); return BMP_ESHAPE; }
    if (n1 > BMP_MAX_ATOMS || n2 > BMP_MAX_ATOMS) {     // coattn_big.cu: C^T and S in a per-CTA slice of the caller's workspace
        const size_t need = bmp_coattn_large_workspace_bytes(n1, n2, H, variant == BMP_COATTN_FINE ? head : 0);
        if (!need) {
            set_error("coattn: n1=%d n2=%d hidden=%d: above %d atoms hidden must be a multiple of 4 <= 192", n1, n2, H, BMP_MAX_ATOMS);
            return BMP_ESHAPE;
        }
        if (!ws || ws_bytes < need) {
            set_error("coattn: n1=%d n2=%d hidden=%d needs a tc_workspace of %zu bytes (bmp_coattn_large_workspace_bytes), %zu given",
                      n1, n2, H, need, ws ? ws_bytes : (size_t)0);
            return BMP_ESHAPE;
        }
        return BMP_OK;
    }
    if (co_smem_floats(H, head > 0 ? head : 1) * sizeof(float) > 227 * 1024) {
        set_error("coattn: hidden=%d does not fit the shared-memory resident kernel", H);
        return BMP_ESHAPE;
    }
    return BMP_OK;
}

}  // namespace bmp

using namespace bmp;

bool bmp_coattn_tc_supported(int H, int head, int variant, bool bwd);
int bmp_coattn_forward_tc(const bmp_coattn_fwd_t *a, void *stream);
int bmp_coattn_backward_tc(const bmp_coattn_bwd_t *a, void *stream);
int bmp_coattn_big(const bmp_coattn_fwd_t *f, const bmp_coattn_bwd_t *bw, void *stream);   // coattn_big.cu: 65..256 atoms

static long long *g_co_dbg = nullptr;
extern "C" void bmp_debug_set_buffer_co(void *p) { g_co_dbg = (long long *)p; }

static CoArgs make_args(int mb, int n1, int n2, int H, int O, int head, int variant, int act,
                        const float *a1, const float *a2, const float *W, const float *V1, const float *V2,
                        const float *b, const float *lt1, const float *lt2, const float *wa1, const float *wa2,
                        const float *Wj, const float *bj) {
    CoArgs A;
    A.dbg = g_co_dbg;
    A.mb = mb; A.n1 = n1; A.n2 = n2; A.H = H; A.O = O; A.head = head > 0 ? head : 1; A.variant = variant; A.act = act;
    A.atoms_1 = a1; A.atoms_2 = a2; A.W = W; A.V1 = V1; A.V2 = V2; A.b = b;
    A.lt_1 = lt1; A.lt_2 = lt2; A.wa_1 = wa1; A.wa_2 = wa2; A.W_j = Wj; A.b_j = bj;
    return A;
}

extern "C" int bmp_coattn_forward(const bmp_coattn_fwd_t *a, void *stream) {
    if (!a || !a->atoms_1 || !a->atoms_2 || !a->W || !a->V1 || !a->V2 || !a->b || !a->W_j || !a->b_j ||
        !a->compact_1 || !a->compact_2) {
        set_error("bmp_coattn_forward: null argument");
        return BMP_EINVAL;
    }
    if (a->variant == BMP_COATTN_FINE && (!a->lt_1 || !a->lt_2 || !a->wa_1 || !a->wa_2)) {
        set_error("bmp_coattn_forward: null head parameters");
        return BMP_EINVAL;
    }
    int rc = co_check(a->mb, a->n1, a->n2, a->hidden, a->out_dim, a->head, a->variant, a->tc_workspace, a->tc_workspace_bytes);
    if (rc) return rc;
    if (!aligned16({a->atoms_1, a->atoms_2, a->W})) { set_error("bmp_coattn_forward: atoms_1, atoms_2, W must be 16-byte aligned"); return BMP_EINVAL; }
    if (a->n1 > BMP_MAX_ATOMS || a->n2 > BMP_MAX_ATOMS) return bmp_coattn_big(a, nullptr, stream);     // fp32 in either mode
    if (a->mode == BMP_MODE_BF16 && bmp_coattn_tc_supported(a->hidden, a->head, a->variant, false)) return bmp_coattn_forward_tc(a, stream);
    CoArgs A = make_args(a->mb, a->n1, a->n2, a->hidden, a->out_dim, a->head, a->variant, a->act, a->atoms_1, a->atoms_2,
                         a->W, a->V1, a->V2, a->b, a->lt_1, a->lt_2, a->wa_1, a->wa_2, a->W_j, a->b_j);
    size_t smem = co_smem_floats(A.H, A.head) * sizeof(float);
    int grid = a->mb < 148 ? a->mb : 148;
    cudaFuncSetAttribute(coattn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    coattn_fwd_kernel<<<grid, NTHREADS, smem, (cudaStream_t)stream>>>(A, a->compact_1, a->compact_2);
    count_launch();
    return check_launch("coattn_fwd_kernel");
}

static int coattn_backward_impl(const bmp_coattn_bwd_t *a, void *stream) {
    if (!a || !a->atoms_1 || !a->atoms_2 || !a->W || !a->V1 || !a->V2 || !a->b || !a->W_j || !a->b_j ||
        !a->d_compact_1 || !a->d_compact_2 || !a->R || !a->P1 || !a->P2 || !a->d_atoms_1 || !a->d_atoms_2) {
        set_error("bmp_coattn_backward: null argument");
        return BMP_EINVAL;
    }
    const bool fine = a->variant == BMP_COATTN_FINE;
    if (fine && (!a->lt_1 || !a->lt_2 || !a->wa_1 || !a->wa_2 || !a->DL1 || !a->DL2)) {
        set_error("bmp_coattn_backward: null head parameters / workspaces");
        return BMP_EINVAL;
    }
    int rc = co_check(a->mb, a->n1, a->n2, a->hidden, a->out_dim, a->head, a->variant, a->tc_workspace, a->tc_workspace_bytes);
    if (rc) return rc;
    if (a->hidden > BMP_MAX_HIDDEN) { set_error("coattn backward: hidden > %d", BMP_MAX_HIDDEN); return BMP_ESHAPE; }
    if (!aligned16({a->atoms_1, a->atoms_2, a->W, a->R, a->d_atoms_1, a->d_atoms_2})) { set_error("bmp_coattn_backward: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    const bool big = a->n1 > BMP_MAX_ATOMS || a->n2 > BMP_MAX_ATOMS;     // fp32 kernel and fp32 weight gradients in either mode
    const bool tc_data = !big && a->mode == BMP_MODE_BF16 && bmp_coattn_tc_supported(a->hidden, a->head, a->variant, true);
    if (tc_data) {     // also accumulates d W, d lt_k, d V_k, d wa_k, d b inside the kernel
        if ((rc = bmp_coattn_backward_tc(a, stream))) return rc;
    } else if (big) {
        if ((rc = bmp_coattn_big(nullptr, a, stream))) return rc;
    } else {
        CoArgs A = make_args(a->mb, a->n1, a->n2, a->hidden, a->out_dim, a->head, a->variant, a->act, a->atoms_1, a->atoms_2,
                             a->W, a->V1, a->V2, a->b, a->lt_1, a->lt_2, a->wa_1, a->wa_2, a->W_j, a->b_j);
        CoBwd B;
        B.dc1 = a->d_compact_1; B.dc2 = a->d_compact_2; B.R = a->R; B.P1 = a->P1; B.P2 = a->P2;
        B.DL1 = a->DL1; B.DL2 = a->DL2; B.d_a1 = a->d_atoms_1; B.d_a2 = a->d_atoms_2;
        B.d_V1 = a->d_V1; B.d_V2 = a->d_V2; B.d_b = a->d_b; B.d_wa_1 = a->d_wa_1; B.d_wa_2 = a->d_wa_2;
        size_t smem = co_smem_floats(A.H, A.head) * sizeof(float);
        int grid = a->mb < 148 ? a->mb : 148;
        Partials pt((cudaStream_t)stream);
        if ((rc = co_det_begin(pt, B.det, A.H, grid))) return rc;
        cudaFuncSetAttribute(coattn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        coattn_bwd_kernel<<<grid, NTHREADS, smem, (cudaStream_t)stream>>>(A, B);
        count_launch();
        if ((rc = check_launch("coattn_bwd_kernel"))) return rc;
        if ((rc = co_det_end(pt, B.det, grid, fine ? a->head : 0, nullptr, nullptr, nullptr, a->d_V1, a->d_V2, a->d_wa_1, a->d_wa_2,
                             a->d_b, false, "det_reduce_kernel (coattn_bwd)")))
            return rc;
    }
    const int H = a->hidden, O = a->out_dim, hd = a->head;
    const long rows1 = (long)a->mb * a->n1, rows2 = (long)a->mb * a->n2;
    // d W[h][k] += sum_{pairs,j} a1[j][h] R[j][k]
    const bool tcw = !big && a->mode == BMP_MODE_BF16 && (H == 64 || H == 128 || H == 256);
    auto WG = [&](const float *A_, int lda, const float *B_, float *C_, long r_, int M_) -> int {
        if (tcw && (M_ & 3) == 0) return bmp_wgrad_tc(A_, lda, B_, H, C_, H, r_, M_, H, nullptr, 1, stream);
        return bmp_wgrad(A_, lda, B_, H, C_, H, r_, M_, H, stream);
    };
    if (!tc_data && a->d_W && (rc = WG(a->atoms_1, H, a->R, a->d_W, rows1, H))) return rc;
    if (a->d_W_j) {
        if ((rc = WG(a->d_compact_1, O, a->P1, a->d_W_j, a->mb, O))) return rc;
        if ((rc = WG(a->d_compact_2, O, a->P2, a->d_W_j, a->mb, O))) return rc;
    }
    if (a->d_b_j) {
        if ((rc = bmp_colsum(a->d_compact_1, O, a->d_b_j, 1, a->mb, O, stream))) return rc;
        if ((rc = bmp_colsum(a->d_compact_2, O, a->d_b_j, 1, a->mb, O, stream))) return rc;
    }
    if (fine && !tc_data) {
        if (a->d_lt_1 && (rc = bmp_wgrad(a->DL1, hd, a->atoms_1, H, a->d_lt_1, H, rows1, hd, H, stream))) return rc;
        if (a->d_lt_2 && (rc = bmp_wgrad(a->DL2, hd, a->atoms_2, H, a->d_lt_2, H, rows2, hd, H, stream))) return rc;
    }
    return BMP_OK;
}

// Bytes of det_scratch (deterministic mode, det.cuh) that bmp_coattn_backward needs for this filled-in struct; 0 = no shape to cover.
extern "C" size_t bmp_coattn_backward_det_bytes(const bmp_coattn_bwd_t *a) {
    if (!a) return 0;
    if (a->mb <= 0 || a->n1 <= 0 || a->n2 <= 0 || a->hidden <= 0 || a->out_dim <= 0) return 0;
    const int H = a->hidden, O = a->out_dim, M = H > O ? (H > a->head ? H : a->head) : (O > a->head ? O : a->head);
    return det_max({det_coattn_bytes(a->mb, H), det_wgrad_bytes(M, H), det_wgrad_tc_bytes(M, H), det_colsum_bytes(O)});
}
extern "C" int bmp_coattn_backward(const bmp_coattn_bwd_t *a, void *stream) {
    if (a && a->det_scratch) {
        int rc = det_check("bmp_coattn_backward", a->det_scratch, a->det_scratch_bytes, bmp_coattn_backward_det_bytes(a));
        if (rc) return rc;
    }
    DetScope ds(a ? a->det_scratch : nullptr, a ? a->det_scratch_bytes : 0);
    return coattn_backward_impl(a, stream);
}
