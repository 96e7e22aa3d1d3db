// coattn_big.cu -- fine-grained co-attention (variants FINE and POOL) for pairs where a molecule has 65..256 atoms, fp32.
// Same formulas as coattn.cu (nie_coattention.py:335-396, PoolingFineCoattention.py:31-83), one pair per CTA of a persistent
// grid.  The N1 x N2 energy C^T and the product S = a1 W do not fit shared memory at this size, so each CTA keeps them in its own
// slice of a caller-owned workspace (at most 448 KB a slice, 148 slices: L2-resident).  Every contraction runs as 64 x 64
// register tiles with both operands staged through shared memory; the softmaxes never materialise: L_1 / L_2 are recomputed from
// C^T and the row / column statistics wherever they are needed.
//   S[j][k]   = sum_h a1[j][h] W[h][k]
//   C^T[j][i] = act(sum_k S[j][k] a2[i][k] + V1.a1_j + V2.a2_i + b)          i: atoms_2, j: atoms_1
// The backward recomputes the forward into the same slice, overwrites C^T with dC^T and writes R, P1/P2, DL1/DL2 and d_atoms_k
// with the meanings of bmp_coattn_bwd_t, so the parameter-gradient calls of bmp_coattn_backward are shared with coattn.cu.
#include <cstring>
#include "det.cuh"

namespace bmp {
namespace big {

constexpr int NMAX = BMP_X3_MAX_ATOMS;   // 256 atoms per molecule
constexpr int HMAX = 192;                // widest atoms: same bound as the shared-memory-resident kernel of coattn.cu
constexpr int MAXHEAD = 16;
constexpr int CTAS = 148;                // persistent grid = workspace slices
constexpr int TLD = 65;                  // ld of the L_1 / L_2 tiles
constexpr int SLD = 68;                  // ld of the staged operand chunks [KT][SLD]

// element (r, c) of a global matrix: t ? p[c * ld + r] : p[r * ld + c]
struct Op {
    const float *p;
    int ld;
    bool t;
};

__host__ __device__ inline int c_ld(int n2) { return (n2 + 3) & ~3; }
__host__ __device__ inline size_t slice_floats(int n1, int n2, int H) {
    return (((size_t)n1 * c_ld(n2) + (size_t)n1 * H) + 63) & ~(size_t)63;
}

struct Smem {
    float *v1, *v2, *m1, *s1, *m2, *s2, *attn1, *attn2, *u1, *u2, *cs, *rsum;   // [NMAX]
    float *lt1, *lt2, *H1, *H2, *dp1, *dp2;                                    // [head][NMAX]  (dp: dpre_k)
    float *p1, *p2, *dc1, *dc2;                                                // [H]           (dc: dp_k = W_j^T dc_k)
    float *La, *Lb;                                                            // [64][TLD]
    float *sx, *sy;                                                            // [2][KT][SLD]
};

__host__ __device__ inline size_t smem_floats(int H, int head) {
    return (size_t)12 * NMAX + (size_t)6 * head * NMAX + 4 * H + 2 * AT * TLD + 4 * KT * SLD + 16;
}

__device__ inline Smem carve(float *p, int H, int hd) {
    Smem s;
    float **v[12] = {&s.v1, &s.v2, &s.m1, &s.s1, &s.m2, &s.s2, &s.attn1, &s.attn2, &s.u1, &s.u2, &s.cs, &s.rsum};
    for (int q = 0; q < 12; ++q) { *v[q] = p; p += NMAX; }
    float **w[6] = {&s.lt1, &s.lt2, &s.H1, &s.H2, &s.dp1, &s.dp2};
    for (int q = 0; q < 6; ++q) { *w[q] = p; p += hd * NMAX; }
    s.p1 = p; p += H;
    s.p2 = p; p += H;
    s.dc1 = p; p += H;
    s.dc2 = p; p += H;
    p = (float *)(((uintptr_t)p + 15) & ~(uintptr_t)15);
    s.La = p; p += AT * TLD;
    s.Lb = p; p += AT * TLD;
    s.sx = p; p += 2 * KT * SLD;
    s.sy = p;
    return s;
}

struct Args {
    int mb, n1, n2, H, O, head, variant, act;
    const float *atoms_1, *atoms_2, *W, *V1, *V2, *b, *lt_1, *lt_2, *wa_1, *wa_2, *W_j, *b_j;
    float *ws;                                  // CTAS slices of slice_floats(n1, n2, H)
    float *c1, *c2;                             // forward outputs
    const float *dc1, *dc2;                     // backward
    float *R, *P1, *P2, *DL1, *DL2, *d_a1, *d_a2;
    float *d_V1, *d_V2, *d_b, *d_wa_1, *d_wa_2;
    CoDet det;                                  // deterministic mode: per-CTA slots of the vector gradients (det.cuh)
};

__device__ __forceinline__ float wsum(float v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float wmax(float v) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// one KT chunk [KT k][64 r] of op element (r0 + r, k0 + k) into shared memory with 4-byte async copies that zero-fill outside
// r < rlim, k < K (src-size 0: nothing is read).  Coalesced along the contiguous index.
__device__ __forceinline__ void stage(float *dst, const Op &X, int r0, int rlim, int k0, int K) {
    for (int e = threadIdx.x; e < KT * AT; e += NTHREADS) {
        int r, k;
        if (X.t) { r = e & 63; k = e >> 6; } else { k = e & (KT - 1); r = e >> 5; }
        const int rr = r0 + r, kk = k0 + k;
        const bool live = rr < rlim && kk < K;
        const float *src = live ? (X.t ? X.p + (long)kk * X.ld + rr : X.p + (long)rr * X.ld + kk) : X.p;
        const unsigned d = (unsigned)__cvta_generic_to_shared(dst + k * SLD + r);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(src), "r"(live ? 4 : 0));
    }
}

// C(o, i) = sum_{k < K} X(o, k) Y(k, i) over o < olim, i < ilim in 64 x 64 tiles (4 x 4 per thread); epi(o, i, value) per element.
// Y is passed as its transpose (element (i, k)) so both operands stage the same way.  The next KT chunk is in flight while the
// current one is contracted (two staging buffers per operand).  Entry and exit synchronised.
template <class Epi>
__device__ void gemm(const Op &X, int olim, const Op &Yt, int ilim, int K, float *sx, float *sy, Epi epi) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4, o0 = ty * 4, i0 = tx * 4;
    constexpr int BUF = KT * SLD;
    const int nk = (K + KT - 1) / KT;
    for (int ob = 0; ob < olim; ob += AT)
        for (int ib = 0; ib < ilim; ib += AT) {
            float acc[4][4];
            zero_acc(acc);
            stage(sx, X, ob, olim, 0, K);
            stage(sy, Yt, ib, ilim, 0, K);
            cp_async_commit();
            for (int c = 0; c < nk; ++c) {
                if (c + 1 < nk) {
                    stage(sx + ((c + 1) & 1) * BUF, X, ob, olim, (c + 1) * KT, K);
                    stage(sy + ((c + 1) & 1) * BUF, Yt, ib, ilim, (c + 1) * KT, K);
                    cp_async_commit();
                    cp_async_wait<1>();
                } else {
                    cp_async_wait<0>();
                }
                __syncthreads();
                const float *cx = sx + (c & 1) * BUF, *cy = sy + (c & 1) * BUF;
#pragma unroll 8
                for (int k = 0; k < KT; ++k) {
                    const float4 x = *reinterpret_cast<const float4 *>(cx + k * SLD + o0);
                    const float4 y = *reinterpret_cast<const float4 *>(cy + k * SLD + i0);
                    const float xa[4] = {x.x, x.y, x.z, x.w}, ya[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int q = 0; q < 4; ++q) acc[a][q] += xa[a] * ya[q];
                }
                __syncthreads();
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (ob + o0 + a < olim && ib + i0 + q < ilim) epi(ob + o0 + a, ib + i0 + q, acc[a][q]);
        }
    __syncthreads();
}

// L_1[j][i] = softmax over atoms_1 (index j) of column i; L_2[i][j] = softmax over atoms_2 (index i) of row j
__device__ __forceinline__ float l1v(float c, const Smem &S, int i) { return expf(c - S.m1[i]) / S.s1[i]; }
__device__ __forceinline__ float l2v(float c, const Smem &S, int j) { return expf(c - S.m2[j]) / S.s2[j]; }

// Over all 64 x 64 tiles of C^T: La = L_1, Lb = L_2 (0 outside the molecules), then
//   yj[d][j] += sum_i Pj[j][i] xi[d][i],   yi[d][i] += sum_j Pi[j][i] xj[d][j]
// with (Pj, Pi) = (La, Lb) for the forward H_1 / H_2 and (Lb, La) for the backward G_2 / G_1.  A (d, row) entry of yj / yi is
// owned by one thread in every tile.
__device__ void l_pass(const float *Ct, int ldc, int N1, int N2, int hd, const Smem &S, bool swap, const float *xj,
                       const float *xi, float *yj, float *yi) {
    const float *Pj = swap ? S.Lb : S.La, *Pi = swap ? S.La : S.Lb;
    for (int jb = 0; jb < N1; jb += AT)
        for (int ib = 0; ib < N2; ib += AT) {
            for (int e = threadIdx.x; e < AT * AT; e += NTHREADS) {
                const int j = e >> 6, i = e & 63, jj = jb + j, ii = ib + i;
                float a = 0.f, b = 0.f;
                if (jj < N1 && ii < N2) {
                    const float c = Ct[(long)jj * ldc + ii];
                    a = l1v(c, S, ii);
                    b = l2v(c, S, jj);
                }
                S.La[j * TLD + i] = a;
                S.Lb[j * TLD + i] = b;
            }
            __syncthreads();
            const int ni = min(AT, N2 - ib), nj = min(AT, N1 - jb);
            for (int e = threadIdx.x; e < hd * AT; e += NTHREADS) {
                const int d = e >> 6, r = e & 63;
                if (jb + r < N1) {
                    float s = 0.f;
                    for (int i = 0; i < ni; ++i) s += Pj[r * TLD + i] * xi[d * NMAX + ib + i];
                    yj[d * NMAX + jb + r] += s;
                }
                if (ib + r < N2) {
                    float s = 0.f;
                    for (int j = 0; j < nj; ++j) s += Pi[j * TLD + r] * xj[d * NMAX + jb + j];
                    yi[d * NMAX + ib + r] += s;
                }
            }
            __syncthreads();
        }
}

// softmax over n <= NMAX entries of x by one warp, in place
__device__ __forceinline__ void softmax_warp(float *x, int n, int lane) {
    float m = -INFINITY;
    for (int q = lane; q < n; q += 32) m = fmaxf(m, x[q]);
    m = wmax(m);
    float s = 0.f;
    for (int q = lane; q < n; q += 32) s += expf(x[q] - m);
    s = wsum(s);
    for (int q = lane; q < n; q += 32) x[q] = expf(x[q] - m) / s;
}

// Forward of one pair.  On exit: the slice holds C^T (post-activation) and S; m*, s*, lt*, H*, attn*, p* are valid.
__device__ void forward(const Args &A, const Smem &S, float *Ct, float *Sg, int pair) {
    const int H = A.H, N1 = A.n1, N2 = A.n2, hd = A.head, ldc = c_ld(N2);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *a1 = A.atoms_1 + (long)pair * N1 * H, *a2 = A.atoms_2 + (long)pair * N2 * H;
    // v1[j] = V1 . a1_j, v2[i] = V2 . a2_i   (warp per atom)
    for (int r = warp; r < N1 + N2; r += NTHREADS / 32) {
        const bool one = r < N1;
        const float *x = one ? a1 + (long)r * H : a2 + (long)(r - N1) * H, *V = one ? A.V1 : A.V2;
        float s = 0.f;
        for (int h = lane; h < H; h += 32) s += V[h] * x[h];
        s = wsum(s);
        if (lane == 0) (one ? S.v1 : S.v2)[one ? r : r - N1] = s;
    }
    // S = a1 W
    gemm(Op{a1, H, false}, N1, Op{A.W, H, true}, H, H, S.sx, S.sy, [&](int j, int k, float v) { Sg[(long)j * H + k] = v; });
    // C^T = act(S a2^T + v1 + v2 + b)
    const float bias = A.b[0];
    gemm(Op{Sg, H, false}, N1, Op{a2, H, false}, N2, H, S.sx, S.sy,
         [&](int j, int i, float v) { Ct[(long)j * ldc + i] = act_fwd(A.act, v + S.v1[j] + S.v2[i] + bias); });
    if (A.variant == BMP_COATTN_FINE) {
        // m1/s1 over j for each column i (thread per i); m2/s2 over i for each row j (warp per j)
        if (tid < N2) {
            float m = -INFINITY, s = 0.f;
            for (int j = 0; j < N1; ++j) m = fmaxf(m, Ct[(long)j * ldc + tid]);
            for (int j = 0; j < N1; ++j) s += expf(Ct[(long)j * ldc + tid] - m);
            S.m1[tid] = m; S.s1[tid] = s;
        }
        for (int j = warp; j < N1; j += NTHREADS / 32) {
            const float *row = Ct + (long)j * ldc;
            float m = -INFINITY;
            for (int i = lane; i < N2; i += 32) m = fmaxf(m, row[i]);
            m = wmax(m);
            float s = 0.f;
            for (int i = lane; i < N2; i += 32) s += expf(row[i] - m);
            s = wsum(s);
            if (lane == 0) { S.m2[j] = m; S.s2[j] = s; }
        }
        // lt_k[d][n] = lt_k[d] . a_k[n]
        gemm(Op{a1, H, false}, N1, Op{A.lt_1, H, false}, hd, H, S.sx, S.sy, [&](int j, int d, float v) { S.lt1[d * NMAX + j] = v; });
        gemm(Op{a2, H, false}, N2, Op{A.lt_2, H, false}, hd, H, S.sx, S.sy, [&](int i, int d, float v) { S.lt2[d * NMAX + i] = v; });
        for (int e = tid; e < hd * NMAX; e += NTHREADS) { S.H1[e] = S.lt1[e]; S.H2[e] = S.lt2[e]; }
        __syncthreads();
        // H_1[j][d] = tanh(lt_1[j][d] + sum_i L_1[j][i] lt_2[i][d]);  H_2[i][d] = tanh(lt_2[i][d] + sum_j L_2[i][j] lt_1[j][d])
        l_pass(Ct, ldc, N1, N2, hd, S, false, S.lt1, S.lt2, S.H1, S.H2);
        for (int e = tid; e < hd * NMAX; e += NTHREADS) { S.H1[e] = tanhf(S.H1[e]); S.H2[e] = tanhf(S.H2[e]); }
        __syncthreads();
        for (int r = tid; r < N1 + N2; r += NTHREADS) {
            const bool one = r < N1;
            const int n = one ? r : r - N1;
            const float *Hk = one ? S.H1 : S.H2, *wa = one ? A.wa_1 : A.wa_2;
            float s = 0.f;
            for (int d = 0; d < hd; ++d) s += wa[d] * Hk[d * NMAX + n];
            (one ? S.attn1 : S.attn2)[n] = s;
        }
    } else {   // POOL: attn_1 = softmax_j(mean_i C), attn_2 = softmax_i(mean_j C)
        if (tid < N2) {
            float s = 0.f;
            for (int j = 0; j < N1; ++j) s += Ct[(long)j * ldc + tid];
            S.attn2[tid] = s / (float)N1;
        }
        for (int j = warp; j < N1; j += NTHREADS / 32) {
            float s = 0.f;
            for (int i = lane; i < N2; i += 32) s += Ct[(long)j * ldc + i];
            s = wsum(s);
            if (lane == 0) S.attn1[j] = s / (float)N2;
        }
    }
    __syncthreads();
    if (warp == 0) softmax_warp(S.attn1, N1, lane);
    if (warp == 1) softmax_warp(S.attn2, N2, lane);
    __syncthreads();
    // pooled atoms p_k[h] = sum_n attn_k[n] a_k[n][h]   (thread per channel)
    for (int r = tid; r < 2 * H; r += NTHREADS) {
        const bool one = r < H;
        const int h = one ? r : r - H, n = one ? N1 : N2;
        const float *x = (one ? a1 : a2) + h, *at = one ? S.attn1 : S.attn2;
        float s = 0.f;
        for (int q = 0; q < n; ++q) s += at[q] * x[(long)q * H];
        (one ? S.p1 : S.p2)[h] = s;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(NTHREADS, 1) coattn_big_fwd_kernel(const Args A) {
    extern __shared__ __align__(16) float smem[];
    const Smem S = carve(smem, A.H, A.head);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *Ct = A.ws + (size_t)blockIdx.x * slice_floats(A.n1, A.n2, A.H), *Sg = Ct + (size_t)A.n1 * c_ld(A.n2);
    for (int pair = blockIdx.x; pair < A.mb; pair += gridDim.x) {
        __syncthreads();
        forward(A, S, Ct, Sg, pair);
        // compact_k[o] = W_j[o] . p_k + b_j[o]   (warp per output)
        for (int r = warp; r < 2 * A.O; r += NTHREADS / 32) {
            const bool one = r < A.O;
            const int o = one ? r : r - A.O;
            const float *p = one ? S.p1 : S.p2, *w = A.W_j + (long)o * A.H;
            float s = 0.f;
            for (int h = lane; h < A.H; h += 32) s += w[h] * p[h];
            s = wsum(s);
            if (lane == 0) (one ? A.c1 : A.c2)[(long)pair * A.O + o] = s + A.b_j[o];
        }
    }
}

__global__ void __launch_bounds__(NTHREADS, 1) coattn_big_bwd_kernel(const Args A) {
    extern __shared__ __align__(16) float smem[];
    const int H = A.H, N1 = A.n1, N2 = A.n2, hd = A.head, O = A.O, ldc = c_ld(N2);
    const Smem S = carve(smem, H, hd);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool fine = A.variant == BMP_COATTN_FINE;
    // CTA-local accumulators of the small parameter gradients (flushed once at the end)
    __shared__ float gV1[HMAX], gV2[HMAX], gwa1[MAXHEAD], gwa2[MAXHEAD], gb;
    for (int q = tid; q < HMAX; q += NTHREADS) gV1[q] = gV2[q] = 0.f;
    if (tid < MAXHEAD) gwa1[tid] = gwa2[tid] = 0.f;
    if (tid == 0) gb = 0.f;
    float *Ct = A.ws + (size_t)blockIdx.x * slice_floats(N1, N2, H), *Sg = Ct + (size_t)N1 * ldc;

    for (int pair = blockIdx.x; pair < A.mb; pair += gridDim.x) {
        __syncthreads();
        forward(A, S, Ct, Sg, pair);
        const long r1 = (long)pair * N1, r2 = (long)pair * N2;
        const float *a1 = A.atoms_1 + r1 * H, *a2 = A.atoms_2 + r2 * H;
        // pooled atoms for d_W_j;  dp_k[h] = sum_o W_j[o][h] dc_k[o]
        for (int r = tid; r < 2 * H; r += NTHREADS) {
            const bool one = r < H;
            const int h = one ? r : r - H;
            (one ? A.P1 : A.P2)[(long)pair * H + h] = (one ? S.p1 : S.p2)[h];
            const float *dc = (one ? A.dc1 : A.dc2) + (long)pair * O;
            float s = 0.f;
            for (int o = 0; o < O; ++o) s += A.W_j[(long)o * H + h] * dc[o];
            (one ? S.dc1 : S.dc2)[h] = s;
        }
        __syncthreads();
        // d attn_k[n] = dp_k . a_k[n]  (warp per atom, into u1 / u2)
        for (int r = warp; r < N1 + N2; r += NTHREADS / 32) {
            const bool one = r < N1;
            const float *x = one ? a1 + (long)r * H : a2 + (long)(r - N1) * H, *dp = one ? S.dc1 : S.dc2;
            float s = 0.f;
            for (int h = lane; h < H; h += 32) s += dp[h] * x[h];
            s = wsum(s);
            if (lane == 0) (one ? S.u1 : S.u2)[one ? r : r - N1] = s;
        }
        __syncthreads();
        // softmax backward: ds_k[n] = attn_k[n] (d attn_k[n] - sum attn_k d attn_k)   -> cs (side 1) / rsum (side 2)
        if (warp < 2) {
            const float *at = warp ? S.attn2 : S.attn1, *da = warp ? S.u2 : S.u1;
            float *ds = warp ? S.rsum : S.cs;
            const int n = warp ? N2 : N1;
            float dot = 0.f;
            for (int q = lane; q < n; q += 32) dot += at[q] * da[q];
            dot = wsum(dot);
            for (int q = lane; q < n; q += 32) ds[q] = at[q] * (da[q] - dot);
        }
        __syncthreads();
        if (fine) {
            // dpre_k[d][n] = ds_k[n] wa_k[d] (1 - H_k^2);  d wa_k[d] += sum_n ds_k[n] H_k[d][n]
            for (int e = tid; e < hd * NMAX; e += NTHREADS) {
                const int d = e / NMAX, n = e % NMAX;
                const float h1 = S.H1[e], h2 = S.H2[e];
                S.dp1[e] = n < N1 ? S.cs[n] * A.wa_1[d] * (1.f - h1 * h1) : 0.f;
                S.dp2[e] = n < N2 ? S.rsum[n] * A.wa_2[d] * (1.f - h2 * h2) : 0.f;
            }
            for (int r = warp; r < 2 * hd; r += NTHREADS / 32) {
                const bool one = r < hd;
                const int d = one ? r : r - hd, n = one ? N1 : N2;
                const float *Hk = (one ? S.H1 : S.H2) + d * NMAX, *ds = one ? S.cs : S.rsum;
                float s = 0.f;
                for (int q = lane; q < n; q += 32) s += ds[q] * Hk[q];
                s = wsum(s);
                if (lane == 0) (one ? gwa1 : gwa2)[d] += s;
            }
            __syncthreads();
            // G_2[d][j] = sum_i L_2[i][j] dpre2[d][i] and G_1[d][i] = sum_j L_1[j][i] dpre1[d][j], accumulated onto dpre into H_k:
            // H_1 <- d lt_1 = dpre1 + G_2,  H_2 <- d lt_2 = dpre2 + G_1
            for (int e = tid; e < hd * NMAX; e += NTHREADS) { S.H1[e] = S.dp1[e]; S.H2[e] = S.dp2[e]; }
            __syncthreads();
            l_pass(Ct, ldc, N1, N2, hd, S, true, S.dp1, S.dp2, S.H1, S.H2);
            // softmax-backward inner products  u1[i] = sum_j L_1[j][i] dL_1[j][i] = sum_d lt2[d][i] G_1[d][i],
            //                                  u2[j] = sum_i L_2[i][j] dL_2[i][j] = sum_d lt1[d][j] G_2[d][j];  DL_k out
            for (int r = tid; r < N1 + N2; r += NTHREADS) {
                const bool one = r < N1;
                const int n = one ? r : r - N1;
                const float *dl = one ? S.H1 : S.H2, *dpre = one ? S.dp1 : S.dp2, *lt = one ? S.lt1 : S.lt2;
                float *DL = one ? A.DL1 + (r1 + n) * hd : A.DL2 + (r2 + n) * hd;
                float u = 0.f;
                for (int d = 0; d < hd; ++d) {
                    const float v = dl[d * NMAX + n];
                    u += lt[d * NMAX + n] * (v - dpre[d * NMAX + n]);
                    DL[d] = v;
                }
                (one ? S.u2 : S.u1)[n] = u;
            }
            __syncthreads();
            // dC^T[j][i] (pre-activation) in place of C^T
            for (long e = tid; e < (long)N1 * N2; e += NTHREADS) {
                const int j = (int)(e / N2), i = (int)(e - (long)j * N2);
                float dl1 = 0.f, dl2 = 0.f;
                for (int d = 0; d < hd; ++d) {
                    dl1 += S.dp1[d * NMAX + j] * S.lt2[d * NMAX + i];
                    dl2 += S.dp2[d * NMAX + i] * S.lt1[d * NMAX + j];
                }
                const float c = Ct[(long)j * ldc + i];
                const float g = l1v(c, S, i) * (dl1 - S.u1[i]) + l2v(c, S, j) * (dl2 - S.u2[j]);
                Ct[(long)j * ldc + i] = g * act_bwd(A.act, c, c);
            }
        } else {
            // POOL: scores are means of C: dC[i][j] = ds_1[j] / N2 + ds_2[i] / N1
            for (long e = tid; e < (long)N1 * N2; e += NTHREADS) {
                const int j = (int)(e / N2), i = (int)(e - (long)j * N2);
                const float c = Ct[(long)j * ldc + i];
                Ct[(long)j * ldc + i] = (S.cs[j] / (float)N2 + S.rsum[i] / (float)N1) * act_bwd(A.act, c, c);
            }
        }
        __syncthreads();
        // ds_k are consumed: u1 <- rsum[i] = sum_j dC[i][j], u2 <- cs[j] = sum_i dC[i][j]
        if (tid < N2) {
            float s = 0.f;
            for (int j = 0; j < N1; ++j) s += Ct[(long)j * ldc + tid];
            S.u1[tid] = s;
        }
        for (int j = warp; j < N1; j += NTHREADS / 32) {
            float s = 0.f;
            for (int i = lane; i < N2; i += 32) s += Ct[(long)j * ldc + i];
            s = wsum(s);
            if (lane == 0) S.u2[j] = s;
        }
        __syncthreads();
        const float *rs = S.u1, *cs = S.u2;
        if (warp == 0) {
            float s = 0.f;
            for (int i = lane; i < N2; i += 32) s += rs[i];
            s = wsum(s);
            if (lane == 0) gb += s;
        }
        // d V1[h] += sum_j a1[j][h] cs[j] ; d V2[h] += sum_i a2[i][h] rsum[i]   (thread per channel)
        for (int r = tid; r < 2 * H; r += NTHREADS) {
            const bool one = r < H;
            const int h = one ? r : r - H, n = one ? N1 : N2;
            const float *x = (one ? a1 : a2) + h, *w = one ? cs : rs;
            float s = 0.f;
            for (int q = 0; q < n; ++q) s += x[(long)q * H] * w[q];
            (one ? gV1 : gV2)[h] += s;
        }
        // R[j][k] = sum_i dC^T[j][i] a2[i][k]
        float *R = A.R + r1 * H;
        gemm(Op{Ct, ldc, false}, N1, Op{a2, H, true}, H, N2, S.sx, S.sy, [&](int j, int k, float v) { R[(long)j * H + k] = v; });
        // d a1[j][h] = sum_k R[j][k] W[h][k] + V1[h] cs[j] + attn_1[j] dp1[h] + sum_d lt_1[d][h] d lt_1[j][d]
        float *da1 = A.d_a1 + r1 * H, *da2 = A.d_a2 + r2 * H;
        gemm(Op{R, H, false}, N1, Op{A.W, H, false}, H, H, S.sx, S.sy, [&](int j, int h, float v) {
            v += A.V1[h] * cs[j] + S.attn1[j] * S.dc1[h];
            if (fine)
                for (int d = 0; d < hd; ++d) v += A.lt_1[(long)d * H + h] * S.H1[d * NMAX + j];
            da1[(long)j * H + h] = v;
        });
        // d a2[i][k] = sum_j dC^T[j][i] S[j][k] + V2[k] rsum[i] + attn_2[i] dp2[k] + sum_d lt_2[d][k] d lt_2[i][d]
        gemm(Op{Ct, ldc, true}, N2, Op{Sg, H, true}, H, N1, S.sx, S.sy, [&](int i, int k, float v) {
            v += A.V2[k] * rs[i] + S.attn2[i] * S.dc2[k];
            if (fine)
                for (int d = 0; d < hd; ++d) v += A.lt_2[(long)d * H + k] * S.H2[d * NMAX + i];
            da2[(long)i * H + k] = v;
        });
    }
    __syncthreads();
    for (int h = tid; h < H; h += NTHREADS) {
        if (A.d_V1) det_put(A.d_V1 + h, A.det.slot(A.det.v(0) + h), gV1[h]);
        if (A.d_V2) det_put(A.d_V2 + h, A.det.slot(A.det.v(1) + h), gV2[h]);
    }
    if (tid < hd && fine) {
        if (A.d_wa_1) det_put(A.d_wa_1 + tid, A.det.slot(A.det.wa(0) + tid), gwa1[tid]);
        if (A.d_wa_2) det_put(A.d_wa_2 + tid, A.det.slot(A.det.wa(1) + tid), gwa2[tid]);
    }
    if (tid == 0 && A.d_b) det_put(A.d_b, A.det.slot(A.det.b()), gb);
}

}  // namespace big
}  // namespace bmp

using namespace bmp;
using namespace bmp::big;

extern "C" size_t bmp_coattn_large_workspace_bytes(int n1, int n2, int hidden, int head) {
    if (n1 <= 0 || n2 <= 0 || (n1 <= BMP_MAX_ATOMS && n2 <= BMP_MAX_ATOMS) || n1 > NMAX || n2 > NMAX) return 0;
    if (hidden <= 0 || (hidden & 3) || hidden > HMAX || head < 0 || head > MAXHEAD) return 0;
    return (size_t)CTAS * slice_floats(n1, n2, hidden) * sizeof(float) + 256;
}

// Called by bmp_coattn_forward / _backward (coattn.cu) once the arguments are validated and the workspace is known to be large
// enough.  bwd == nullptr: forward.
int bmp_coattn_big(const bmp_coattn_fwd_t *f, const bmp_coattn_bwd_t *bw, void *stream) {
    Args A;
    memset(&A, 0, sizeof(A));
    auto common = [&A](const auto *s) {      // the fields bmp_coattn_fwd_t and bmp_coattn_bwd_t share
        A.mb = s->mb; A.n1 = s->n1; A.n2 = s->n2; A.H = s->hidden; A.O = s->out_dim;
        A.head = s->variant == BMP_COATTN_FINE ? s->head : 1;
        A.variant = s->variant; A.act = s->act; A.atoms_1 = s->atoms_1; A.atoms_2 = s->atoms_2;
        A.W = s->W; A.V1 = s->V1; A.V2 = s->V2; A.b = s->b; A.lt_1 = s->lt_1; A.lt_2 = s->lt_2; A.wa_1 = s->wa_1; A.wa_2 = s->wa_2;
        A.W_j = s->W_j; A.b_j = s->b_j;
        A.ws = (float *)(((uintptr_t)s->tc_workspace + 255) & ~(uintptr_t)255);
    };
    if (bw) {
        common(bw);
        A.dc1 = bw->d_compact_1; A.dc2 = bw->d_compact_2; A.R = bw->R; A.P1 = bw->P1; A.P2 = bw->P2; A.DL1 = bw->DL1; A.DL2 = bw->DL2;
        A.d_a1 = bw->d_atoms_1; A.d_a2 = bw->d_atoms_2; A.d_V1 = bw->d_V1; A.d_V2 = bw->d_V2; A.d_b = bw->d_b;
        A.d_wa_1 = bw->d_wa_1; A.d_wa_2 = bw->d_wa_2;
    } else {
        common(f);
        A.c1 = f->compact_1; A.c2 = f->compact_2;
    }
    const size_t smem = smem_floats(A.H, A.head) * sizeof(float);
    const int grid = A.mb < CTAS ? A.mb : CTAS;
    const cudaStream_t st = (cudaStream_t)stream;
    Partials pt(st);
    if (bw) {
        if (co_det_begin(pt, A.det, A.H, grid)) return BMP_EINVAL;
        cudaFuncSetAttribute(coattn_big_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        coattn_big_bwd_kernel<<<grid, NTHREADS, smem, st>>>(A);
        count_launch();
        int rc = check_launch("coattn_big_bwd_kernel");
        if (rc) return rc;
        return co_det_end(pt, A.det, grid, A.variant == BMP_COATTN_FINE ? A.head : 0, nullptr, nullptr, nullptr, A.d_V1, A.d_V2,
                          A.d_wa_1, A.d_wa_2, A.d_b, false, "det_reduce_kernel (coattn_big)");
    } else {
        cudaFuncSetAttribute(coattn_big_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        coattn_big_fwd_kernel<<<grid, NTHREADS, smem, st>>>(A);
    }
    count_launch();
    return check_launch(bw ? "coattn_big_bwd_kernel" : "coattn_big_fwd_kernel");
}
