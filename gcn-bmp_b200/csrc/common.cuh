// common.cuh -- shared device helpers for the fp32 (BMP_MODE_F32) kernels.
//
// Data layout inside a CTA: one padded molecule (<= 64 atoms) is kept in shared
// memory CHANNEL-MAJOR, buf[c][i] with a fixed leading dimension of 64 atoms, so
// that every contraction of the hot path has the shape
//     out[o][i] (+)= sum_k X(o,k) * Y[k][i]
// with Y such a buffer, X a weight matrix streamed from L2 through a
// cp.async double-buffered staging tile (or another smem buffer), and the
// 64x64 output tile held in registers as 4x4 per thread (256 threads).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <initializer_list>
#include "../../include/gcnbmp.h"

namespace bmp {

constexpr int AT = 64;             // atoms tile = leading dimension of channel-major buffers
constexpr int NTHREADS = 256;
constexpr int KT = 32;             // k chunk of the staged X tile
constexpr int XLD = KT + 4;        // [64][36]  X tile, k contiguous
constexpr int XLDT = 64 + 4;       // [32][68]  X tile, o contiguous (transposed use)
constexpr int STAGE_FLOATS = 2 * 64 * XLD;   // two buffers (>= 2*32*68)

void set_error(const char *fmt, ...);
void count_launch(int n = 1);
int check_launch(const char *what);
// true when every non-null pointer is 16-byte aligned (cp.async / float4 paths)
bool aligned16(std::initializer_list<const void *> ps);
// Optional per-kernel timing (bmp_profile_enable): CUDA events recorded on the launching stream right before and after a
// hot kernel's launch, so a caller can time individual kernels INSIDE a real step.  No-op (one relaxed load) when off.
struct ProfScope {
    int kind;
    cudaStream_t st;
    void *slot;
    ProfScope(int kind, cudaStream_t st);
    ~ProfScope();
};
// two steps may share one packed weight image only when EVERY parameter pointer that goes into it is the same
inline bool same_gru(const bmp_gru_t &x, const bmp_gru_t &y) {
    return x.W_r == y.W_r && x.b_Wr == y.b_Wr && x.U_r == y.U_r && x.b_Ur == y.b_Ur && x.W_z == y.W_z && x.b_Wz == y.b_Wz &&
           x.U_z == y.U_z && x.b_Uz == y.b_Uz && x.W == y.W && x.b_W == y.b_W && x.U == y.U && x.b_U == y.b_U;
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// rescale_adj's column scale of one molecule (models/relgcn.py:20-28): inv[j] = 1 / sum_{e,i} adj[e][i][j], 1 where that sum is 0,
// for j < N <= BMP_X3_MAX_ATOMS.  256 threads; per 64-column chunk four partial sums per column (rows r = p mod 4).
__device__ __forceinline__ void column_inverse_degree(const float *__restrict__ adj, int E, int N, float (*part)[64], float *inv) {
    const int j = threadIdx.x & 63, p = threadIdx.x >> 6;
    for (int j0 = 0; j0 < N; j0 += 64) {
        float s = 0.f;
        if (j0 + j < N)
            for (int r = p; r < E * N; r += 4) s += __ldg(adj + (long)r * N + j0 + j);
        part[p][j] = s;
        __syncthreads();
        if (threadIdx.x < 64 && j0 + (int)threadIdx.x < N) {
            const float t = (part[0][threadIdx.x] + part[1][threadIdx.x]) + (part[2][threadIdx.x] + part[3][threadIdx.x]);
            inv[j0 + threadIdx.x] = t != 0.f ? 1.f / t : 1.f;
        }
        __syncthreads();
    }
}

__device__ __forceinline__ float act_fwd(int act, float x) {
    switch (act) {
        case BMP_ACT_TANH: return tanhf(x);
        case BMP_ACT_RELU: return x > 0.f ? x : 0.f;
        case BMP_ACT_SIGMOID: return sigmoidf_(x);
        default: return x;
    }
}
// derivative expressed through the activation OUTPUT y (and input x for relu)
__device__ __forceinline__ float act_bwd(int act, float x, float y) {
    switch (act) {
        case BMP_ACT_TANH: return 1.f - y * y;
        case BMP_ACT_RELU: return x > 0.f ? 1.f : 0.f;
        case BMP_ACT_SIGMOID: return y * (1.f - y);
        default: return 1.f;
    }
}

__device__ __forceinline__ void zero_acc(float (&acc)[4][4]) {
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
}

// ---- staged X tile loads ----------------------------------------------------
// TRANS = false: X(o,k) = Xg[(o_base+o)*ldx + k], tile [64 o][KT k]
// TRANS = true : X(o,k) = Xg[k*ldx + o_base + o], tile [KT k][64 o]
template <bool TRANS>
__device__ __forceinline__ void stage_tile(float *buf, const float *__restrict__ Xg, long ldx,
                                           int o_base, int o_lim, int k0, int K) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        int idx = tid + it * NTHREADS;
        if (!TRANS) {
            int row = idx >> 3, kq = (idx & 7) * 4;
            float *dst = buf + row * XLD + kq;
            if (o_base + row < o_lim && k0 + kq < K)
                cp_async16(dst, Xg + (long)(o_base + row) * ldx + k0 + kq);
            else
                *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            int krow = idx >> 4, oq = (idx & 15) * 4;
            float *dst = buf + krow * XLDT + oq;
            if (k0 + krow < K && o_base + oq < o_lim)
                cp_async16(dst, Xg + (long)(k0 + krow) * ldx + o_base + oq);
            else
                *reinterpret_cast<float4 *>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

// acc[a][b] += sum_k X(o0+a, k) * Ys[k*AT + i0+b],   o0 = 4*(tid/16), i0 = 4*(tid%16)
// X streamed from global memory.  Entry: Ys ready (caller synchronised), staging
// buffer free.  Exit: ends with __syncthreads().  K % 4 == 0.
template <bool TRANS>
__device__ __forceinline__ void gemm64_g(float (&acc)[4][4], const float *__restrict__ Xg, long ldx,
                                         int o_base, int o_lim, int K, const float *Ys, float *stage) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = ty * 4, i0 = tx * 4;
    const int nchunks = (K + KT - 1) / KT;
    constexpr int BUF = 64 * XLD;
    stage_tile<TRANS>(stage, Xg, ldx, o_base, o_lim, 0, K);
    cp_async_commit();
    for (int c = 0; c < nchunks; ++c) {
        float *cur = stage + (c & 1) * BUF;
        if (c + 1 < nchunks) {
            stage_tile<TRANS>(stage + ((c + 1) & 1) * BUF, Xg, ldx, o_base, o_lim, (c + 1) * KT, K);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const int k0 = c * KT;
        const int kmax = min(KT, K - k0);
        const float *Yk = Ys + (long)k0 * AT + i0;
        if (!TRANS) {
            for (int kk = 0; kk < kmax; kk += 4) {
                float4 x[4], y[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) x[a] = *reinterpret_cast<const float4 *>(cur + (o0 + a) * XLD + kk);
#pragma unroll
                for (int q = 0; q < 4; ++q) y[q] = *reinterpret_cast<const float4 *>(Yk + (kk + q) * AT);
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    acc[a][0] += x[a].x * y[0].x + x[a].y * y[1].x + x[a].z * y[2].x + x[a].w * y[3].x;
                    acc[a][1] += x[a].x * y[0].y + x[a].y * y[1].y + x[a].z * y[2].y + x[a].w * y[3].y;
                    acc[a][2] += x[a].x * y[0].z + x[a].y * y[1].z + x[a].z * y[2].z + x[a].w * y[3].z;
                    acc[a][3] += x[a].x * y[0].w + x[a].y * y[1].w + x[a].z * y[2].w + x[a].w * y[3].w;
                }
            }
        } else {
#pragma unroll 4
            for (int kk = 0; kk < kmax; ++kk) {
                float4 x = *reinterpret_cast<const float4 *>(cur + kk * XLDT + o0);
                float4 y = *reinterpret_cast<const float4 *>(Yk + kk * AT);
                acc[0][0] += x.x * y.x; acc[0][1] += x.x * y.y; acc[0][2] += x.x * y.z; acc[0][3] += x.x * y.w;
                acc[1][0] += x.y * y.x; acc[1][1] += x.y * y.y; acc[1][2] += x.y * y.z; acc[1][3] += x.y * y.w;
                acc[2][0] += x.z * y.x; acc[2][1] += x.z * y.y; acc[2][2] += x.z * y.z; acc[2][3] += x.z * y.w;
                acc[3][0] += x.w * y.x; acc[3][1] += x.w * y.y; acc[3][2] += x.w * y.z; acc[3][3] += x.w * y.w;
            }
        }
        __syncthreads();
    }
}

// Same contraction with X resident in shared memory, X(o,k) = Xs[(o_base+o)*ldx + k]
// (k contiguous).  No internal synchronisation.  K % 4 == 0.
__device__ __forceinline__ void gemm64_s(float (&acc)[4][4], const float *Xs, int ldx, int o_base, int K,
                                         const float *Ys) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = o_base + ty * 4, i0 = tx * 4;
    for (int kk = 0; kk < K; kk += 4) {
        float4 x[4], y[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) x[a] = *reinterpret_cast<const float4 *>(Xs + (o0 + a) * ldx + kk);
#pragma unroll
        for (int q = 0; q < 4; ++q) y[q] = *reinterpret_cast<const float4 *>(Ys + (kk + q) * AT + i0);
#pragma unroll
        for (int a = 0; a < 4; ++a) {
            acc[a][0] += x[a].x * y[0].x + x[a].y * y[1].x + x[a].z * y[2].x + x[a].w * y[3].x;
            acc[a][1] += x[a].x * y[0].y + x[a].y * y[1].y + x[a].z * y[2].y + x[a].w * y[3].y;
            acc[a][2] += x[a].x * y[0].z + x[a].y * y[1].z + x[a].z * y[2].z + x[a].w * y[3].z;
            acc[a][3] += x[a].x * y[0].w + x[a].y * y[1].w + x[a].z * y[2].w + x[a].w * y[3].w;
        }
    }
}

// ---- global <-> channel-major smem ------------------------------------------
// src is (n, C) row-major (atom-major) in global memory; dst[c*AT + i].
// Lane <-> atom, 8 channels (32 B) per access.  Columns i >= n are zero-filled.
// C % 8 == 0 is NOT required: C % 4 == 0 handled with float4 granularity.
__device__ __forceinline__ void load_cm(float *dst, const float *__restrict__ src, int n, int C) {
    const int nq = C >> 2;
    for (int idx = threadIdx.x; idx < nq * AT; idx += NTHREADS) {
        int i = idx & (AT - 1), cq = idx >> 6;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) v = *reinterpret_cast<const float4 *>(src + (long)i * C + cq * 4);
        float *d = dst + (cq * 4) * AT + i;
        d[0] = v.x; d[AT] = v.y; d[2 * AT] = v.z; d[3 * AT] = v.w;
    }
}
// embedding gather: dst[c][i] = W[ids[i]][c]
__device__ __forceinline__ void load_embed_cm(float *dst, const int32_t *__restrict__ ids,
                                              const float *__restrict__ W, int n, int C, int n_types) {
    const int nq = C >> 2;
    for (int idx = threadIdx.x; idx < nq * AT; idx += NTHREADS) {
        int i = idx & (AT - 1), cq = idx >> 6;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) {
            int id = ids[i];
            id = id < 0 ? 0 : (id >= n_types ? n_types - 1 : id);
            v = *reinterpret_cast<const float4 *>(W + (long)id * C + cq * 4);
        }
        float *d = dst + (cq * 4) * AT + i;
        d[0] = v.x; d[AT] = v.y; d[2 * AT] = v.z; d[3 * AT] = v.w;
    }
}
// store a channel-major smem buffer to (n, C) row-major global (+ column offset / ld)
__device__ __forceinline__ void store_cm(float *__restrict__ dst, long ld, const float *src, int n, int C) {
    const int nq = C >> 2;
    for (int idx = threadIdx.x; idx < nq * AT; idx += NTHREADS) {
        int i = idx & (AT - 1), cq = idx >> 6;
        if (i < n) {
            const float *s = src + (cq * 4) * AT + i;
            *reinterpret_cast<float4 *>(dst + (long)i * ld + cq * 4) = make_float4(s[0], s[AT], s[2 * AT], s[3 * AT]);
        }
    }
}
// thread-tile <-> global (atom-major): element (o0+a, i0+b) lives at g[(i0+b)*ld + o0+a]
__device__ __forceinline__ void tile_store_g(float *__restrict__ g, long ld, int o_base, int o_lim, int n,
                                             const float (&v)[4][4]) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = o_base + ty * 4, i0 = tx * 4;
    if (o0 >= o_lim) return;
#pragma unroll
    for (int b = 0; b < 4; ++b)
        if (i0 + b < n)
            *reinterpret_cast<float4 *>(g + (long)(i0 + b) * ld + o0) = make_float4(v[0][b], v[1][b], v[2][b], v[3][b]);
}
__device__ __forceinline__ void tile_load_g(const float *__restrict__ g, long ld, int o_base, int o_lim, int n,
                                            float (&v)[4][4]) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = o_base + ty * 4, i0 = tx * 4;
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (o0 < o_lim && i0 + b < n) t = *reinterpret_cast<const float4 *>(g + (long)(i0 + b) * ld + o0);
        v[0][b] = t.x; v[1][b] = t.y; v[2][b] = t.z; v[3][b] = t.w;
    }
}
// thread-tile <-> channel-major smem
__device__ __forceinline__ void tile_store_s(float *s, int o_base, const float (&v)[4][4]) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = o_base + ty * 4, i0 = tx * 4;
#pragma unroll
    for (int a = 0; a < 4; ++a)
        *reinterpret_cast<float4 *>(s + (o0 + a) * AT + i0) = make_float4(v[a][0], v[a][1], v[a][2], v[a][3]);
}
__device__ __forceinline__ void tile_load_s(const float *s, int o_base, float (&v)[4][4]) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int o0 = o_base + ty * 4, i0 = tx * 4;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        float4 t = *reinterpret_cast<const float4 *>(s + (o0 + a) * AT + i0);
        v[a][0] = t.x; v[a][1] = t.y; v[a][2] = t.z; v[a][3] = t.w;
    }
}

// adjacency of one edge type (n x n, row-major in global) into smem.
//   TRANSPOSE = true : dst[j*AT + i] = adj[i][j]  (Y operand of  out[c][i] = sum_j h[c][j] A[i][j])
//   TRANSPOSE = false: dst[i*AT + j] = adj[i][j]  (Y operand of  P[c][j] = sum_i dm[c][i] A[i][j])
// Rows/cols >= n are zero.  deg (optional, TRANSPOSE only) = row sums deg[i] = sum_j adj[i][j].
// colscale (optional): adj[i][j] *= colscale[j]   (rescale_adj, models/relgcn.py:20-28)
template <bool TRANSPOSE>
__device__ __forceinline__ void load_adj(float *dst, const float *__restrict__ adj, int n,
                                         const float *colscale = nullptr) {
    if (TRANSPOSE) {
        // lane <-> row i, 4 consecutive j per access (n % 4 may be != 0: scalar tail)
        for (int idx = threadIdx.x; idx < 16 * AT; idx += NTHREADS) {
            int i = idx & (AT - 1), jq = (idx >> 6) * 4;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (i < n) {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (jq + q < n) {
                        v[q] = adj[(long)i * n + jq + q];
                        if (colscale) v[q] *= colscale[jq + q];
                    }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) dst[(jq + q) * AT + i] = v[q];
        }
    } else {
        for (int idx = threadIdx.x; idx < AT * AT; idx += NTHREADS) {
            int i = idx >> 6, j = idx & (AT - 1);
            float v = 0.f;
            if (i < n && j < n) {
                v = adj[(long)i * n + j];
                if (colscale) v *= colscale[j];
            }
            dst[i * AT + j] = v;
        }
    }
}

}  // namespace bmp
