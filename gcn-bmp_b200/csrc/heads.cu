// heads.cu -- the remaining link-prediction heads of the reference (SURVEY 8 f-4) and the optimizer hooks (f-2), fp32.
//   pair features   SymMLP input [l + r | l * r] (models/mlp.py:104-105), DistMult product l * r (BilinearDiag, mlp.py:154-197:
//                   a diagonal bilinear form is Linear(l * r)), MLP input [l | r] (train_binary.py:98-100)
//   bilinear        chainer.links.Bilinear(left, right, out) of the NTN head (mlp.py:47-74):
//                   y[b,k] = sum_ij e1[b,i] W[i,j,k] e2[b,j] + e1 V1 + e2 V2 + b, contracted as u = e1 W_flat (GEMM) and a
//                   rank-R reduction -- Chainer's (B, L, R) outer product is never materialised
//   gradient hooks  GradientClipping -> WeightDecay -> Lasso in the order train_binary.py:537-543 adds them
// HBM-bound elementwise / reduction work: grid-stride loops, float4 where the shapes allow.
#include "common.cuh"

namespace bmp {

// ---------------------------------------------------------------- pair features
__global__ void pairfeat_fwd_kernel(const float *__restrict__ l, const float *__restrict__ r, float *__restrict__ out,
                                    long n, int D, int kind) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const long b = i / D;
        const int c = (int)(i - b * D);
        const float x = l[i], y = r[i];
        if (kind == BMP_PAIR_SYM) { out[b * 2 * D + c] = x + y; out[b * 2 * D + D + c] = x * y; }
        else if (kind == BMP_PAIR_PROD) out[i] = x * y;
        else { out[b * 2 * D + c] = x; out[b * 2 * D + D + c] = y; }
    }
}
__global__ void pairfeat_bwd_kernel(const float *__restrict__ l, const float *__restrict__ r, const float *__restrict__ dout,
                                    float *__restrict__ dl, float *__restrict__ dr, long n, int D, int kind) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const long b = i / D;
        const int c = (int)(i - b * D);
        if (kind == BMP_PAIR_SYM) {
            const float ds = dout[b * 2 * D + c], dp = dout[b * 2 * D + D + c];
            dl[i] = ds + dp * r[i];
            dr[i] = ds + dp * l[i];
        } else if (kind == BMP_PAIR_PROD) {
            const float dp = dout[i];
            dl[i] = dp * r[i];
            dr[i] = dp * l[i];
        } else {
            dl[i] = dout[b * 2 * D + c];
            dr[i] = dout[b * 2 * D + D + c];
        }
    }
}

// ---------------------------------------------------------------- bilinear (NTN)
// y[b,k] = sum_j u[b,j,k] e2[b,j] + sum_i e1[b,i] V1[i,k] + sum_j e2[b,j] V2[j,k] + bias[k]; one thread per (b,k)
__global__ void bilinear_reduce_kernel(const float *__restrict__ u, const float *__restrict__ e1, const float *__restrict__ e2,
                                       const float *__restrict__ V1, const float *__restrict__ V2, const float *__restrict__ bias,
                                       float *__restrict__ y, long rows, int L, int R, int K) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < rows * K; t += (long)gridDim.x * blockDim.x) {
        const long b = t / K;
        const int k = (int)(t - b * K);
        const float *ub = u + b * (long)R * K, *x1 = e1 + b * L, *x2 = e2 + b * R;
        float s = bias ? bias[k] : 0.f;
        for (int j = 0; j < R; ++j) s = fmaf(ub[(long)j * K + k] + (V2 ? V2[(long)j * K + k] : 0.f), x2[j], s);
        if (V1)
            for (int i = 0; i < L; ++i) s = fmaf(x1[i], V1[(long)i * K + k], s);
        y[t] = s;
    }
}
// du[b,j,k] = dy[b,k] e2[b,j];  de2[b,j] = sum_k (u[b,j,k] + V2[j,k]) dy[b,k]; one thread per (b,j)
__global__ void bilinear_bwd_right_kernel(const float *__restrict__ u, const float *__restrict__ e2, const float *__restrict__ V2,
                                          const float *__restrict__ dy, float *__restrict__ du, float *__restrict__ de2,
                                          long rows, int R, int K) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < rows * R; t += (long)gridDim.x * blockDim.x) {
        const long b = t / R;
        const int j = (int)(t - b * R);
        const float x = e2[t];
        const float *g = dy + b * K, *uj = u + t * K;
        float s = 0.f;
        for (int k = 0; k < K; ++k) {
            du[t * K + k] = g[k] * x;
            s = fmaf(uj[k] + (V2 ? V2[(long)j * K + k] : 0.f), g[k], s);
        }
        de2[t] = s;
    }
}
// de1[b,i] += sum_k V1[i,k] dy[b,k]
__global__ void bilinear_bwd_left_kernel(const float *__restrict__ V1, const float *__restrict__ dy, float *__restrict__ de1,
                                         long rows, int L, int K) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < rows * L; t += (long)gridDim.x * blockDim.x) {
        const long b = t / L;
        const int i = (int)(t - b * L);
        float s = 0.f;
        for (int k = 0; k < K; ++k) s = fmaf(V1[(long)i * K + k], dy[b * K + k], s);
        de1[t] += s;
    }
}

// ---------------------------------------------------------------- atom-wise primitives of the vector-query co-attentions
// (alternating_coattention.py, parallel_coattention.py): a (mb, O) query vector against the (mb, N, C) atom arrays.
// y[b,n,c] = act(x[b,n,c] + v[b,c]); x == NULL: tile of v (F.tile over the atoms); v == NULL: plain activation
__global__ void bcast_add_act_fwd_kernel(const float *__restrict__ x, const float *__restrict__ v, float *__restrict__ y,
                                         long total, int n_atoms, int ch, int act) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const long b = i / ((long)n_atoms * ch);
        const int c = (int)(i % ch);
        y[i] = act_fwd(act, (x ? x[i] : 0.f) + (v ? v[b * ch + c] : 0.f));
    }
}
// dx = dy * act'(y) (optional); dv[b,c] = sum_n of the same (optional); one thread per (b,c)
__global__ void bcast_add_act_bwd_kernel(const float *__restrict__ y, const float *__restrict__ dy, float *__restrict__ dx,
                                         float *__restrict__ dv, long mbch, int n_atoms, int ch, int act) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < mbch; t += (long)gridDim.x * blockDim.x) {
        const long b = t / ch;
        const int c = (int)(t - b * ch);
        float s = 0.f;
        for (int n = 0; n < n_atoms; ++n) {
            const long i = (b * n_atoms + n) * ch + c;
            const float yy = y[i];
            const float g = dy[i] * act_bwd(act, yy, yy);
            if (dx) dx[i] = g;
            s += g;
        }
        if (dv) dv[t] = s;
    }
}
// softmax over the atoms axis (F.softmax default axis=1 on (mb, N, C)); one thread per (b,c)
__global__ void atoms_softmax_fwd_kernel(const float *__restrict__ x, float *__restrict__ y, long mbch, int n_atoms, int ch) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < mbch; t += (long)gridDim.x * blockDim.x) {
        const long b = t / ch;
        const int c = (int)(t - b * ch);
        const float *xb = x + b * n_atoms * ch + c;
        float m = -INFINITY, s = 0.f;
        for (int n = 0; n < n_atoms; ++n) m = fmaxf(m, xb[(long)n * ch]);
        for (int n = 0; n < n_atoms; ++n) s += expf(xb[(long)n * ch] - m);
        const float inv = 1.f / s;
        float *yb = y + b * n_atoms * ch + c;
        for (int n = 0; n < n_atoms; ++n) yb[(long)n * ch] = expf(xb[(long)n * ch] - m) * inv;
    }
}
__global__ void atoms_softmax_bwd_kernel(const float *__restrict__ y, const float *__restrict__ dy, float *__restrict__ dx,
                                         long mbch, int n_atoms, int ch) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < mbch; t += (long)gridDim.x * blockDim.x) {
        const long b = t / ch;
        const int c = (int)(t - b * ch);
        const long base = b * n_atoms * ch + c;
        float s = 0.f;
        for (int n = 0; n < n_atoms; ++n) s = fmaf(y[base + (long)n * ch], dy[base + (long)n * ch], s);
        for (int n = 0; n < n_atoms; ++n) dx[base + (long)n * ch] = y[base + (long)n * ch] * (dy[base + (long)n * ch] - s);
    }
}
// out[b,c] = sum_n a[b,n,(a_ch == 1 ? 0 : c)] * z[b,n,c]   (F.sum(F.tile(attn) * z, axis=1)); one thread per (b,c)
__global__ void atoms_pool_fwd_kernel(const float *__restrict__ a, int a_ch, const float *__restrict__ z, float *__restrict__ out,
                                      long mbch, int n_atoms, int ch) {
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < mbch; t += (long)gridDim.x * blockDim.x) {
        const long b = t / ch;
        const int c = (int)(t - b * ch);
        float s = 0.f;
        for (int n = 0; n < n_atoms; ++n) {
            const long r = b * n_atoms + n;
            s = fmaf(a[r * a_ch + (a_ch == 1 ? 0 : c)], z[r * ch + c], s);
        }
        out[t] = s;
    }
}
// dz = a * dout;  da = dout * z (a_ch == ch) or sum_c dout z (a_ch == 1); one warp per (b,n)
__global__ void atoms_pool_bwd_kernel(const float *__restrict__ a, int a_ch, const float *__restrict__ z, const float *__restrict__ dout,
                                      float *__restrict__ da, float *__restrict__ dz, long rows, int n_atoms, int ch) {
    const int lane = threadIdx.x & 31;
    for (long r = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += ((long)gridDim.x * blockDim.x) >> 5) {
        const long b = r / n_atoms;
        float s = 0.f;
        for (int c = lane; c < ch; c += 32) {
            const float g = dout[b * ch + c], zz = z[r * ch + c];
            dz[r * ch + c] = a[r * a_ch + (a_ch == 1 ? 0 : c)] * g;
            if (a_ch == 1) s = fmaf(g, zz, s);
            else da[r * ch + c] = g * zz;
        }
        if (a_ch == 1) {
#pragma unroll
            for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) da[r] = s;
        }
    }
}

// ---------------------------------------------------------------- GIN aggregation (models/gin.py:88-94)
// out[b,i,:] = h[b,i,:] + sum_e sum_j A[b,e,i,j] h[b,j,:]   (TRANS: A[b,e,j,i] -- the backward with respect to h).
// One CTA per molecule: h is staged in shared memory, the bond types are summed into a tile of RB output rows x N (all N rows
// when they fit, up to 64 atoms), then every thread owns channels c, c + blockDim.x, ... of the tile's atoms.
template <bool TRANS>
__global__ void __launch_bounds__(256) gin_aggregate_kernel(const float *__restrict__ adj, const float *__restrict__ h,
                                                            float *__restrict__ out, int mb, int E, int N, int H, int RB) {
    extern __shared__ float sm[];
    float *As = sm;                  // [RB][N+1]
    float *hs = sm + RB * (N + 1);   // [N][H]
    for (int b = blockIdx.x; b < mb; b += gridDim.x) {
        for (int idx = threadIdx.x; idx < N * H; idx += blockDim.x) hs[idx] = h[(long)b * N * H + idx];
        for (int i0 = 0; i0 < N; i0 += RB) {
            const int rb = N - i0 < RB ? N - i0 : RB;
            for (int idx = threadIdx.x; idx < rb * N; idx += blockDim.x) {
                // consecutive threads read consecutive addresses of the adjacency
                const int i = TRANS ? idx % rb : idx / N, j = TRANS ? idx / rb : idx % N;
                float s = 0.f;
                for (int e = 0; e < E; ++e) s += adj[(((long)b * E + e) * N + (TRANS ? j : i0 + i)) * N + (TRANS ? i0 + i : j)];
                As[i * (N + 1) + j] = s;
            }
            __syncthreads();
            for (int idx = threadIdx.x; idx < rb * H; idx += blockDim.x) {
                const int i = idx / H, c = idx - i * H;
                float s = hs[(i0 + i) * H + c];
                for (int j = 0; j < N; ++j) s = fmaf(As[i * (N + 1) + j], hs[j * H + c], s);
                out[(long)b * N * H + (long)(i0 + i) * H + c] = s;
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------- NFP update (models/models/nfp.py:35-59) + EmbedID forward
// X[b,i,(d-1)*C + c] = fv[b,i,c] when the degree of atom i equals d (1..D), zero otherwise, with fv = adj[b] . h[b] and
// degree[b,i] = sum_{i'} adj[b,i',i] (nfp.py:152: xp.sum(adj, axis=1)).  The D degree-specific GraphLinears of the reference,
// each applied to where(deg == d, fv, 0), are then ONE Linear over X with the weights concatenated along the input axis (and
// all D biases added to every atom, as the reference's zero-masked inputs still pick up every bias).
// One CTA per molecule; h (N x C) staged in shared memory, adj (forward) or adj^T (backward) in tiles of RB output rows x N (all N
// rows when they fit, up to 64 atoms).  BWD: dfv = the degree block of dX, dh = adj^T dfv.
template <bool BWD>
__global__ void __launch_bounds__(256) nfp_gather_kernel(const float *__restrict__ adj, const float *__restrict__ src,
                                                         float *__restrict__ dst, int mb, int N, int C, int D, int RB) {
    extern __shared__ float sm[];
    float *As = sm;                       // [RB][N+1]  rows i0.. of adj (forward) or of adj^T (backward)
    float *hs = As + RB * (N + 1);        // [N][C]   forward: h ; backward: dfv
    int *deg = reinterpret_cast<int *>(hs + N * C);   // [N] degree block index (0..D-1) or -1
    for (int b = blockIdx.x; b < mb; b += gridDim.x) {
        const float *Ab = adj + (long)b * N * N;
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            float s = 0.f;
            for (int r = 0; r < N; ++r) s += Ab[(long)r * N + i];
            int d = -1;
            for (int k = 1; k <= D; ++k)
                if (s - (float)k == 0.f) d = k - 1;
            deg[i] = d;
        }
        __syncthreads();
        if (!BWD) {
            for (int idx = threadIdx.x; idx < N * C; idx += blockDim.x) hs[idx] = src[(long)b * N * C + idx];
        } else {
            const float *dX = src + (long)b * N * D * C;
            for (int idx = threadIdx.x; idx < N * C; idx += blockDim.x) {
                const int i = idx / C, c = idx - i * C;
                hs[idx] = deg[i] >= 0 ? dX[(long)i * D * C + deg[i] * C + c] : 0.f;
            }
        }
        for (int i0 = 0; i0 < N; i0 += RB) {
            const int rb = N - i0 < RB ? N - i0 : RB;
            for (int idx = threadIdx.x; idx < rb * N; idx += blockDim.x) {
                const int i = BWD ? idx % rb : idx / N, j = BWD ? idx / rb : idx % N;
                As[i * (N + 1) + j] = BWD ? Ab[(long)j * N + i0 + i] : Ab[(long)(i0 + i) * N + j];
            }
            __syncthreads();
            if (!BWD) {
                float *X = dst + (long)b * N * D * C + (long)i0 * D * C;
                for (int idx = threadIdx.x; idx < rb * D * C; idx += blockDim.x) {
                    const int i = idx / (D * C), r = idx - i * D * C, d = r / C, c = r - d * C;
                    float v = 0.f;
                    if (d == deg[i0 + i])
                        for (int j = 0; j < N; ++j) v = fmaf(As[i * (N + 1) + j], hs[j * C + c], v);
                    X[idx] = v;
                }
            } else {
                for (int idx = threadIdx.x; idx < rb * C; idx += blockDim.x) {
                    const int jj = idx / C, c = idx - jj * C;
                    float v = 0.f;
                    for (int i = 0; i < N; ++i) v = fmaf(As[jj * (N + 1) + i], hs[i * C + c], v);
                    dst[(long)b * N * C + (long)(i0 + jj) * C + c] = v;
                }
            }
            __syncthreads();
        }
    }
}

// rows of the adjacency tile that fit next to the `fixed` floats: all N when they fit, else as many as fit (0: none)
static int adjacency_tile_rows(int N, size_t fixed) {
    const size_t cap = 227 * 1024 / sizeof(float);
    if (fixed + (size_t)N * (N + 1) <= cap) return N;
    return fixed >= cap ? 0 : (int)((cap - fixed) / (N + 1) < (size_t)N ? (cap - fixed) / (N + 1) : N);
}

__global__ void embed_fwd_kernel(const int32_t *__restrict__ ids, const float *__restrict__ W, float *__restrict__ out, long rows,
                                 int H, int n_types) {
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < rows * H; idx += (long)gridDim.x * blockDim.x) {
        const long r = idx / H;
        int id = ids[r];
        id = id < 0 ? 0 : (id >= n_types ? n_types - 1 : id);
        out[idx] = W[(long)id * H + (idx - r * H)];
    }
}

// ---------------------------------------------------------------- optimizer hooks
__global__ void sumsq_kernel(const float *__restrict__ g, long n, float *__restrict__ out) {
    float s = 0.f;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) s = fmaf(g[i], g[i], s);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ float red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        float tot = 0.f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
        atomicAdd(out, tot);
    }
}
__global__ void hooks_kernel(float *__restrict__ g, const float *__restrict__ p, long n, float clip, float l2, float l1,
                             const float *__restrict__ sumsq) {
    float scale = 1.f;
    if (clip > 0.f) {
        const float rate = clip / sqrtf(*sumsq);       // chainer.optimizer.GradientClipping: rate = threshold / norm
        if (rate < 1.f) scale = rate;
    }
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const float w = p[i];
        float v = g[i] * scale;
        v = fmaf(l2, w, v);                                                // WeightDecay: g += rate * p
        v = fmaf(l1, w > 0.f ? 1.f : (w < 0.f ? -1.f : 0.f), v);           // Lasso: g += rate * sign(p)
        g[i] = v;
    }
}

static int grid_for(long n) {
    long g = (n + 255) / 256;
    return (int)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}

}  // namespace bmp

using namespace bmp;

extern "C" int bmp_pair_features_forward(const float *left, const float *right, float *out, int rows, int dim, int kind, void *stream) {
    if (!left || !right || !out) { set_error("bmp_pair_features_forward: null pointer"); return BMP_EINVAL; }
    if (kind < BMP_PAIR_SYM || kind > BMP_PAIR_CONCAT) { set_error("bmp_pair_features_forward: bad kind %d", kind); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    if (dim <= 0) { set_error("bmp_pair_features_forward: bad dim %d", dim); return BMP_ESHAPE; }
    const long n = (long)rows * dim;
    pairfeat_fwd_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(left, right, out, n, dim, kind);
    count_launch();
    return check_launch("pairfeat_fwd_kernel");
}

extern "C" int bmp_pair_features_backward(const float *left, const float *right, const float *d_out, float *d_left, float *d_right,
                                          int rows, int dim, int kind, void *stream) {
    if (!left || !right || !d_out || !d_left || !d_right) { set_error("bmp_pair_features_backward: null pointer"); return BMP_EINVAL; }
    if (kind < BMP_PAIR_SYM || kind > BMP_PAIR_CONCAT) { set_error("bmp_pair_features_backward: bad kind %d", kind); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    const long n = (long)rows * dim;
    pairfeat_bwd_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(left, right, d_out, d_left, d_right, n, dim, kind);
    count_launch();
    return check_launch("pairfeat_bwd_kernel");
}

extern "C" int bmp_bilinear_forward(const float *e1, const float *e2, const float *W, const float *V1, const float *V2, const float *b,
                                    float *u, float *y, int rows, int left, int right, int out, void *stream) {
    if (!e1 || !e2 || !W || !u || !y) { set_error("bmp_bilinear_forward: null pointer"); return BMP_EINVAL; }
    if ((V1 != nullptr) != (V2 != nullptr)) { set_error("bmp_bilinear_forward: V1 and V2 come together"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    if (left <= 0 || right <= 0 || out <= 0) { set_error("bmp_bilinear_forward: bad dims"); return BMP_ESHAPE; }
    // u (rows, right*out) = e1 (rows, left) x W viewed as (left, right*out): the data-gradient form of the Linear kernel
    int rc = bmp_linear_backward(e1, W, nullptr, const_cast<float *>(e1), u, nullptr, nullptr, rows, right * out, left, BMP_ACT_IDENTITY, stream);
    if (rc) return rc;
    bilinear_reduce_kernel<<<grid_for((long)rows * out), 256, 0, (cudaStream_t)stream>>>(u, e1, e2, V1, V2, b, y, rows, left, right, out);
    count_launch();
    return check_launch("bilinear_reduce_kernel");
}

extern "C" int bmp_bilinear_backward(const float *e1, const float *e2, const float *W, const float *V1, const float *V2, const float *u,
                                     const float *dy, float *du, float *de1, float *de2, float *dW, float *dV1, float *dV2, float *db,
                                     int rows, int left, int right, int out, void *stream) {
    if (!e1 || !e2 || !W || !u || !dy || !du || !de1 || !de2) { set_error("bmp_bilinear_backward: null pointer"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    bilinear_bwd_right_kernel<<<grid_for((long)rows * right), 256, 0, st>>>(u, e2, V2, dy, du, de2, rows, right, out);
    count_launch();
    if ((rc = check_launch("bilinear_bwd_right_kernel"))) return rc;
    // de1 = du W_flat^T: the forward form of the Linear kernel with W_flat as a (left, right*out) weight
    if ((rc = bmp_linear_forward(du, W, nullptr, de1, rows, right * out, left, BMP_ACT_IDENTITY, stream))) return rc;
    if (V1) {
        bilinear_bwd_left_kernel<<<grid_for((long)rows * left), 256, 0, st>>>(V1, dy, de1, rows, left, out);
        count_launch();
        if ((rc = check_launch("bilinear_bwd_left_kernel"))) return rc;
    }
    if (dW && (rc = bmp_wgrad(e1, left, du, right * out, dW, right * out, rows, left, right * out, stream))) return rc;
    if (dV1 && (rc = bmp_wgrad(e1, left, dy, out, dV1, out, rows, left, out, stream))) return rc;
    if (dV2 && (rc = bmp_wgrad(e2, right, dy, out, dV2, out, rows, right, out, stream))) return rc;
    if (db && (rc = bmp_colsum(dy, out, db, 1, rows, out, stream))) return rc;
    return BMP_OK;
}

extern "C" int bmp_atoms_bcast_add_act_forward(const float *x, const float *v, float *y, int mb, int n_atoms, int ch, int act, void *stream) {
    if (!y || (!x && !v)) { set_error("bmp_atoms_bcast_add_act_forward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (n_atoms <= 0 || ch <= 0) { set_error("bmp_atoms_bcast_add_act_forward: bad shape"); return BMP_ESHAPE; }
    const long total = (long)mb * n_atoms * ch;
    bcast_add_act_fwd_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(x, v, y, total, n_atoms, ch, act);
    count_launch();
    return check_launch("bcast_add_act_fwd_kernel");
}

extern "C" int bmp_atoms_bcast_add_act_backward(const float *y, const float *dy, float *dx, float *dv, int mb, int n_atoms, int ch, int act, void *stream) {
    if (!y || !dy || (!dx && !dv)) { set_error("bmp_atoms_bcast_add_act_backward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    const long mbch = (long)mb * ch;
    bcast_add_act_bwd_kernel<<<grid_for(mbch), 256, 0, (cudaStream_t)stream>>>(y, dy, dx, dv, mbch, n_atoms, ch, act);
    count_launch();
    return check_launch("bcast_add_act_bwd_kernel");
}

extern "C" int bmp_atoms_softmax_forward(const float *x, float *y, int mb, int n_atoms, int ch, void *stream) {
    if (!x || !y) { set_error("bmp_atoms_softmax_forward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (n_atoms <= 0 || ch <= 0) { set_error("bmp_atoms_softmax_forward: bad shape"); return BMP_ESHAPE; }
    const long mbch = (long)mb * ch;
    atoms_softmax_fwd_kernel<<<grid_for(mbch), 256, 0, (cudaStream_t)stream>>>(x, y, mbch, n_atoms, ch);
    count_launch();
    return check_launch("atoms_softmax_fwd_kernel");
}

extern "C" int bmp_atoms_softmax_backward(const float *y, const float *dy, float *dx, int mb, int n_atoms, int ch, void *stream) {
    if (!y || !dy || !dx) { set_error("bmp_atoms_softmax_backward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    const long mbch = (long)mb * ch;
    atoms_softmax_bwd_kernel<<<grid_for(mbch), 256, 0, (cudaStream_t)stream>>>(y, dy, dx, mbch, n_atoms, ch);
    count_launch();
    return check_launch("atoms_softmax_bwd_kernel");
}

extern "C" int bmp_atoms_pool_forward(const float *a, int a_ch, const float *z, float *out, int mb, int n_atoms, int ch, void *stream) {
    if (!a || !z || !out) { set_error("bmp_atoms_pool_forward: null pointer"); return BMP_EINVAL; }
    if (a_ch != 1 && a_ch != ch) { set_error("bmp_atoms_pool_forward: attention width %d must be 1 or %d", a_ch, ch); return BMP_ESHAPE; }
    if (mb <= 0) return BMP_OK;
    const long mbch = (long)mb * ch;
    atoms_pool_fwd_kernel<<<grid_for(mbch), 256, 0, (cudaStream_t)stream>>>(a, a_ch, z, out, mbch, n_atoms, ch);
    count_launch();
    return check_launch("atoms_pool_fwd_kernel");
}

extern "C" int bmp_atoms_pool_backward(const float *a, int a_ch, const float *z, const float *d_out, float *da, float *dz,
                                       int mb, int n_atoms, int ch, void *stream) {
    if (!a || !z || !d_out || !da || !dz) { set_error("bmp_atoms_pool_backward: null pointer"); return BMP_EINVAL; }
    if (a_ch != 1 && a_ch != ch) { set_error("bmp_atoms_pool_backward: attention width %d must be 1 or %d", a_ch, ch); return BMP_ESHAPE; }
    if (mb <= 0) return BMP_OK;
    const long rows = (long)mb * n_atoms;
    atoms_pool_bwd_kernel<<<grid_for(rows * 32), 256, 0, (cudaStream_t)stream>>>(a, a_ch, z, d_out, da, dz, rows, n_atoms, ch);
    count_launch();
    return check_launch("atoms_pool_bwd_kernel");
}

extern "C" int bmp_gin_aggregate(const float *adj, const float *h, float *out, int mb, int n_edge, int n_atoms, int hidden,
                                 int transpose, void *stream) {
    if (!adj || !h || !out) { set_error("bmp_gin_aggregate: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (n_atoms <= 0 || n_atoms > BMP_X3_MAX_ATOMS || hidden <= 0 || n_edge <= 0) { set_error("bmp_gin_aggregate: bad shape n_atoms=%d H=%d E=%d", n_atoms, hidden, n_edge); return BMP_ESHAPE; }
    const int RB = adjacency_tile_rows(n_atoms, (size_t)n_atoms * hidden);
    if (RB < 8) { set_error("bmp_gin_aggregate: n_atoms=%d, hidden=%d do not fit in shared memory", n_atoms, hidden); return BMP_ESHAPE; }
    const size_t smem = sizeof(float) * ((size_t)RB * (n_atoms + 1) + (size_t)n_atoms * hidden);
    const int grid = mb < 148 * 4 ? mb : 148 * 4;
    cudaStream_t st = (cudaStream_t)stream;
    if (transpose) {
        cudaFuncSetAttribute(gin_aggregate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gin_aggregate_kernel<true><<<grid, 256, smem, st>>>(adj, h, out, mb, n_edge, n_atoms, hidden, RB);
    } else {
        cudaFuncSetAttribute(gin_aggregate_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gin_aggregate_kernel<false><<<grid, 256, smem, st>>>(adj, h, out, mb, n_edge, n_atoms, hidden, RB);
    }
    count_launch();
    return check_launch("gin_aggregate_kernel");
}

extern "C" int bmp_nfp_gather(const float *adj, const float *src, float *dst, int mb, int n_atoms, int ch, int n_degree,
                              int backward, void *stream) {
    if (!adj || !src || !dst) { set_error("bmp_nfp_gather: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (n_atoms <= 0 || n_atoms > BMP_X3_MAX_ATOMS || ch <= 0 || n_degree <= 0) { set_error("bmp_nfp_gather: bad shape n_atoms=%d C=%d D=%d", n_atoms, ch, n_degree); return BMP_ESHAPE; }
    const int RB = adjacency_tile_rows(n_atoms, (size_t)n_atoms * ch + n_atoms);
    if (RB < 8) { set_error("bmp_nfp_gather: n_atoms=%d, channels=%d do not fit in shared memory", n_atoms, ch); return BMP_ESHAPE; }
    const size_t smem = sizeof(float) * ((size_t)RB * (n_atoms + 1) + (size_t)n_atoms * ch + n_atoms);
    const int grid = mb < 148 * 4 ? mb : 148 * 4;
    cudaStream_t st = (cudaStream_t)stream;
    if (backward) {
        cudaFuncSetAttribute(nfp_gather_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        nfp_gather_kernel<true><<<grid, 256, smem, st>>>(adj, src, dst, mb, n_atoms, ch, n_degree, RB);
    } else {
        cudaFuncSetAttribute(nfp_gather_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        nfp_gather_kernel<false><<<grid, 256, smem, st>>>(adj, src, dst, mb, n_atoms, ch, n_degree, RB);
    }
    count_launch();
    return check_launch("nfp_gather_kernel");
}

extern "C" int bmp_embed_forward(const int32_t *atoms, const float *embed_W, float *out, int rows, int hidden, int n_atom_types,
                                 void *stream) {
    if (!atoms || !embed_W || !out) { set_error("bmp_embed_forward: null pointer"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    if (hidden <= 0 || n_atom_types <= 0) { set_error("bmp_embed_forward: bad shape"); return BMP_ESHAPE; }
    embed_fwd_kernel<<<grid_for((long)rows * hidden), 256, 0, (cudaStream_t)stream>>>(atoms, embed_W, out, rows, hidden, n_atom_types);
    count_launch();
    return check_launch("embed_fwd_kernel");
}

extern "C" int bmp_grad_hooks(float *grad, const float *param, int n, float clip_threshold, float l2_rate, float l1_rate,
                              float *norm_ws, void *stream) {
    if (!grad || !param) { set_error("bmp_grad_hooks: null pointer"); return BMP_EINVAL; }
    if (n <= 0 || (clip_threshold <= 0.f && l2_rate == 0.f && l1_rate == 0.f)) return BMP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (clip_threshold > 0.f) {
        if (!norm_ws) { set_error("bmp_grad_hooks: GradientClipping needs one float of device scratch (norm_ws)"); return BMP_EINVAL; }
        if (cudaMemsetAsync(norm_ws, 0, sizeof(float), st) != cudaSuccess) { set_error("bmp_grad_hooks: memset failed"); return BMP_ECUDA; }
        sumsq_kernel<<<grid_for(n), 256, 0, st>>>(grad, n, norm_ws);
        count_launch();
        if ((rc = check_launch("sumsq_kernel"))) return rc;
    }
    hooks_kernel<<<grid_for(n), 256, 0, st>>>(grad, param, n, clip_threshold, l2_rate, l1_rate, norm_ws);
    count_launch();
    return check_launch("hooks_kernel");
}
