// gemm.cu -- the dense pieces that are not per-molecule: parameter-gradient
// contractions over all atoms of a batch (C += A^T B), column sums for bias
// gradients, and the links.Linear layers of the heads (hole.py:21-26).
#include "det.cuh"

namespace bmp {

constexpr int RT = 32;           // rows per staged chunk
constexpr int WLD = 64 + 4;

// ---- C (M,N; ldc) += A^T B, A (rows,M; lda), B (rows,N; ldb) -----------------
// grid.x = tilesM*tilesN, grid.y = split over rows.  64x64 C tile per CTA, 4x4 per thread.
__global__ void __launch_bounds__(NTHREADS) wgrad_kernel(const float *__restrict__ A, int lda,
                                                         const float *__restrict__ B, int ldb,
                                                         float *__restrict__ C, int ldc,
                                                         long rows, int M, int N, int tilesN, long rows_per_cta,
                                                         int vec, float *__restrict__ part) {
    __shared__ __align__(16) float As[2][RT][WLD];
    __shared__ __align__(16) float Bs[2][RT][WLD];
    const int tid = threadIdx.x;
    const int tm = (blockIdx.x / tilesN) * 64, tn = (blockIdx.x % tilesN) * 64;
    const long r_begin = (long)blockIdx.y * rows_per_cta;
    const long r_end = min(rows, r_begin + rows_per_cta);
    if (r_begin >= r_end) return;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = ty * 4, n0 = tx * 4;
    float acc[4][4];
    zero_acc(acc);

    auto stage = [&](int buf, long r0) {
#pragma unroll
        for (int it = 0; it < 2; ++it) {
            int idx = tid + it * NTHREADS;           // 512 float4 per operand
            int rr = idx >> 4, cq = (idx & 15) * 4;
            long r = r0 + rr;
            float *da = &As[buf][rr][cq], *db = &Bs[buf][rr][cq];
            if (vec) {
                if (r < r_end && tm + cq < M) cp_async16(da, A + r * lda + tm + cq);
                else *reinterpret_cast<float4 *>(da) = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < r_end && tn + cq < N) cp_async16(db, B + r * ldb + tn + cq);
                else *reinterpret_cast<float4 *>(db) = make_float4(0.f, 0.f, 0.f, 0.f);
            } else {   // unaligned operands (e.g. an 86-class head): scalar staging
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    da[q] = (r < r_end && tm + cq + q < M) ? A[r * lda + tm + cq + q] : 0.f;
                    db[q] = (r < r_end && tn + cq + q < N) ? B[r * ldb + tn + cq + q] : 0.f;
                }
            }
        }
    };
    const long nchunks = (r_end - r_begin + RT - 1) / RT;
    stage(0, r_begin);
    cp_async_commit();
    for (long c = 0; c < nchunks; ++c) {
        const int cur = c & 1;
        if (c + 1 < nchunks) {
            stage(cur ^ 1, r_begin + (c + 1) * RT);
            cp_async_commit();
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < RT; ++kk) {
            float4 x = *reinterpret_cast<const float4 *>(&As[cur][kk][m0]);
            float4 y = *reinterpret_cast<const float4 *>(&Bs[cur][kk][n0]);
            acc[0][0] += x.x * y.x; acc[0][1] += x.x * y.y; acc[0][2] += x.x * y.z; acc[0][3] += x.x * y.w;
            acc[1][0] += x.y * y.x; acc[1][1] += x.y * y.y; acc[1][2] += x.y * y.z; acc[1][3] += x.y * y.w;
            acc[2][0] += x.z * y.x; acc[2][1] += x.z * y.y; acc[2][2] += x.z * y.z; acc[2][3] += x.z * y.w;
            acc[3][0] += x.w * y.x; acc[3][1] += x.w * y.y; acc[3][2] += x.w * y.z; acc[3][3] += x.w * y.w;
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
            if (tm + m0 + a < M && tn + n0 + b < N)       // deterministic mode: slot blockIdx.y of the (M,N) partials
                det_put(C + (long)(tm + m0 + a) * ldc + tn + n0 + b,
                        part ? part + ((long)blockIdx.y * M + tm + m0 + a) * N + tn + n0 + b : nullptr, acc[a][b]);
}

// out[n*ostride] += sum_r B[r*ldb + n]
__global__ void __launch_bounds__(NTHREADS) colsum_kernel(const float *__restrict__ B, int ldb,
                                                          float *__restrict__ out, int ostride, long rows, int N,
                                                          long rows_per_cta, float *__restrict__ part) {
    __shared__ float red[4][64];
    const int col = blockIdx.x * 64 + (threadIdx.x & 63), rg = threadIdx.x >> 6;
    const long r_begin = (long)blockIdx.y * rows_per_cta;
    const long r_end = min(rows, r_begin + rows_per_cta);
    float s = 0.f;
    if (col < N)
        for (long r = r_begin + rg; r < r_end; r += 4) s += B[r * ldb + col];
    red[rg][threadIdx.x & 63] = s;
    __syncthreads();
    if (rg == 0 && col < N) {
        s = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
        det_put(out + (long)col * ostride, part ? part + (long)blockIdx.y * N + col : nullptr, s);
    }
}

// ---- links.Linear -------------------------------------------------------------
// MODE 0: Y[r][o] = act(sum_k X[r][k] W[o][k] + b[o])       (forward,  W (out,in))
// MODE 1: Y[r][k] = sum_o X[r][o] W[o][k]                    (backward data)
// 64x64 tile of Y per CTA; thread rows are interleaved (tx + 16 a) to keep the
// k-contiguous float4 reads of the X tile conflict-free.
template <int MODE>
__global__ void __launch_bounds__(NTHREADS) linear_kernel(const float *__restrict__ X, const float *__restrict__ W,
                                                          const float *__restrict__ bias, float *__restrict__ Y,
                                                          long rows, int in_dim, int out_dim, int act) {
    // X tile [64 r][KT k] (k contiguous); W tile MODE0: [64 o][KT k]; MODE1: [KT o][64 k]
    __shared__ __align__(16) float Xs[64][XLD];
    __shared__ __align__(16) float Ws[64 * XLD];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const long r0 = (long)blockIdx.x * 64;
    const int c0 = blockIdx.y * 64;                 // output-column tile
    const int Kred = MODE == 0 ? in_dim : out_dim;  // reduction length
    const int Nout = MODE == 0 ? out_dim : in_dim;
    const int ldx = Kred, ldw = in_dim;
    float acc[4][4];
    zero_acc(acc);
    for (int k0 = 0; k0 < Kred; k0 += KT) {
        for (int idx = tid; idx < 64 * KT; idx += NTHREADS) {
            int rr = idx / KT, kk = idx % KT;
            long r = r0 + rr;
            Xs[rr][kk] = (r < rows && k0 + kk < Kred) ? X[r * ldx + k0 + kk] : 0.f;
        }
        if (MODE == 0) {
            for (int idx = tid; idx < 64 * KT; idx += NTHREADS) {
                int oo = idx / KT, kk = idx % KT;
                Ws[oo * XLD + kk] = (c0 + oo < out_dim && k0 + kk < in_dim) ? W[(long)(c0 + oo) * ldw + k0 + kk] : 0.f;
            }
        } else {
            for (int idx = tid; idx < KT * 64; idx += NTHREADS) {
                int oo = idx / 64, kk = idx % 64;   // oo: reduction (out) index, kk: output (in) column
                Ws[oo * WLD + kk] = (k0 + oo < out_dim && c0 + kk < in_dim) ? W[(long)(k0 + oo) * ldw + c0 + kk] : 0.f;
            }
        }
        __syncthreads();
        if (MODE == 0) {
#pragma unroll
            for (int kk = 0; kk < KT; kk += 4) {
                float4 x[4], w[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) x[a] = *reinterpret_cast<const float4 *>(&Xs[tx + 16 * a][kk]);
#pragma unroll
                for (int b = 0; b < 4; ++b) w[b] = *reinterpret_cast<const float4 *>(&Ws[(ty * 4 + b) * XLD + kk]);
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b)
                        acc[a][b] += x[a].x * w[b].x + x[a].y * w[b].y + x[a].z * w[b].z + x[a].w * w[b].w;
            }
        } else {
#pragma unroll
            for (int kk = 0; kk < KT; kk += 4) {
                float4 x[4], w[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) x[a] = *reinterpret_cast<const float4 *>(&Xs[tx + 16 * a][kk]);
#pragma unroll
                for (int q = 0; q < 4; ++q) w[q] = *reinterpret_cast<const float4 *>(&Ws[(kk + q) * WLD + ty * 4]);
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    acc[a][0] += x[a].x * w[0].x + x[a].y * w[1].x + x[a].z * w[2].x + x[a].w * w[3].x;
                    acc[a][1] += x[a].x * w[0].y + x[a].y * w[1].y + x[a].z * w[2].y + x[a].w * w[3].y;
                    acc[a][2] += x[a].x * w[0].z + x[a].y * w[1].z + x[a].z * w[2].z + x[a].w * w[3].z;
                    acc[a][3] += x[a].x * w[0].w + x[a].y * w[1].w + x[a].z * w[2].w + x[a].w * w[3].w;
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        long r = r0 + tx + 16 * a;
        if (r >= rows) continue;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int c = c0 + ty * 4 + b;
            if (c >= Nout) continue;
            float v = acc[a][b];
            if (MODE == 0) {
                if (bias) v += bias[c];
                v = act_fwd(act, v);
            }
            Y[r * Nout + c] = v;
        }
    }
}

// dy <- dy * act'(y)   (derivative through the activation OUTPUT)
__global__ void act_bwd_kernel(float *__restrict__ dy, const float *__restrict__ y, long n, int act) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float yy = y[i], d = 1.f;
    if (act == BMP_ACT_TANH) d = 1.f - yy * yy;
    else if (act == BMP_ACT_RELU) d = yy > 0.f ? 1.f : 0.f;
    else if (act == BMP_ACT_SIGMOID) d = yy * (1.f - yy);
    dy[i] *= d;
}

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

}  // namespace bmp

using namespace bmp;

extern "C" int bmp_wgrad(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                         int64_t rows, int M, int N, void *stream) {
    if (!A || !B || !C) { set_error("bmp_wgrad: null pointer"); return BMP_EINVAL; }
    if (rows <= 0 || M <= 0 || N <= 0) return BMP_OK;
    const int vec = !((lda & 3) || (ldb & 3) || (M & 3) || (N & 3) || ((uintptr_t)A & 15) || ((uintptr_t)B & 15));
    const int tilesM = (M + 63) / 64, tilesN = (N + 63) / 64;
    const int tiles = tilesM * tilesN;
    long split = (4L * sm_count() + tiles - 1) / tiles;
    long max_split = (rows + 4 * RT - 1) / (4 * RT);
    if (split > max_split) split = max_split;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    long rpc = (rows + split - 1) / split;
    rpc = (rpc + RT - 1) / RT * RT;
    split = (rows + rpc - 1) / rpc;
    dim3 grid(tiles, (unsigned)split);
    Partials pt((cudaStream_t)stream);
    float *part = det_on() ? pt.take(split * M * N) : nullptr;
    if (det_on() && !part) return BMP_EINVAL;
    wgrad_kernel<<<grid, NTHREADS, 0, (cudaStream_t)stream>>>(A, lda, B, ldb, C, ldc, rows, M, N, tilesN, rpc, vec, part);
    count_launch();
    int rc = check_launch("wgrad_kernel");
    if (rc || !part) return rc;
    pt.add(C, ldc, M, N, part, (int)split, (long)M * N);
    return pt.reduce("det_reduce_kernel (bmp_wgrad)");
}

extern "C" int bmp_colsum(const float *B, int ldb, float *out, int out_stride, int64_t rows, int N, void *stream) {
    if (!B || !out) { set_error("bmp_colsum: null pointer"); return BMP_EINVAL; }
    if (rows <= 0 || N <= 0) return BMP_OK;
    const int tiles = (N + 63) / 64;
    long split = (2L * sm_count() + tiles - 1) / tiles;
    long max_split = (rows + 255) / 256;
    if (split > max_split) split = max_split;
    if (split < 1) split = 1;
    if (split > 65535) split = 65535;
    long rpc = (rows + split - 1) / split;
    split = (rows + rpc - 1) / rpc;
    dim3 grid(tiles, (unsigned)split);
    Partials pt((cudaStream_t)stream);
    float *part = det_on() ? pt.take(split * N) : nullptr;
    if (det_on() && !part) return BMP_EINVAL;
    colsum_kernel<<<grid, NTHREADS, 0, (cudaStream_t)stream>>>(B, ldb, out, out_stride, rows, N, rpc, part);
    count_launch();
    int rc = check_launch("colsum_kernel");
    if (rc || !part) return rc;
    pt.add(out, out_stride, N, 1, part, (int)split, N);
    return pt.reduce("det_reduce_kernel (bmp_colsum)");
}

extern "C" int bmp_linear_forward(const float *x, const float *W, const float *b, float *y,
                                  int rows, int in_dim, int out_dim, int act, void *stream) {
    if (!x || !W || !y) { set_error("bmp_linear_forward: null pointer"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    if (in_dim <= 0 || out_dim <= 0) { set_error("bmp_linear_forward: bad dims"); return BMP_ESHAPE; }
    dim3 grid((rows + 63) / 64, (out_dim + 63) / 64);
    linear_kernel<0><<<grid, NTHREADS, 0, (cudaStream_t)stream>>>(x, W, b, y, rows, in_dim, out_dim, act);
    count_launch();
    return check_launch("linear_kernel<0>");
}

extern "C" int bmp_linear_backward(const float *x, const float *W, const float *y, float *dy,
                                   float *dx, float *dW, float *db,
                                   int rows, int in_dim, int out_dim, int act, void *stream) {
    if (!x || !W || !dy) { set_error("bmp_linear_backward: null pointer"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (act != BMP_ACT_IDENTITY) {
        if (!y) { set_error("bmp_linear_backward: y needed for a non-identity activation"); return BMP_EINVAL; }
        long n = (long)rows * out_dim;
        act_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dy, y, n, act);
        count_launch();
        if ((rc = check_launch("act_bwd_kernel"))) return rc;
    }
    if (dx) {
        dim3 grid((rows + 63) / 64, (in_dim + 63) / 64);
        linear_kernel<1><<<grid, NTHREADS, 0, st>>>(dy, W, nullptr, dx, rows, in_dim, out_dim, 0);
        count_launch();
        if ((rc = check_launch("linear_kernel<1>"))) return rc;
    }
    if (dW) {
        if ((rc = bmp_wgrad(dy, out_dim, x, in_dim, dW, in_dim, rows, out_dim, in_dim, stream))) return rc;
    }
    if (db && (rc = bmp_colsum(dy, out_dim, db, 1, rows, out_dim, stream))) return rc;
    return BMP_OK;
}

// Deterministic sibling (det.cuh): dW / db summed over the row split in fixed order in `scratch`.
extern "C" size_t bmp_linear_backward_det_bytes(int rows, int in_dim, int out_dim) {
    if (rows <= 0 || in_dim <= 0 || out_dim <= 0) return 0;
    const size_t a = det_wgrad_bytes(out_dim, in_dim), b = det_colsum_bytes(out_dim);
    return a > b ? a : b;
}
extern "C" int bmp_linear_backward_det(const float *x, const float *W, const float *y, float *dy, float *dx, float *dW, float *db,
                                       int rows, int in_dim, int out_dim, int act, void *stream, void *scratch, size_t scratch_bytes) {
    if (!scratch) { set_error("bmp_linear_backward_det: NULL scratch"); return BMP_EINVAL; }
    int rc = det_check("bmp_linear_backward_det", scratch, scratch_bytes, bmp_linear_backward_det_bytes(rows, in_dim, out_dim));
    if (rc) return rc;
    DetScope ds(scratch, scratch_bytes);
    return bmp_linear_backward(x, W, y, dy, dx, dW, db, rows, in_dim, out_dim, act, stream);
}
