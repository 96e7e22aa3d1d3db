// misc.cu -- library housekeeping + the small warp-level kernels of the path:
// HolE circular correlation (models/link_prediction/hole.py:28-50), EmbedAtomID
// backward, sigmoid cross-entropy (train_binary.py:524), Adam (train_binary.py:533).
#include <cstdarg>
#include <cstdio>
#include <atomic>
#include <mutex>
#include <vector>
#include "det.cuh"

namespace bmp {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
bool aligned16(std::initializer_list<const void *> ps) {
    for (const void *q : ps)
        if (q && ((uintptr_t)q & 15)) return false;
    return true;
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

// ---- per-kernel timing with CUDA events on the launching stream (bench.py's roofline legs)
static std::atomic<int> g_prof_on{0};
struct ProfRec { int kind; cudaEvent_t e0, e1; };
static std::mutex g_prof_mu;
static std::vector<ProfRec> g_prof;
ProfScope::ProfScope(int kind_, cudaStream_t st_) : kind(kind_), st(st_), slot(nullptr) {
    if (!g_prof_on.load(std::memory_order_relaxed)) return;
    ProfRec *r = new ProfRec;
    r->kind = kind;
    cudaEventCreate(&r->e0);
    cudaEventCreate(&r->e1);
    cudaEventRecord(r->e0, st);
    slot = r;
}
ProfScope::~ProfScope() {
    if (!slot) return;
    ProfRec *r = (ProfRec *)slot;
    cudaEventRecord(r->e1, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(*r);
    delete r;
}
int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return BMP_ECUDA;
    }
    return BMP_OK;
}

// ---- HolE: c[k] = sum_i l[i] r[(i+k) mod D].  One warp per pair, vectors in smem.
constexpr int HOLE_WARPS = 8;
__global__ void __launch_bounds__(HOLE_WARPS * 32) hole_fwd_kernel(const float *__restrict__ L, const float *__restrict__ R,
                                                                   float *__restrict__ out, int mb, int D) {
    extern __shared__ float sm[];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *l = sm + w * 3 * D, *r2 = l + D;       // r2 holds r twice: no modulo in the inner loop
    for (int p = blockIdx.x * HOLE_WARPS + w; p < mb; p += gridDim.x * HOLE_WARPS) {
        __syncwarp();
        for (int i = lane; i < D; i += 32) {
            l[i] = L[(long)p * D + i];
            float v = R[(long)p * D + i];
            r2[i] = v;
            r2[i + D] = v;
        }
        __syncwarp();
        for (int k = lane; k < D; k += 32) {
            float s = 0.f;
            for (int i = 0; i < D; ++i) s += l[i] * r2[i + k];
            out[(long)p * D + k] = s;
        }
    }
}

// dl[i] = sum_k dc[k] r[(i+k) mod D] ; dr[j] = sum_k dc[k] l[(j-k) mod D]
__global__ void __launch_bounds__(HOLE_WARPS * 32) hole_bwd_kernel(const float *__restrict__ L, const float *__restrict__ R,
                                                                   const float *__restrict__ dC, float *__restrict__ dL,
                                                                   float *__restrict__ dR, int mb, int D) {
    extern __shared__ float sm[];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *l2 = sm + w * 5 * D, *r2 = l2 + 2 * D, *dc = r2 + 2 * D;
    for (int p = blockIdx.x * HOLE_WARPS + w; p < mb; p += gridDim.x * HOLE_WARPS) {
        __syncwarp();
        for (int i = lane; i < D; i += 32) {
            float a = L[(long)p * D + i], b = R[(long)p * D + i];
            l2[i] = a; l2[i + D] = a;
            r2[i] = b; r2[i + D] = b;
            dc[i] = dC[(long)p * D + i];
        }
        __syncwarp();
        for (int i = lane; i < D; i += 32) {
            float s1 = 0.f, s2 = 0.f;
            for (int k = 0; k < D; ++k) {
                s1 += dc[k] * r2[i + k];
                s2 += dc[k] * l2[i + D - k];
            }
            dL[(long)p * D + i] = s1;
            dR[(long)p * D + i] = s2;
        }
    }
}

// ---- EmbedAtomID backward: per-CTA smem table, then global atomics -------------
__global__ void __launch_bounds__(256) embed_bwd_kernel(const int32_t *__restrict__ ids, const float *__restrict__ dh,
                                                        float *__restrict__ dW, long rows, int H, int n_types,
                                                        long rows_per_cta) {
    extern __shared__ float tab[];   // [n_types][H]
    const int n = n_types * H;
    for (int i = threadIdx.x; i < n; i += blockDim.x) tab[i] = 0.f;
    __syncthreads();
    const long r0 = (long)blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
    for (long e = r0 * H + threadIdx.x; e < r1 * H; e += blockDim.x) {
        long r = e / H;
        int c = (int)(e - r * H);
        int id = ids[r];
        id = id < 0 ? 0 : (id >= n_types ? n_types - 1 : id);
        atomicAdd(&tab[id * H + c], dh[e]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float v = tab[i];
        if (v != 0.f) atomicAdd(dW + i, v);
    }
}

// (ldh = row stride of dh: H, or the full width when a deterministic call runs one column tile of a wide table.)
// Atomic-free variant: a CTA owns a contiguous block of rows; its 256 threads form two row partitions of 128
// column owners.  A thread is the only writer of "its" columns of its partition's private table, so the
// scatter-add is a plain shared-memory read-modify-write in row order; the two tables are merged on the way out.
// (fp32 shared-memory atomics are compare-and-swap loops and serialise on the few frequent atom types.)
constexpr int EMB_U = 16;
__global__ void __launch_bounds__(256) embed_bwd_owner_kernel(const int32_t *__restrict__ ids, const float *__restrict__ dh,
                                                              float *__restrict__ dW, long rows, int H, int n_types,
                                                              long rows_per_cta, float *__restrict__ slots, long ldh) {
    extern __shared__ float tab[];   // [2][n_types][H]
    const int n = n_types * H;
    for (int i = threadIdx.x; i < 2 * n; i += blockDim.x) tab[i] = 0.f;
    __syncthreads();
    const int part = threadIdx.x >> 7, t = threadIdx.x & 127;
    float *mine = tab + part * n;
    const long r0 = (long)blockIdx.x * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
    for (int c = t; c < H; c += 128) {
        // partitions interleave blocks of EMB_U rows; the next block's loads are in flight while this one is applied
        int id[2][EMB_U];
        float v[2][EMB_U];
        auto fetch = [&](int b, long r) {
#pragma unroll
            for (int u = 0; u < EMB_U; ++u) {
                const bool ok = r + u < r1;
                const int x = ok ? __ldg(ids + r + u) : 0;
                id[b][u] = x < 0 ? 0 : (x >= n_types ? n_types - 1 : x);
                v[b][u] = ok ? __ldg(dh + (r + u) * ldh + c) : 0.f;
            }
        };
        long r = r0 + part * EMB_U;
        if (r < r1) fetch(0, r);
        for (; r < r1; r += 4 * EMB_U) {
            if (r + 2 * EMB_U < r1) fetch(1, r + 2 * EMB_U);
#pragma unroll
            for (int u = 0; u < EMB_U; ++u) mine[id[0][u] * H + c] += v[0][u];
            if (r + 2 * EMB_U >= r1) break;
            if (r + 4 * EMB_U < r1) fetch(0, r + 4 * EMB_U);
#pragma unroll
            for (int u = 0; u < EMB_U; ++u) mine[id[1][u] * H + c] += v[1][u];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = tab[i] + tab[n + i];
        if (slots) slots[(long)blockIdx.x * n + i] = v;       // deterministic mode: slot blockIdx.x
        else if (v != 0.f) atomicAdd(dW + i, v);
    }
}

// ---- sigmoid cross entropy ------------------------------------------------------
__global__ void __launch_bounds__(256) sce_kernel(const float *__restrict__ x, const int32_t *__restrict__ t,
                                                  float *__restrict__ loss, float *__restrict__ dx, long n, float inv_count,
                                                  float *__restrict__ part) {
    __shared__ float red[8];
    float s = 0.f;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        float xv = x[i];
        int tv = t[i];
        float keep = tv != -1 ? 1.f : 0.f;
        float per = -(xv * ((float)tv - (xv >= 0.f ? 1.f : 0.f)) - log1pf(expf(-fabsf(xv))));
        s += keep * per;
        if (dx) dx[i] = keep * (sigmoidf_(xv) - (float)tv) * inv_count;
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 8) {
        s = red[threadIdx.x];
        for (int o = 4; o; o >>= 1) s += __shfl_xor_sync(0xffu, s, o);
        if (threadIdx.x == 0 && loss) det_put(loss, part ? part + blockIdx.x : nullptr, s * inv_count);
    }
}

// ---- Adam (chainer.optimizers.Adam: alpha_t = alpha*sqrt(1-b2^t)/(1-b1^t); decoupled weight decay)
__global__ void adam_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                            float *__restrict__ v, long n, float alpha_t, float beta1, float beta2, float eps,
                            float wd, float eta) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float gi = g[i];
    float mi = m[i] + (1.f - beta1) * (gi - m[i]);
    float vi = v[i] + (1.f - beta2) * (gi * gi - v[i]);
    m[i] = mi;
    v[i] = vi;
    p[i] -= eta * (alpha_t * mi / (sqrtf(vi) + eps) + wd * p[i]);
}

}  // namespace bmp

using namespace bmp;

extern "C" const char *bmp_last_error(void) { return g_err; }
extern "C" int bmp_version(void) { return 101; }
extern "C" uint64_t bmp_launch_count(void) { return g_launches.load(); }
extern "C" void bmp_reset_launch_count(void) { g_launches.store(0); }

extern "C" void bmp_profile_enable(int on) { bmp::g_prof_on.store(on != 0); }
extern "C" int bmp_profile_read(double *ms, long long *launches, int n_kinds) {
    using namespace bmp;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int i = 0; i < n_kinds; ++i) { ms[i] = 0.0; launches[i] = 0; }
    int rc = BMP_OK;
    for (auto &r : g_prof) {
        float t = 0.f;
        if (cudaEventSynchronize(r.e1) != cudaSuccess || cudaEventElapsedTime(&t, r.e0, r.e1) != cudaSuccess) rc = BMP_ECUDA;
        if (r.kind >= 0 && r.kind < n_kinds) { ms[r.kind] += t; launches[r.kind] += 1; }
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    g_prof.clear();
    return rc;
}

extern "C" int bmp_device_check(void) {
    int dev = 0, major = 0, minor = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { set_error("no CUDA device"); return BMP_ECUDA; }
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    if (major != 10) { set_error("device is sm_%d%d; this library is built for sm_100a only", major, minor); return BMP_EARCH; }
    return BMP_OK;
}

extern "C" int bmp_hole_corr_forward(const float *left, const float *right, float *out, int mb, int dim, void *stream) {
    if (!left || !right || !out) { set_error("bmp_hole_corr_forward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (dim <= 0 || dim > 1024) { set_error("bmp_hole_corr_forward: dim=%d outside 1..1024", dim); return BMP_ESHAPE; }
    size_t smem = (size_t)HOLE_WARPS * 3 * dim * sizeof(float);
    int grid = (mb + HOLE_WARPS - 1) / HOLE_WARPS;
    if (grid > 148 * 8) grid = 148 * 8;
    cudaFuncSetAttribute(hole_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    hole_fwd_kernel<<<grid, HOLE_WARPS * 32, smem, (cudaStream_t)stream>>>(left, right, out, mb, dim);
    count_launch();
    return check_launch("hole_fwd_kernel");
}

extern "C" int bmp_hole_corr_backward(const float *left, const float *right, const float *d_out,
                                      float *d_left, float *d_right, int mb, int dim, void *stream) {
    if (!left || !right || !d_out || !d_left || !d_right) { set_error("bmp_hole_corr_backward: null pointer"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_OK;
    if (dim <= 0 || dim > 1024) { set_error("bmp_hole_corr_backward: dim=%d outside 1..1024", dim); return BMP_ESHAPE; }
    size_t smem = (size_t)HOLE_WARPS * 5 * dim * sizeof(float);
    int grid = (mb + HOLE_WARPS - 1) / HOLE_WARPS;
    if (grid > 148 * 8) grid = 148 * 8;
    cudaFuncSetAttribute(hole_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    hole_bwd_kernel<<<grid, HOLE_WARPS * 32, smem, (cudaStream_t)stream>>>(left, right, d_out, d_left, d_right, mb, dim);
    count_launch();
    return check_launch("hole_bwd_kernel");
}

// Columns per launch of the owner kernel: its two [n_types][cols] tables fit 200 KB of shared memory.  The default path runs it
// when the whole table fits; the deterministic path also runs wider tables as column tiles (the fallback kernel below
// scatters with shared-memory atomics, whose order is not fixed).
static int embed_tile_cols(int hidden, int n_atom_types) {
    const long c = 200L * 1024 / (2 * sizeof(float)) / (n_atom_types > 0 ? n_atom_types : 1);
    return c >= hidden ? hidden : (int)(c & ~3L);
}
static size_t embed_det_bytes(int rows, int hidden, int n_atom_types) {
    const int tc = embed_tile_cols(hidden, n_atom_types);
    if (rows <= 0 || hidden <= 0 || n_atom_types <= 0 || tc < 4) return 0;
    return 148 * (size_t)n_atom_types * tc * sizeof(float) + 512;
}

// One owner-kernel launch over columns [c0, c0 + cols) of the table (all of it when cols == hidden).
static int embed_owner(const int32_t *atoms, const float *dh, float *d_embed_W, int rows, int hidden, int c0, int cols,
                       int n_atom_types, cudaStream_t st) {
    const size_t smem = (size_t)n_atom_types * cols * sizeof(float);
    const int ctas = 148;
    long rpc = ((long)rows + ctas - 1) / ctas;
    rpc = (rpc + 2 * EMB_U - 1) / (2 * EMB_U) * (2 * EMB_U);
    const int grid = (int)(((long)rows + rpc - 1) / rpc);
    Partials pt(st);
    const long n = (long)n_atom_types * cols;
    float *part = det_on() ? pt.take(grid * n) : nullptr;
    if (det_on() && !part) return BMP_EINVAL;
    cudaFuncSetAttribute(embed_bwd_owner_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * smem));
    embed_bwd_owner_kernel<<<grid, 256, 2 * smem, st>>>(atoms, dh + c0, d_embed_W + c0, rows, cols, n_atom_types, rpc, part, hidden);
    count_launch();
    int rc = check_launch("embed_bwd_owner_kernel");
    if (rc || !part) return rc;
    pt.add(d_embed_W + c0, hidden, n_atom_types, cols, part, grid, n);
    return pt.reduce("det_reduce_kernel (bmp_embed_backward)");
}

extern "C" int bmp_embed_backward(const int32_t *atoms, const float *dh, float *d_embed_W,
                                  int rows, int hidden, int n_atom_types, void *stream) {
    if (!atoms || !dh || !d_embed_W) { set_error("bmp_embed_backward: null pointer"); return BMP_EINVAL; }
    if (rows <= 0) return BMP_OK;
    size_t smem = (size_t)n_atom_types * hidden * sizeof(float);
    const cudaStream_t st = (cudaStream_t)stream;
    if (2 * smem <= 200 * 1024) return embed_owner(atoms, dh, d_embed_W, rows, hidden, 0, hidden, n_atom_types, st);
    if (det_on()) {
        const int tc = embed_tile_cols(hidden, n_atom_types);
        if (tc < 4) { set_error("bmp_embed_backward_det: %d atom types do not fit a 4-column tile", n_atom_types); return BMP_ESHAPE; }
        for (int c0 = 0; c0 < hidden; c0 += tc) {
            const int rc = embed_owner(atoms, dh, d_embed_W, rows, hidden, c0, hidden - c0 < tc ? hidden - c0 : tc, n_atom_types, st);
            if (rc) return rc;
        }
        return BMP_OK;
    }
    if (smem > 200 * 1024) { set_error("bmp_embed_backward: table %d x %d does not fit shared memory", n_atom_types, hidden); return BMP_ESHAPE; }
    int grid = 148 * 2;
    long rpc = ((long)rows + grid - 1) / grid;
    if (rpc < 64) rpc = 64;
    grid = (int)(((long)rows + rpc - 1) / rpc);
    cudaFuncSetAttribute(embed_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    embed_bwd_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(atoms, dh, d_embed_W, rows, hidden, n_atom_types, rpc);
    count_launch();
    return check_launch("embed_bwd_kernel");
}

extern "C" int bmp_sigmoid_ce(const float *logits, const int32_t *labels, float *loss_sum,
                              float *d_logits, int n, float count, void *stream) {
    if (!logits || !labels) { set_error("bmp_sigmoid_ce: null pointer"); return BMP_EINVAL; }
    if (n <= 0) return BMP_OK;
    int grid = (n + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    Partials pt((cudaStream_t)stream);
    float *part = det_on() && loss_sum ? pt.take(grid) : nullptr;
    if (det_on() && loss_sum && !part) return BMP_EINVAL;
    sce_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logits, labels, loss_sum, d_logits, n, 1.f / (count > 0.f ? count : 1.f), part);
    count_launch();
    int rc = check_launch("sce_kernel");
    if (rc || !part) return rc;
    pt.add(loss_sum, 1, 1, 1, part, grid, 1);
    return pt.reduce("det_reduce_kernel (bmp_sigmoid_ce)");
}

// ---- deterministic siblings (det.cuh): the same work with fixed-order cross-CTA sums in `scratch`
extern "C" size_t bmp_embed_backward_det_bytes(int rows, int hidden, int n_atom_types) {
    return embed_det_bytes(rows, hidden, n_atom_types);
}
extern "C" int bmp_embed_backward_det(const int32_t *atoms, const float *dh, float *d_embed_W, int rows, int hidden,
                                      int n_atom_types, void *stream, void *scratch, size_t scratch_bytes) {
    if (!scratch) { set_error("bmp_embed_backward_det: NULL scratch"); return BMP_EINVAL; }
    int rc = det_check("bmp_embed_backward_det", scratch, scratch_bytes, embed_det_bytes(rows, hidden, n_atom_types));
    if (rc) return rc;
    DetScope ds(scratch, scratch_bytes);
    return bmp_embed_backward(atoms, dh, d_embed_W, rows, hidden, n_atom_types, stream);
}
extern "C" size_t bmp_sigmoid_ce_det_bytes(int n) {
    if (n <= 0) return 0;
    const long grid = (n + 255) / 256 > 148 * 8 ? 148 * 8 : (n + 255) / 256;
    return (size_t)grid * sizeof(float) + 512;
}
extern "C" int bmp_sigmoid_ce_det(const float *logits, const int32_t *labels, float *loss_sum, float *d_logits, int n, float count,
                                  void *stream, void *scratch, size_t scratch_bytes) {
    if (!scratch) { set_error("bmp_sigmoid_ce_det: NULL scratch"); return BMP_EINVAL; }
    int rc = det_check("bmp_sigmoid_ce_det", scratch, scratch_bytes, bmp_sigmoid_ce_det_bytes(n));
    if (rc) return rc;
    DetScope ds(scratch, scratch_bytes);
    return bmp_sigmoid_ce(logits, labels, loss_sum, d_logits, n, count, stream);
}

extern "C" int bmp_adam_step(float *param, const float *grad, float *m, float *v, int n,
                             float alpha, float beta1, float beta2, float eps,
                             float weight_decay_rate, int step, void *stream) {
    if (!param || !grad || !m || !v) { set_error("bmp_adam_step: null pointer"); return BMP_EINVAL; }
    if (n <= 0) return BMP_OK;
    double fix1 = 1.0 - pow((double)beta1, step), fix2 = 1.0 - pow((double)beta2, step);
    float alpha_t = (float)(alpha * sqrt(fix2) / fix1);
    adam_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(param, grad, m, v, n, alpha_t, beta1, beta2, eps,
                                                                  weight_decay_rate, 1.f);
    count_launch();
    return check_launch("adam_kernel");
}
