// det.cuh -- fixed-order cross-CTA reductions (deterministic mode).
//
// By default every parameter gradient, the loss sum and the clipping norm are finished with fp32 atomics across CTAs,
// so the order of the additions follows CTA timing and two runs differ in the last bits.  A caller that passes a
// deterministic scratch buffer (bmp_*_bwd_t.det_scratch, the *_det entry points) opens a DetScope for the call.  Inside
// it every such site instead gives each CTA its own slot of the scratch -- a zeroed [parts][len] fp32 array taken with
// Partials::take -- writes its partial there with det_put / det_put4, and after the kernel one shared reduce kernel
// (det_reduce) adds the slots into the destinations in slot order:  dst[i] += ((p_0 + p_1) + ...) + p_{P-1}.
// Sites run one after another on the stream, so they reuse the scratch from its start.  Without a scope nothing changes.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include "common.cuh"

namespace bmp {

// ---- host side
struct DetScope {                   // makes (scratch, bytes), when non-NULL, the deterministic scratch of this thread's call
    DetScope(void *scratch, size_t bytes);
    ~DetScope();
    void *prev; size_t prev_bytes;
};
bool det_on();                      // inside a DetScope with a non-NULL scratch
int sm_count_det();                 // SM count of the current device (148 when it cannot be read), as the sites size their grids

// One reduction segment: dst[r * ld + c] += sum_{p < parts} src[p * pstride + r * cols + c] for r < rows, c < cols.
// Segments of one det_reduce call are applied in list order by the same thread for the same (r, c), so two segments may
// name the same destination (tied parameters) without a race.
struct DetSeg {
    float *dst;
    const float *src;
    long ld, pstride;
    int rows, cols, parts;
};
constexpr int DET_MAX_SEGS = 96;

struct Partials {                   // the scratch of one site: bump allocation from the start of the buffer
    cudaStream_t st;
    size_t used = 0;
    DetSeg segs[DET_MAX_SEGS];
    int nseg = 0, rc = 0;
    explicit Partials(cudaStream_t s) : st(s) {}
    float *take(long floats);       // zeroed, 16-byte aligned; nullptr (error set) when the scratch is too small
    void add(float *dst, long ld, int rows, int cols, const float *src, int parts, long pstride);
    int reduce(const char *site);   // one launch of det_reduce_kernel over the collected segments
};

// Bytes of deterministic scratch the sites need (upper bounds that follow their launch configurations).
size_t det_wgrad_bytes(int M, int N);          // bmp_wgrad
size_t det_colsum_bytes(int N);                // bmp_colsum
size_t det_wgrad_tc_bytes(int M, int N);       // bmp_wgrad_tc / bmp_wgrad_tc3
size_t det_panels_bytes();                     // bmp_wgrad_panels_multi
size_t det_coattn_bytes(int mb, int H);        // the co-attention kernels' own flush
inline size_t det_max(std::initializer_list<size_t> v) {
    size_t m = 0;
    for (size_t x : v) m = x > m ? x : m;
    return m;
}
// Checks a caller's buffer against `need`; sets the error (naming `who` and the bytes) and returns BMP_EINVAL if short.
int det_check(const char *who, const void *scratch, size_t bytes, size_t need);

// ---- device side: the partial of this CTA (part != nullptr) or today's atomic (part == nullptr)
__device__ __forceinline__ void det_put(float *dst, float *part, float v) {
    if (part) *part += v;
    else atomicAdd(dst, v);
}
__device__ __forceinline__ void det_put4(float *dst, float *part, float4 v) {
    if (part) {
        float4 *p = reinterpret_cast<float4 *>(part);
        float4 o = *p;
        *p = make_float4(o.x + v.x, o.y + v.y, o.z + v.z, o.w + v.w);
    } else {
        atomicAdd(reinterpret_cast<float4 *>(dst), v);
    }
}

// Co-attention slot layout shared by coattn.cu, coattn_big.cu and coattn_tc.cu (per CTA):
//   [d W (H*H) | d lt_1 (16*H) | d lt_2 (16*H) | d V1 (H) | d V2 (H) | d wa_1 (16) | d wa_2 (16) | d b (1), padded to 4]
struct CoDet {
    float *base;        // nullptr: atomics
    long len;
    int H;
    __host__ __device__ long w() const { return 0; }
    __host__ __device__ long lt(int k) const { return (long)H * H + (long)k * 16 * H; }
    __host__ __device__ long v(int k) const { return (long)H * H + 32L * H + (long)k * H; }
    __host__ __device__ long wa(int k) const { return (long)H * H + 34L * H + 16L * k; }
    __host__ __device__ long b() const { return (long)H * H + 34L * H + 32; }
    __device__ float *slot(long off) const { return base ? base + (long)blockIdx.x * len + off : nullptr; }
};
__host__ __device__ inline long co_det_len(int H) { return ((long)H * H + 34L * H + 33 + 3) & ~3L; }
// Host: take the co-attention slots for `grid` CTAs (det mode) or return an inert CoDet.
int co_det_begin(Partials &pt, CoDet &cd, int H, int grid);
// Host: after the kernel, reduce the slots into the vector gradients (+ W / lt when `with_w`).
int co_det_end(Partials &pt, const CoDet &cd, int grid, int head, float *dW, float *dlt1, float *dlt2, float *dV1, float *dV2,
               float *dwa1, float *dwa2, float *db, bool with_w, const char *site);

}  // namespace bmp
