// det.cu -- the deterministic scratch of a call and the one fixed-order reduce kernel every site shares (det.cuh).
#include "det.cuh"

namespace bmp {

static thread_local void *g_det = nullptr;
static thread_local size_t g_det_bytes = 0;

DetScope::DetScope(void *scratch, size_t bytes) : prev(g_det), prev_bytes(g_det_bytes) {
    if (scratch) {          // NULL keeps the enclosing call's choice
        g_det = scratch;
        g_det_bytes = bytes;
    }
}
DetScope::~DetScope() {
    g_det = prev;
    g_det_bytes = prev_bytes;
}
bool det_on() { return g_det != nullptr; }

int sm_count_det() {
    static int sms = 0;
    if (!sms) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            sms = n;
        else {
            cudaGetLastError();
            return 148;
        }
    }
    return sms;
}

float *Partials::take(long floats) {
    const size_t off = (used + 255) & ~(size_t)255;
    const size_t need = off + (size_t)floats * sizeof(float);
    uint8_t *base = (uint8_t *)(((uintptr_t)g_det + 255) & ~(uintptr_t)255);
    const size_t have = g_det_bytes > (size_t)(base - (uint8_t *)g_det) ? g_det_bytes - (size_t)(base - (uint8_t *)g_det) : 0;
    if (!g_det || need > have) {
        set_error("deterministic scratch of %zu bytes is too small: this reduction needs %zu", g_det_bytes, need + 256);
        return nullptr;
    }
    if (cudaMemsetAsync(base + off, 0, (size_t)floats * sizeof(float), st) != cudaSuccess) {
        set_error("deterministic scratch: memset failed");
        return nullptr;
    }
    used = need;
    return (float *)(base + off);
}

void Partials::add(float *dst, long ld, int rows, int cols, const float *src, int parts, long pstride) {
    if (!dst || rows <= 0 || cols <= 0 || parts <= 0) return;
    if (nseg == DET_MAX_SEGS && !rc) rc = reduce("det_reduce_kernel");      // a full list: its launch runs first, in order
    segs[nseg++] = DetSeg{dst, src, ld, pstride, rows, cols, parts};
}

struct SegList {
    DetSeg s[DET_MAX_SEGS];
    int n;
};

// Thread (r, 4 columns): dst += the partials summed in slot order, fp32.  serial: every segment in list order (some
// destinations overlap); else segment blockIdx.y only (disjoint destinations: the order per element is the same).
__global__ void __launch_bounds__(256) det_reduce_kernel(const __grid_constant__ SegList L, int cq, long total, int serial) {
    const int k0 = serial ? 0 : (int)blockIdx.y, k1 = serial ? L.n : (int)blockIdx.y + 1;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int r = (int)(t / cq), c = (int)(t % cq) * 4;
#pragma unroll 1
        for (int k = k0; k < k1; ++k) {
            const DetSeg g = L.s[k];
            if (r >= g.rows || c >= g.cols) continue;
            const float *s = g.src + (long)r * g.cols + c;
            float *d = g.dst + (long)r * g.ld + c;
            const bool vec = c + 4 <= g.cols && !(g.cols & 3) && !(g.pstride & 3) && !(g.ld & 3) && !((uintptr_t)s & 15) &&
                             !((uintptr_t)d & 15);
            if (vec) {
                float4 a = *reinterpret_cast<const float4 *>(s);
                for (int p = 1; p < g.parts; ++p) {
                    const float4 b = *reinterpret_cast<const float4 *>(s + (long)p * g.pstride);
                    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
                }
                float4 o = *reinterpret_cast<float4 *>(d);
                o.x += a.x; o.y += a.y; o.z += a.z; o.w += a.w;
                *reinterpret_cast<float4 *>(d) = o;
            } else {
                for (int q = 0; q < 4 && c + q < g.cols; ++q) {
                    float a = s[q];
                    for (int p = 1; p < g.parts; ++p) a += s[(long)p * g.pstride + q];
                    d[q] += a;
                }
            }
        }
    }
}

// Whether two segments' destinations share an element.  Same leading dimension: compare row and column intervals (one
// segment shifted by the pointer difference, with the wrap into the next row); else compare the address ranges.
static bool overlap(const DetSeg &p, const DetSeg &q) {
    const DetSeg &x = p.dst <= q.dst ? p : q, &y = p.dst <= q.dst ? q : p;
    if (x.ld == y.ld && x.ld > 0) {
        const long d = (long)(y.dst - x.dst), rs = d / x.ld, cs = d % x.ld;
        auto hit = [&](long r0, long c0) { return r0 < x.rows && r0 + y.rows > 0 && c0 < x.cols && c0 + y.cols > 0; };
        return hit(rs, cs) || hit(rs + 1, cs - x.ld);
    }
    const float *x1 = x.dst + (long)(x.rows - 1) * x.ld + x.cols;
    return y.dst < x1;
}

int Partials::reduce(const char *site) {
    if (rc) return rc;
    if (!nseg) return BMP_OK;
    SegList L;
    L.n = nseg;
    int maxr = 0, maxc = 0;
    for (int k = 0; k < nseg; ++k) {
        L.s[k] = segs[k];
        maxr = segs[k].rows > maxr ? segs[k].rows : maxr;
        maxc = segs[k].cols > maxc ? segs[k].cols : maxc;
    }
    // destinations that overlap (tied parameters, the two targets of one sum) must be added by one thread in list order
    int serial = 0;
    for (int i = 0; i < nseg && !serial; ++i)
        for (int j = i + 1; j < nseg && !serial; ++j) {
            serial = overlap(segs[i], segs[j]);
        }
    const int cq = (maxc + 3) / 4;
    const long total = (long)maxr * cq;
    const int ny = serial ? 1 : nseg;
    long grid = (total + 255) / 256, cap = (8L * sm_count_det() + ny - 1) / ny;
    if (grid > cap) grid = cap;
    det_reduce_kernel<<<dim3((unsigned)grid, (unsigned)ny), 256, 0, st>>>(L, cq, total, serial);
    count_launch();
    nseg = 0;
    return check_launch(site);
}

// ---- sizes.  Each bound follows its site's split rule and is monotone in M and N: the split shrinks as the tile count grows,
// but split * M * N <= (S + tiles) * tile_area.  So a struct query may evaluate it at the largest M and the largest N of the
// calls it covers, and the result holds for every one of those calls.
static size_t pad(size_t floats) { return ((floats * sizeof(float) + 255) & ~(size_t)255); }
size_t det_wgrad_bytes(int M, int N) {          // gemm.cu bmp_wgrad: split <= ceil(4 S / tiles), 64 x 64 tiles
    if (M <= 0 || N <= 0) return 0;
    const size_t tiles = (size_t)((M + 63) / 64) * ((N + 63) / 64);
    return pad((4 * (size_t)sm_count_det() + tiles) * 4096) + 256;
}
size_t det_colsum_bytes(int N) {                // gemm.cu bmp_colsum: split <= ceil(2 S / tiles), 64-column tiles
    if (N <= 0) return 0;
    const size_t tiles = (N + 63) / 64;
    return pad((2 * (size_t)sm_count_det() + tiles) * 64) + 256;
}
size_t det_wgrad_tc_bytes(int M, int N) {       // wgrad_tc.cu: split <= ceil(S / mtiles), 128-row tiles, + bias partials
    if (M <= 0 || N <= 0) return 0;
    const size_t mt = (M + 127) / 128, parts = (size_t)sm_count_det() + mt;
    return pad(parts * 128 * (size_t)N) + pad(parts * 128) + 256;
}
size_t det_panels_bytes() {
    // per class at most 2 x 2 A blocks x 3 B blocks or 1 x 2 x 6 of 64 x 64 targets, plus 2 x 2 x 64 bias rows
    const long ctas = sm_count_det() > 6 ? sm_count_det() : 6;
    return (size_t)ctas * (49152 + 256) * sizeof(float) + 6 * 256 + 256;
}
size_t det_coattn_bytes(int mb, int H) {
    const long grid = mb < sm_count_det() ? mb : sm_count_det();
    return grid > 0 ? pad((size_t)grid * co_det_len(H)) + 256 : 0;
}

int det_check(const char *who, const void *scratch, size_t bytes, size_t need) {
    if (scratch && bytes < need) {
        set_error("%s: det_scratch of %zu bytes is too small, %zu bytes needed", who, bytes, need);
        return BMP_EINVAL;
    }
    return BMP_OK;
}

int co_det_begin(Partials &pt, CoDet &cd, int H, int grid) {
    cd.base = nullptr;
    cd.H = H;
    cd.len = co_det_len(H);
    if (!det_on()) return BMP_OK;
    cd.base = pt.take((long)grid * cd.len);
    return cd.base ? BMP_OK : BMP_EINVAL;
}

int co_det_end(Partials &pt, const CoDet &cd, int grid, int head, float *dW, float *dlt1, float *dlt2, float *dV1, float *dV2,
               float *dwa1, float *dwa2, float *db, bool with_w, const char *site) {
    if (!cd.base) return BMP_OK;
    const int H = cd.H;
    if (with_w) {
        pt.add(dW, H, H, H, cd.base + cd.w(), grid, cd.len);
        if (head > 0) {
            pt.add(dlt1, H, head, H, cd.base + cd.lt(0), grid, cd.len);
            pt.add(dlt2, H, head, H, cd.base + cd.lt(1), grid, cd.len);
        }
    }
    pt.add(dV1, H, 1, H, cd.base + cd.v(0), grid, cd.len);
    pt.add(dV2, H, 1, H, cd.base + cd.v(1), grid, cd.len);
    if (head > 0) {
        pt.add(dwa1, head, 1, head, cd.base + cd.wa(0), grid, cd.len);
        pt.add(dwa2, head, 1, head, cd.base + cd.wa(1), grid, cd.len);
    }
    pt.add(db, 1, 1, 1, cd.base + cd.b(), grid, cd.len);
    return pt.reduce(site);
}

}  // namespace bmp
