// wgrad_tc.cu -- parameter-gradient contraction C (M,N) += A^T B on tcgen05.
//
// A (rows, M) and B (rows, N) are the fp32 stashes of a micro-batch (rows = atoms x steps, millions);
// the reduction runs over rows, so both operands are "MN-major" for the tensor core: a staged chunk of
// 64 rows is converted to bf16 and stored as SW128 MN-major blocks [64 k-rows][64 columns] by 8 loader
// warps, one elected lane issues M=128 x N x 16 UMMAs into a TMEM accumulator that lives for the whole
// row range of the CTA, and the epilogue adds the tile into C with fp32 atomics (split over rows across
// CTAs).  Column sums of A (the bias gradients) are accumulated by the loaders on the way.
//
// SPLIT = true (bmp_wgrad_tc3, used by BMP_MODE_F32): fp32-grade contraction on the same pipeline -- every operand is staged as a
// bf16 hi / lo pair (x = hi + lo up to 2^-17 relative) and each k-step issues three UMMAs, hi.hi + lo.hi + hi.lo, into the fp32
// TMEM accumulator (the lo.lo term is below fp32 rounding of the sum).
#include <cuda_bf16.h>
#include "det.cuh"

namespace bmp {
namespace wtc {

constexpr int KT = 64;
constexpr int NLOAD = 256;
constexpr int NTHR = 288;
constexpr int STAGES = 2;
constexpr int BLK = 64 * 128;     // one MN block: 64 k-rows x 64 columns bf16

__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
constexpr uint32_t MBAR_SUSPEND_NS = 20000;     // suspend-time hint of try_wait (see tc_common.cuh)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(MBAR_SUSPEND_NS) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t *>(&t);
}
// MN-major SW128 descriptor: LBO = stride between 64-column blocks, SBO = 8 k-rows = 1024 B
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(BLK >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
__host__ __device__ constexpr uint32_t idesc_mnmn(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}

// lo part of a hi / lo bf16 split: bf16(x - float(hi)), for four values packed like `hi`
__device__ __forceinline__ uint2 lo_of(const float4 &v, const uint2 &hi) {
    const float h0 = __uint_as_float(hi.x << 16), h1 = __uint_as_float(hi.x & 0xFFFF0000u);
    const float h2 = __uint_as_float(hi.y << 16), h3 = __uint_as_float(hi.y & 0xFFFF0000u);
    return make_uint2(pack_bf16(v.x - h0, v.y - h1), pack_bf16(v.z - h2, v.w - h3));
}

struct Args {
    const float *A, *B;
    float *C, *dbias;
    int lda, ldb, ldc, M, N, bias_stride;
    long rows, rows_per_cta;
    float *part, *bpart;     // deterministic mode: [split][M][N] and [split][M] partials (slot blockIdx.y), else nullptr
};

template <int N, bool SPLIT>
__global__ void __launch_bounds__(NTHR, SPLIT ? 1 : 2) wgrad_tc_kernel(const Args a) {
    constexpr int NB = N / 64;                       // MN blocks of the B stage
    constexpr int A_BYTES = 2 * BLK, B_BYTES = NB * BLK, HALF_BYTES = A_BYTES + B_BYTES;
    constexpr int STAGE_BYTES = (SPLIT ? 2 : 1) * HALF_BYTES;      // SPLIT: [A_hi | B_hi | A_lo | B_lo]
    constexpr int BQ = N / 4;                        // float4 per B row
    constexpr int BJ = KT * BQ / NLOAD;              // float4 of B per loader thread per chunk
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const uint32_t sbase = s32(smem);
    const uint32_t s_bar = sbase + STAGES * STAGE_BYTES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + STAGES * STAGE_BYTES + 64);
    float *cs_red = reinterpret_cast<float *>(smem + STAGES * STAGE_BYTES + 128);    // [8][128]
    auto FULL = [&](int s) { return s_bar + 8u * s; };
    auto EMPTY = [&](int s) { return s_bar + 8u * (STAGES + s); };
    const uint32_t DONE = s_bar + 8u * (2 * STAGES);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tm = blockIdx.x * 128;
    const long r_begin = (long)blockIdx.y * a.rows_per_cta;
    const long r_end = min(a.rows, r_begin + a.rows_per_cta);
    const int nchunks = (int)((r_end - r_begin + KT - 1) / KT);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(FULL(s), NLOAD); mbar_init(EMPTY(s), 1); }
        mbar_init(DONE, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"(N));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp == 8) {
        if (lane == 0) {
            constexpr uint32_t ID = idesc_mnmn(N);
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % STAGES;
                mbar_wait(FULL(s), (c / STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t sa = sbase + s * STAGE_BYTES, sb = sa + A_BYTES;
#pragma unroll
                for (int k = 0; k < KT / 16; ++k) {
                    const uint64_t da = desc_mn(sa + k * 16 * 128), db = desc_mn(sb + k * 16 * 128);
                    const uint32_t acc = (c | k) ? 1u : 0u;
                    auto mma = [&](uint64_t xa, uint64_t xb, uint32_t ac) {
                        asm volatile(
                            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                            ::"r"(tmem), "l"(xa), "l"(xb), "r"(ID), "r"(ac) : "memory");
                    };
                    mma(da, db, acc);                                                  // hi . hi
                    if (SPLIT) {
                        const uint64_t la = desc_mn(sa + HALF_BYTES + k * 16 * 128), lb = desc_mn(sb + HALF_BYTES + k * 16 * 128);
                        mma(la, db, 1u);                                               // lo . hi
                        mma(da, lb, 1u);                                               // hi . lo
                    }
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(EMPTY(s)) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(DONE) : "memory");
        }
    } else {
        // ---------------- loaders: fp32 global -> bf16 SW128 MN-major blocks ----------------
        const int am4 = (tid & 31) * 4, ak0 = tid >> 5;              // A: column group, first row (rows ak0 + 8 j)
        const int bn4 = (tid % BQ) * 4, bk0 = tid / BQ;              // B: column group, first row (rows bk0 + (NLOAD/BQ) j)
        const bool a_live = tm + am4 < a.M;
        float csum[4] = {0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < nchunks; ++c) {
            const int s = c % STAGES;
            const long r0 = r_begin + (long)c * KT;
            float4 va[8], vb[BJ];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const long r = r0 + ak0 + 8 * j;
                va[j] = (a_live && r < r_end) ? __ldg(reinterpret_cast<const float4 *>(a.A + r * a.lda + tm + am4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < BJ; ++j) {
                const long r = r0 + bk0 + (NLOAD / BQ) * j;
                vb[j] = (r < r_end) ? __ldg(reinterpret_cast<const float4 *>(a.B + r * a.ldb + bn4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            mbar_wait(EMPTY(s), ((c / STAGES) & 1) ^ 1);
            uint8_t *sa = smem + s * STAGE_BYTES, *sb = sa + A_BYTES;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = ak0 + 8 * j;
                csum[0] += va[j].x; csum[1] += va[j].y; csum[2] += va[j].z; csum[3] += va[j].w;
                const uint32_t off = (am4 >> 6) * BLK + k * 128 + (((((am4 & 63) >> 3) ^ (k & 7)) << 4) | ((am4 & 7) << 1));
                const uint2 hi = make_uint2(pack_bf16(va[j].x, va[j].y), pack_bf16(va[j].z, va[j].w));
                *reinterpret_cast<uint2 *>(sa + off) = hi;
                if (SPLIT) *reinterpret_cast<uint2 *>(sa + HALF_BYTES + off) = lo_of(va[j], hi);
            }
#pragma unroll
            for (int j = 0; j < BJ; ++j) {
                const int k = bk0 + (NLOAD / BQ) * j;
                const uint32_t off = (bn4 >> 6) * BLK + k * 128 + (((((bn4 & 63) >> 3) ^ (k & 7)) << 4) | ((bn4 & 7) << 1));
                const uint2 hi = make_uint2(pack_bf16(vb[j].x, vb[j].y), pack_bf16(vb[j].z, vb[j].w));
                *reinterpret_cast<uint2 *>(sb + off) = hi;
                if (SPLIT) *reinterpret_cast<uint2 *>(sb + HALF_BYTES + off) = lo_of(vb[j], hi);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_arrive(FULL(s));
        }
        // ---------------- bias gradient: column sums of A ----------------
        if (a.dbias) {
            cs_red[(tid >> 5) * 128 + am4 + 0] = csum[0];
            cs_red[(tid >> 5) * 128 + am4 + 1] = csum[1];
            cs_red[(tid >> 5) * 128 + am4 + 2] = csum[2];
            cs_red[(tid >> 5) * 128 + am4 + 3] = csum[3];
            asm volatile("bar.sync 1, %0;" ::"n"(NLOAD));
            if (tid < 128 && tm + tid < a.M) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < 8; ++w) t += cs_red[w * 128 + tid];
                det_put(a.dbias + (long)(tm + tid) * a.bias_stride, a.bpart ? a.bpart + (long)blockIdx.y * a.M + tm + tid : nullptr, t);
            }
        }
        // ---------------- epilogue: TMEM -> C (fp32 atomics) ----------------
        mbar_wait(DONE, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3, hf = warp >> 2;
        const int m = nchunks > 0 ? tm + 32 * q + lane : a.M;    // a CTA without rows adds nothing
        const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16) + hf * (N / 2);
#pragma unroll
        for (int cc = 0; cc < N / 2; cc += 32) {
            uint32_t v[32];
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr + cc) : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (m < a.M) {
                float *dst = a.C + (long)m * a.ldc + hf * (N / 2) + cc;
                if (a.part) {                           // N % 64 == 0: the slot row is 16-byte aligned
                    float *pp = a.part + ((long)blockIdx.y * a.M + m) * N + hf * (N / 2) + cc;
#pragma unroll
                    for (int x = 0; x < 32; x += 4)
                        det_put4(nullptr, pp + x, make_float4(__uint_as_float(v[x]), __uint_as_float(v[x + 1]), __uint_as_float(v[x + 2]), __uint_as_float(v[x + 3])));
                } else if ((((uintptr_t)dst) & 15) == 0) {
#pragma unroll
                    for (int x = 0; x < 32; x += 4)      // 128-bit vector reductions: 4x fewer L2 atomic operations
                        atomicAdd(reinterpret_cast<float4 *>(dst + x),
                                  make_float4(__uint_as_float(v[x]), __uint_as_float(v[x + 1]), __uint_as_float(v[x + 2]), __uint_as_float(v[x + 3])));
                } else {
#pragma unroll
                    for (int x = 0; x < 32; ++x) atomicAdd(dst + x, __uint_as_float(v[x]));
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 8) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(N));
    }
}

template <int N, bool SPLIT>
static int launch(const Args &a, cudaStream_t st, int sms) {
    constexpr int smem = STAGES * (SPLIT ? 2 : 1) * (2 * BLK + (N / 64) * BLK) + 128 + 8 * 128 * 4 + 1024;
    const int mtiles = (a.M + 127) / 128;
    long split = (1L * sms + mtiles - 1) / mtiles;
    long max_split = (a.rows + 8 * KT - 1) / (8 * KT);
    if (split > max_split) split = max_split;
    if (split < 1) split = 1;
    Args k = a;
    k.rows_per_cta = ((a.rows + split - 1) / split + KT - 1) / KT * KT;
    split = (a.rows + k.rows_per_cta - 1) / k.rows_per_cta;
    Partials pt(st);
    k.part = k.bpart = nullptr;
    if (det_on()) {
        if (!(k.part = pt.take(split * a.M * N))) return BMP_EINVAL;
        if (a.dbias && !(k.bpart = pt.take(split * a.M))) return BMP_EINVAL;
    }
    cudaFuncSetAttribute(wgrad_tc_kernel<N, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    wgrad_tc_kernel<N, SPLIT><<<dim3(mtiles, (unsigned)split), NTHR, smem, st>>>(k);
    count_launch();
    int rc = check_launch("wgrad_tc_kernel");
    if (rc || !k.part) return rc;
    pt.add(a.C, a.ldc, a.M, N, k.part, (int)split, (long)a.M * N);
    if (k.bpart) pt.add(a.dbias, a.bias_stride, a.M, 1, k.bpart, (int)split, a.M);
    return pt.reduce("det_reduce_kernel (bmp_wgrad_tc)");
}

}  // namespace wtc
}  // namespace bmp

using namespace bmp;

// C (M,N; ldc) += A^T B on the tensor cores (bf16 operands, fp32 accumulate); dbias[m*bias_stride] +=
// column sums of A when non-NULL.  N must be 64, 128 or 256 and everything 16-byte aligned; returns
// BMP_ESHAPE otherwise so the caller can use the fp32 bmp_wgrad.
static int wgrad_tc_any(bool split3, const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                        int64_t rows, int M, int N, float *dbias, int bias_stride, void *stream) {
    if (!A || !B || !C) { set_error("bmp_wgrad_tc: null pointer"); return BMP_EINVAL; }
    if (rows <= 0 || M <= 0) return BMP_OK;
    if ((N != 64 && N != 128 && N != 256) || (M & 3) || (lda & 3) || (ldb & 3) || !aligned16({A, B})) {
        set_error("bmp_wgrad_tc: unsupported shape/alignment (M=%d N=%d lda=%d ldb=%d)", M, N, lda, ldb);
        return BMP_ESHAPE;
    }
    static int sms = 0;
    if (!sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    wtc::Args a;
    a.A = A; a.B = B; a.C = C; a.dbias = dbias; a.lda = lda; a.ldb = ldb; a.ldc = ldc; a.M = M; a.N = N;
    a.bias_stride = bias_stride; a.rows = rows; a.rows_per_cta = 0;
    cudaStream_t st = (cudaStream_t)stream;
    if (split3) {
        if (N == 64) return wtc::launch<64, true>(a, st, sms);
        if (N == 128) return wtc::launch<128, true>(a, st, sms);
        return wtc::launch<256, true>(a, st, sms);
    }
    if (N == 64) return wtc::launch<64, false>(a, st, sms);
    if (N == 128) return wtc::launch<128, false>(a, st, sms);
    return wtc::launch<256, false>(a, st, sms);
}

// C (M,N; ldc) += A^T B on the tensor cores (bf16 operands, fp32 accumulate); dbias[m*bias_stride] +=
// column sums of A when non-NULL.  N must be 64, 128 or 256 and everything 16-byte aligned; returns
// BMP_ESHAPE otherwise so the caller can use the fp32 bmp_wgrad.
extern "C" int bmp_wgrad_tc(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                            int64_t rows, int M, int N, float *dbias, int bias_stride, void *stream) {
    return wgrad_tc_any(false, A, lda, B, ldb, C, ldc, rows, M, N, dbias, bias_stride, stream);
}

// The same contraction at fp32-grade accuracy: bf16 hi/lo split of both operands, three UMMAs per product, fp32 accumulate
// (relative error ~1e-5 against fp64; the BMP_MODE_F32 encoder backward uses it for its parameter gradients).
extern "C" int bmp_wgrad_tc3(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                             int64_t rows, int M, int N, float *dbias, int bias_stride, void *stream) {
    return wgrad_tc_any(true, A, lda, B, ldb, C, ldc, rows, M, N, dbias, bias_stride, stream);
}
