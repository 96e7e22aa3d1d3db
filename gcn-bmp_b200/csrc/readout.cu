// readout.cu -- gated sum readout atoms -> molecule vector.
// R1: models/readout/ggnn_readout.py:42-58; R2: models/ggnn_att.py:338-346,
// models/ggnn_dev.py:113-122; SUM: models/ggnn_dev.py:167.
// One CTA per molecule; [h | h0] channel-major in shared memory; the two linears
// run as 64x64 register tiles; the sum over atoms is a 16-lane shuffle reduction.
// Molecules of up to BMP_X3_MAX_ATOMS atoms are walked in 64-atom chunks: the forward
// carries the per-molecule sum across chunks in g, the backward needs no cross-chunk
// state (an atom's gradient depends on dg and its own row only).  Up to 64 atoms there
// is one chunk and the arithmetic is that of the single-tile kernel.
#include "common.cuh"
#include "det.cuh"

namespace bmp {

__device__ __forceinline__ float reduce16(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v;
}

// BWD = false: g = act_agg(sum_n mask * sigmoid(u) * act(v))
// BWD = true : recompute u, v; write DU/DV (+ smem copies), then dh1 = W_i^T du + W_j^T dv.
template <bool BWD>
__global__ void __launch_bounds__(NTHREADS, 1) readout_kernel(const bmp_readout_fwd_t f, const bmp_readout_bwd_t bw) {
    extern __shared__ __align__(16) float smem[];
    const int mb = BWD ? bw.mb : f.mb, N = BWD ? bw.n_atoms : f.n_atoms, H = BWD ? bw.hidden : f.hidden;
    const int O = BWD ? bw.out_dim : f.out_dim, variant = BWD ? bw.variant : f.variant;
    const int act = BWD ? bw.act : f.act, act_agg = BWD ? bw.act_agg : f.act_agg;
    const float *h = BWD ? bw.h : f.h, *h0 = BWD ? bw.h0 : f.h0, *mask = BWD ? bw.is_real_node : f.is_real_node;
    const float *W_i = BWD ? bw.W_i : f.W_i, *b_i = BWD ? bw.b_i : f.b_i;
    const float *W_j = BWD ? bw.W_j : f.W_j, *b_j = BWD ? bw.b_j : f.b_j;
    const int Kcat = h0 ? 2 * H : H;
    const int Ki = Kcat, Kj = (variant == BMP_READOUT_R2) ? H : Kcat;
    float *hcat = smem;                       // [Kcat][64]
    float *du_s = hcat + Kcat * AT;           // [O][64]  (BWD only)
    float *dv_s = du_s + (BWD ? O * AT : 0);  // [O][64]
    float *stage = dv_s + (BWD ? O * AT : 0);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, i0 = tx * 4;

    const int nchunks = (N + AT - 1) / AT;
    for (int mol = blockIdx.x; mol < mb; mol += gridDim.x) {
        for (int ch = 0; ch < nchunks; ++ch) {
            const long row0 = (long)mol * N + ch * AT;
            const int n = min(AT, N - ch * AT);
            __syncthreads();
            load_cm(hcat, h + row0 * H, n, H);
            if (h0) load_cm(hcat + H * AT, h0 + row0 * H, n, H);
            __syncthreads();
            float mk[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) mk[b] = (i0 + b < n) ? (mask ? mask[row0 + i0 + b] : 1.f) : 0.f;

            for (int oc = 0; oc * 64 < O; ++oc) {
                float au[4][4], av[4][4];
                zero_acc(au);
                zero_acc(av);
                gemm64_g<false>(au, W_i, Ki, oc * 64, O, Ki, hcat, stage);
                gemm64_g<false>(av, W_j, Kj, oc * 64, O, Kj, hcat, stage);
                const int o0 = oc * 64 + ty * 4;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const bool live = o0 + q < O;
                    const float bi = (live && b_i) ? b_i[o0 + q] : 0.f, bj = (live && b_j) ? b_j[o0 + q] : 0.f;
                    if (!BWD) {
                        float s = 0.f;
#pragma unroll
                        for (int b = 0; b < 4; ++b) s += mk[b] * sigmoidf_(au[q][b] + bi) * act_fwd(act, av[q][b] + bj);
                        s = reduce16(s);
                        if (tx == 0 && live) {     // partial sums of earlier chunks wait in g (same thread)
                            float *gp = f.g + (long)mol * O + o0 + q;
                            if (ch) s += *gp;
                            *gp = ch + 1 == nchunks ? act_fwd(act_agg, s) : s;
                        }
                    } else {
                        float dsum = 0.f;
                        if (live) {
                            float gout = bw.g[(long)mol * O + o0 + q];
                            dsum = bw.dg[(long)mol * O + o0 + q] * act_bwd(act_agg, gout, gout);
                            // relu on the aggregate: derivative through the output sign is exact (y>0 <=> x>0)
                        }
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            float u = au[q][b] + bi, v = av[q][b] + bj;
                            float su = sigmoidf_(u), av_ = act_fwd(act, v);
                            au[q][b] = dsum * mk[b] * av_ * su * (1.f - su);
                            av[q][b] = dsum * mk[b] * su * act_bwd(act, v, av_);
                        }
                    }
                }
                if (BWD && o0 < O) {
                    tile_store_s(du_s, oc * 64, au);
                    tile_store_s(dv_s, oc * 64, av);
                    tile_store_g(bw.DU + row0 * O, O, oc * 64, O, n, au);
                    tile_store_g(bw.DV + row0 * O, O, oc * 64, O, n, av);
                }
            }
            if (BWD) {
                __syncthreads();
                for (int kc = 0; kc * 64 < Kcat; ++kc) {
                    float d[4][4];
                    zero_acc(d);
                    gemm64_g<true>(d, W_i, Ki, kc * 64, Ki, O, du_s, stage);
                    if (kc * 64 < Kj) gemm64_g<true>(d, W_j, Kj, kc * 64, Kj, O, dv_s, stage);
                    // accumulate into dh (k < H) / dh0 (k >= H); a 64-chunk never straddles H unless H % 64 != 0
                    const int k0 = kc * 64 + ty * 4;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        if (i0 + b >= n) continue;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            int k = k0 + q;
                            if (k >= Kcat) continue;
                            float *dst = (k < H) ? bw.dh : bw.dh0;
                            if (dst) dst[(row0 + i0 + b) * H + (k < H ? k : k - H)] += d[q][b];
                        }
                    }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(NTHREADS) readout_sum_kernel(const float *__restrict__ h, const float *__restrict__ mask,
                                                               float *__restrict__ g, int mb, int N, int H) {
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long)mb * H; idx += (long)gridDim.x * blockDim.x) {
        long mol = idx / H;
        int c = (int)(idx - mol * H);
        float s = 0.f;
        for (int i = 0; i < N; ++i) s += h[(mol * N + i) * H + c] * (mask ? mask[mol * N + i] : 1.f);
        g[idx] = s;
    }
}
__global__ void __launch_bounds__(NTHREADS) readout_sum_bwd_kernel(const float *__restrict__ dg, const float *__restrict__ mask,
                                                                   float *__restrict__ dh, int mb, int N, int H) {
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long)mb * N * H; idx += (long)gridDim.x * blockDim.x) {
        long row = idx / H;
        int c = (int)(idx - row * H);
        long mol = row / N;
        dh[idx] += dg[mol * H + c] * (mask ? mask[row] : 1.f);
    }
}

static int readout_check(int mb, int N, int H, int O, int variant, const float *h) {
    if (!h) { set_error("readout: null h"); return BMP_EINVAL; }
    if (mb <= 0) return BMP_ESHAPE;
    if (N <= 0 || N > BMP_X3_MAX_ATOMS) { set_error("readout: n_atoms=%d outside 1..%d", N, BMP_X3_MAX_ATOMS); return BMP_ESHAPE; }
    if (H <= 0 || (H & 3) || H > BMP_MAX_HIDDEN) { set_error("readout: hidden=%d must be a multiple of 4 <= %d", H, BMP_MAX_HIDDEN); return BMP_ESHAPE; }
    if (variant != BMP_READOUT_SUM && (O <= 0 || (O & 3))) { set_error("readout: out_dim=%d must be a positive multiple of 4", O); return BMP_ESHAPE; }
    return BMP_OK;
}

}  // namespace bmp

using namespace bmp;

int bmp_readout_tc(int mb, int N, int H, int O, int variant, int act, int act_agg, const float *h, const float *h0,
                   const float *mask, const float *W_i, const float *b_i, const float *W_j, const float *b_j,
                   float *g, const float *dg, float *DU, float *DV, float *dh, float *dh0, void *ws, size_t ws_bytes,
                   bool images_ready, bool bwd, void *stream);   // readout_tc.cu

bool bmp_readout_x3_usable(const bmp_readout_fwd_t *a);                          // ggnn_x3.cu: BMP_MODE_F32 forward on tcgen05 (split bf16)
int bmp_readout_forward_x3(const bmp_readout_fwd_t *a, void *stream);

extern "C" int bmp_readout_forward(const bmp_readout_fwd_t *a, void *stream) {
    if (!a || !a->g) { set_error("bmp_readout_forward: null argument"); return BMP_EINVAL; }
    int rc = readout_check(a->mb, a->n_atoms, a->hidden, a->out_dim, a->variant, a->h);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (a->variant == BMP_READOUT_SUM) {
        long n = (long)a->mb * a->hidden;
        readout_sum_kernel<<<(unsigned)((n + 255) / 256), NTHREADS, 0, st>>>(a->h, a->is_real_node, a->g, a->mb, a->n_atoms, a->hidden);
        count_launch();
        return check_launch("readout_sum_kernel");
    }
    if (!a->W_i || !a->W_j) { set_error("bmp_readout_forward: null weights"); return BMP_EINVAL; }
    if (!aligned16({a->W_i, a->W_j, a->h, a->h0})) { set_error("bmp_readout_forward: h, h0, W_i, W_j must be 16-byte aligned"); return BMP_EINVAL; }
    // BF16 mode above 64 atoms: the fp32 kernels (the tcgen05 read-out maps one molecule onto a 64-row tile)
    if (a->mode == BMP_MODE_BF16 && a->n_atoms <= BMP_MAX_ATOMS && bmp_readout_tc_workspace_bytes(a->hidden, a->out_dim)) {
        return bmp_readout_tc(a->mb, a->n_atoms, a->hidden, a->out_dim, a->variant, a->act, a->act_agg, a->h, a->h0,
                              a->is_real_node, a->W_i, a->b_i, a->W_j, a->b_j, a->g, nullptr, nullptr, nullptr, nullptr, nullptr,
                              a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, false, stream);
    }
    if (bmp_readout_x3_usable(a)) return bmp_readout_forward_x3(a, stream);
    const int Kcat = a->h0 ? 2 * a->hidden : a->hidden;
    size_t smem = sizeof(float) * ((size_t)Kcat * AT + STAGE_FLOATS);
    int grid = a->mb < 148 * 2 ? a->mb : 148 * 2;
    bmp_readout_bwd_t dummy = {};
    cudaFuncSetAttribute(readout_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    readout_kernel<false><<<grid, NTHREADS, smem, st>>>(*a, dummy);
    count_launch();
    return check_launch("readout_kernel<fwd>");
}

static int readout_backward_impl(const bmp_readout_bwd_t *a, void *stream) {
    if (!a || !a->dg) { set_error("bmp_readout_backward: null argument"); return BMP_EINVAL; }
    int rc = readout_check(a->mb, a->n_atoms, a->hidden, a->out_dim, a->variant, a->h);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int H = a->hidden, O = a->out_dim;
    const long rows = (long)a->mb * a->n_atoms;
    if (a->variant == BMP_READOUT_SUM) {
        if (!a->dh) return BMP_OK;
        long n = rows * H;
        readout_sum_bwd_kernel<<<(unsigned)((n + 255) / 256), NTHREADS, 0, st>>>(a->dg, a->is_real_node, a->dh, a->mb, a->n_atoms, H);
        count_launch();
        return check_launch("readout_sum_bwd_kernel");
    }
    if (!a->W_i || !a->W_j || !a->g || !a->DU || !a->DV) { set_error("bmp_readout_backward: null argument"); return BMP_EINVAL; }
    if (!aligned16({a->W_i, a->W_j, a->h, a->h0, a->DU, a->DV, a->dh, a->dh0})) { set_error("bmp_readout_backward: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    const int Kcat = a->h0 ? 2 * H : H;
    const int Kj = a->variant == BMP_READOUT_R2 ? H : Kcat;
    const bool tc = a->mode == BMP_MODE_BF16 && a->n_atoms <= BMP_MAX_ATOMS && H <= 128 && O <= 128 && bmp_readout_tc_workspace_bytes(H, O) != 0;   // 256: forward-only
    if (tc) {
        if ((rc = bmp_readout_tc(a->mb, a->n_atoms, H, O, a->variant, a->act, a->act_agg, a->h, a->h0, a->is_real_node,
                                 a->W_i, a->b_i, a->W_j, a->b_j, const_cast<float *>(a->g), a->dg, a->DU, a->DV, a->dh, a->dh0,
                                 a->tc_workspace, a->tc_workspace_bytes, a->tc_images_ready != 0, true, stream)))
            return rc;
    } else {
        size_t smem = sizeof(float) * ((size_t)(Kcat + 2 * O) * AT + STAGE_FLOATS);
        if (smem > 227 * 1024) {
            set_error("bmp_readout_backward: hidden=%d out_dim=%d needs %zu B of shared memory", H, O, smem);
            return BMP_ESHAPE;
        }
        int grid = a->mb < 148 ? a->mb : 148;
        bmp_readout_fwd_t dummy = {};
        cudaFuncSetAttribute(readout_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        readout_kernel<true><<<grid, NTHREADS, smem, st>>>(dummy, *a);
        count_launch();
        if ((rc = check_launch("readout_kernel<bwd>"))) return rc;
    }
    // parameter gradients: C += A^T B over all atoms (tcgen05 contraction with fused bias sums in BF16 mode)
    auto WG = [&](const float *A_, const float *B_, float *C_, int ldc, float *db) -> int {
        if (tc) return bmp_wgrad_tc(A_, O, B_, H, C_, ldc, rows, O, H, db, 1, stream);
        int e_ = bmp_wgrad(A_, O, B_, H, C_, ldc, rows, O, H, stream);
        if (!e_ && db) e_ = bmp_colsum(A_, O, db, 1, rows, O, stream);
        return e_;
    };
    bool bi_done = false, bj_done = false;
    if (a->d_W_i) {
        if ((rc = WG(a->DU, a->h, a->d_W_i, Kcat, a->d_b_i))) return rc;
        bi_done = true;
        if (a->h0 && (rc = WG(a->DU, a->h0, a->d_W_i + H, Kcat, nullptr))) return rc;
    }
    if (a->d_W_j) {
        if ((rc = WG(a->DV, a->h, a->d_W_j, Kj, a->d_b_j))) return rc;
        bj_done = true;
        if (a->h0 && Kj > H && (rc = WG(a->DV, a->h0, a->d_W_j + H, Kj, nullptr))) return rc;
    }
    if (a->d_b_i && !bi_done && (rc = bmp_colsum(a->DU, O, a->d_b_i, 1, rows, O, stream))) return rc;
    if (a->d_b_j && !bj_done && (rc = bmp_colsum(a->DV, O, a->d_b_j, 1, rows, O, stream))) return rc;
    return BMP_OK;
}

// Bytes of det_scratch (deterministic mode, det.cuh) that bmp_readout_backward needs for this filled-in struct; 0 = no shape to cover.
extern "C" size_t bmp_readout_backward_det_bytes(const bmp_readout_bwd_t *a) {
    if (!a) return 0;
    if (a->mb <= 0 || a->n_atoms <= 0 || a->hidden <= 0 || a->out_dim <= 0) return 0;
    const int O = a->out_dim, K = 2 * a->hidden;
    return det_max({det_wgrad_bytes(O, K), det_wgrad_tc_bytes(O, K), det_colsum_bytes(O)});
}
extern "C" int bmp_readout_backward(const bmp_readout_bwd_t *a, void *stream) {
    if (a && a->det_scratch) {
        int rc = det_check("bmp_readout_backward", a->det_scratch, a->det_scratch_bytes, bmp_readout_backward_det_bytes(a));
        if (rc) return rc;
    }
    DetScope ds(a ? a->det_scratch : nullptr, a ? a->det_scratch_bytes : 0);
    return readout_backward_impl(a, stream);
}
