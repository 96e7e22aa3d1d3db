// relgcn.cu -- fused RelGCN encoder, fp32.
// Replaces models/relgcn.py:61-73 (embed -> rescale_adj -> L x tanh(RelGCNUpdate)),
// models/relgcn.py:20-28 (rescale_adj) and models/update/relgcn_update.py:24-44.
// One CTA per molecule for all layers; the layer is re-associated as
//   out = W_s h + b_s + sum_e W_e (A_e h) + b_e deg_e,   W_e = W_edge[e::E]
// exactly like the GGNN message (ggnn.cu), with the column-degree normalisation
// folded into the adjacency tile while it is staged.
#include "common.cuh"
#include "det.cuh"

namespace bmp {

__device__ __forceinline__ void colscale_compute(float *cscale, const float *__restrict__ adj, int N, int E) {
    // cscale[j] = 1 / sum_{e,i} adj[e][i][j]   (1 where the sum is 0)
    const int tid = threadIdx.x;
    __shared__ float part[4][AT];
    const int j = tid & 63, g = tid >> 6;
    float s = 0.f;
    if (j < N)
        for (int r = g; r < E * N; r += 4) s += adj[(long)r * N + j];
    part[g][j] = s;
    __syncthreads();
    if (tid < AT) {
        float t = part[0][tid] + part[1][tid] + part[2][tid] + part[3][tid];
        cscale[tid] = (tid < N && t != 0.f) ? 1.f / t : 1.f;
    }
    __syncthreads();
}

template <int HC>
__global__ void __launch_bounds__(NTHREADS, 1) relgcn_fwd_kernel(const bmp_relgcn_fwd_t a, int cmax) {
    extern __shared__ __align__(16) float smem[];
    float *hs = smem, *xs = hs + cmax * AT, *adj = xs + cmax * AT, *deg = adj + AT * AT, *cscale = deg + 8 * AT,
          *stage = cscale + AT;
    const int N = a.n_atoms, E = a.n_edge, L = a.n_layers;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, i0 = tx * 4;
    const long rows_total = (long)a.mb * N;
    const int K4 = (N + 3) & ~3;
    for (int mol = blockIdx.x; mol < a.mb; mol += gridDim.x) {
        const long row0 = (long)mol * N;
        const float *adjm = a.adj + (long)mol * E * N * N;
        __syncthreads();
        if (a.atoms) load_embed_cm(hs, a.atoms + row0, a.embed_W, N, a.ch[0], a.n_atom_types);
        else load_cm(hs, a.h_in + row0 * a.ch[0], N, a.ch[0]);
        if (a.scale_adj) colscale_compute(cscale, adjm, N, E);
        __syncthreads();
        if (a.Hs) store_cm(a.Hs + row0 * a.ch[0], a.ch[0], hs, N, a.ch[0]);
        long stash_off = rows_total * a.ch[0];
        for (int l = 0; l < L; ++l) {
            const int Cin = a.ch[l], Cout = a.ch[l + 1];
            float acc[HC][4][4];
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                zero_acc(acc[oc]);
                if (oc * 64 < Cout) gemm64_g<false>(acc[oc], a.self_W[l], Cin, oc * 64, Cout, Cin, hs, stage);
            }
            for (int e = 0; e < E; ++e) {
                load_adj<true>(adj, adjm + (long)e * N * N, N, a.scale_adj ? cscale : nullptr);
                __syncthreads();
                if (tid < AT) {
                    float d = 0.f;
                    for (int j = 0; j < N; ++j) d += adj[j * AT + tid];
                    deg[e * AT + tid] = d;
                }
                for (int kc = 0; kc * 64 < Cin; ++kc) {
                    if (kc * 64 + ty * 4 < Cin) {
                        float t[4][4];
                        zero_acc(t);
                        gemm64_s(t, hs, AT, kc * 64, K4, adj);
                        tile_store_s(xs, kc * 64, t);
                    }
                }
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc)
                    if (oc * 64 < Cout)
                        gemm64_g<false>(acc[oc], a.edge_W[l] + (long)e * Cin, (long)E * Cin, oc * 64, Cout, Cin, xs, stage);
            }
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                const int o0 = oc * 64 + ty * 4;
                if (oc * 64 >= Cout || o0 >= Cout) continue;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float bs = a.self_b[l] ? a.self_b[l][o0 + q] : 0.f;
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[oc][q][b] += bs;
                    if (a.edge_b[l])
                        for (int e = 0; e < E; ++e) {
                            float bb = a.edge_b[l][(long)(o0 + q) * E + e];
                            float4 d = *reinterpret_cast<const float4 *>(deg + e * AT + i0);
                            acc[oc][q][0] += bb * d.x; acc[oc][q][1] += bb * d.y;
                            acc[oc][q][2] += bb * d.z; acc[oc][q][3] += bb * d.w;
                        }
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[oc][q][b] = act_fwd(a.act, acc[oc][q][b]);
                }
            }
            __syncthreads();   // every reader of hs is done
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= Cout || oc * 64 + ty * 4 >= Cout) continue;
                tile_store_s(hs, oc * 64, acc[oc]);
                if (a.Hs) tile_store_g(a.Hs + stash_off + row0 * Cout, Cout, oc * 64, Cout, N, acc[oc]);
                if (l == L - 1 && a.h_out) tile_store_g(a.h_out + row0 * Cout, Cout, oc * 64, Cout, N, acc[oc]);
            }
            stash_off += rows_total * Cout;
            __syncthreads();
        }
    }
}

template <int HC>
__global__ void __launch_bounds__(NTHREADS, 1) relgcn_bwd_kernel(const bmp_relgcn_bwd_t a, int cmax) {
    extern __shared__ __align__(16) float smem[];
    float *gs = smem, *ps = gs + cmax * AT, *adj = ps + cmax * AT, *cscale = adj + AT * AT, *stage = cscale + AT;
    const int N = a.n_atoms, E = a.n_edge, L = a.n_layers;
    const int tid = threadIdx.x, ty = tid >> 4;
    const long rows_total = (long)a.mb * N;
    const int K4 = (N + 3) & ~3;
    long hs_off[BMP_MAX_STEPS + 2], ds_off[BMP_MAX_STEPS + 1], ps_off[BMP_MAX_STEPS + 1];
    hs_off[0] = 0; ds_off[0] = 0; ps_off[0] = 0;
    for (int l = 0; l < L; ++l) {
        hs_off[l + 1] = hs_off[l] + rows_total * a.ch[l];
        ds_off[l + 1] = ds_off[l] + rows_total * a.ch[l + 1];
        ps_off[l + 1] = ps_off[l] + rows_total * E * a.ch[l + 1];
    }
    for (int mol = blockIdx.x; mol < a.mb; mol += gridDim.x) {
        const long row0 = (long)mol * N;
        const float *adjm = a.adj + (long)mol * E * N * N;
        __syncthreads();
        load_cm(gs, a.d_h_out + row0 * a.ch[L], N, a.ch[L]);
        if (a.scale_adj) colscale_compute(cscale, adjm, N, E);
        __syncthreads();
        for (int l = L - 1; l >= 0; --l) {
            const int Cin = a.ch[l], Cout = a.ch[l + 1];
            // delta = g * (1 - h_{l+1}^2)  -> gs (in place) + Ds (global)
            for (int oc = 0; oc * 64 < Cout; ++oc) {
                if (oc * 64 + ty * 4 >= Cout) continue;
                float g[4][4], y[4][4];
                tile_load_s(gs, oc * 64, g);
                tile_load_g(a.Hs + hs_off[l + 1] + row0 * Cout, Cout, oc * 64, Cout, N, y);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int b = 0; b < 4; ++b) g[q][b] *= act_bwd(a.act, y[q][b], y[q][b]);
                tile_store_s(gs, oc * 64, g);
                tile_store_g(a.Ds + ds_off[l] + row0 * Cout, Cout, oc * 64, Cout, N, g);
            }
            __syncthreads();
            float dh[HC][4][4];
#pragma unroll
            for (int kc = 0; kc < HC; ++kc) {
                zero_acc(dh[kc]);
                if (kc * 64 < Cin) gemm64_g<true>(dh[kc], a.self_W[l], Cin, kc * 64, Cin, Cout, gs, stage);
            }
            for (int e = 0; e < E; ++e) {
                load_adj<false>(adj, adjm + (long)e * N * N, N, a.scale_adj ? cscale : nullptr);
                __syncthreads();
                for (int oc = 0; oc * 64 < Cout; ++oc) {
                    if (oc * 64 + ty * 4 >= Cout) continue;
                    float p[4][4];
                    zero_acc(p);
                    gemm64_s(p, gs, AT, oc * 64, K4, adj);
                    tile_store_s(ps, oc * 64, p);
                    tile_store_g(a.Ps + ps_off[l] + row0 * E * Cout + (long)e * Cout, (long)E * Cout, oc * 64, Cout, N, p);
                }
                __syncthreads();
#pragma unroll
                for (int kc = 0; kc < HC; ++kc)
                    if (kc * 64 < Cin)
                        gemm64_g<true>(dh[kc], a.edge_W[l] + (long)e * Cin, (long)E * Cin, kc * 64, Cin, Cout, ps, stage);
            }
            // g <- dh
#pragma unroll
            for (int kc = 0; kc < HC; ++kc) {
                if (kc * 64 >= Cin || kc * 64 + ty * 4 >= Cin) continue;
                tile_store_s(gs, kc * 64, dh[kc]);
                if (l == 0 && a.d_h0) tile_store_g(a.d_h0 + row0 * Cin, Cin, kc * 64, Cin, N, dh[kc]);
            }
            __syncthreads();
        }
    }
}

static int relgcn_check(int mb, int N, int E, int L, const int *ch, int *cmax, int max_atoms) {
    if (mb <= 0 || L <= 0 || L > BMP_MAX_STEPS) { set_error("relgcn: bad mb=%d or n_layers=%d", mb, L); return BMP_ESHAPE; }
    if (N <= 0 || N > max_atoms) { set_error("relgcn: n_atoms=%d outside 1..%d", N, max_atoms); return BMP_ESHAPE; }
    if (E <= 0 || E > 8) { set_error("relgcn: n_edge=%d outside 1..8", E); return BMP_ESHAPE; }
    *cmax = 0;
    for (int l = 0; l <= L; ++l) {
        if (ch[l] <= 0 || (ch[l] & 3) || ch[l] > BMP_MAX_HIDDEN) {
            set_error("relgcn: channel size %d must be a multiple of 4 in 4..%d", ch[l], BMP_MAX_HIDDEN);
            return BMP_ESHAPE;
        }
        if (ch[l] > *cmax) *cmax = ch[l];
    }
    return BMP_OK;
}

}  // namespace bmp

using namespace bmp;

bool bmp_relgcn_tc_supported(const int *ch, int n_layers, int n_edge);   // relgcn_tc.cu
int bmp_relgcn_forward_tc(const bmp_relgcn_fwd_t *a, void *stream);
int bmp_relgcn_backward_tc(const bmp_relgcn_bwd_t *a, void *stream);
// ggnn_x3.cu: BMP_MODE_F32 above BMP_MAX_ATOMS atoms
const char *bmp_relgcn_x3_refusal(int mb, int N, int E, int L, const int *ch, int act, const void *ws, size_t ws_bytes);
int bmp_relgcn_forward_x3(const bmp_relgcn_fwd_t *a, void *stream);
int bmp_relgcn_backward_x3(const bmp_relgcn_bwd_t *a, void *stream);

extern "C" int bmp_relgcn_forward(const bmp_relgcn_fwd_t *a, void *stream) {
    if (!a || !a->adj || (!a->atoms && !a->h_in) || (a->atoms && !a->embed_W)) {
        set_error("bmp_relgcn_forward: null argument");
        return BMP_EINVAL;
    }
    // BMP_MODE_F32 molecules with more than BMP_MAX_ATOMS atoms: the tensor-core row path of ggnn_x3.cu
    const bool x3 = a->mode == BMP_MODE_F32 && a->n_atoms > BMP_MAX_ATOMS;
    int cmax = 0;
    int rc = relgcn_check(a->mb, a->n_atoms, a->n_edge, a->n_layers, a->ch, &cmax, x3 ? BMP_X3_MAX_ATOMS : BMP_MAX_ATOMS);
    if (rc) return rc;
    for (int l = 0; l < a->n_layers; ++l)
        if (!a->self_W[l] || !a->edge_W[l] || !aligned16({a->self_W[l], a->edge_W[l]})) {
            set_error("bmp_relgcn_forward: null or misaligned (16 B) weights at layer %d", l);
            return BMP_EINVAL;
        }
    if (!aligned16({a->h_in, a->embed_W, a->h_out, a->Hs})) { set_error("bmp_relgcn_forward: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    if (a->mode == BMP_MODE_BF16) {
        if (!bmp_relgcn_tc_supported(a->ch, a->n_layers, a->n_edge)) {
            set_error("BMP_MODE_BF16 RelGCN: needs one channel count in {64,128} for all layers and 4 bond types");
            return BMP_ESHAPE;
        }
        return bmp_relgcn_forward_tc(a, stream);
    }
    if (a->adj_u8) { set_error("bmp_relgcn_forward: a byte adjacency needs BMP_MODE_BF16"); return BMP_EINVAL; }
    if (x3) {
        const char *why = bmp_relgcn_x3_refusal(a->mb, a->n_atoms, a->n_edge, a->n_layers, a->ch, a->act, a->tc_workspace, a->tc_workspace_bytes);
        if (*why) { set_error("relgcn: %s", why); return BMP_ESHAPE; }
        return bmp_relgcn_forward_x3(a, stream);
    }
    size_t smem = sizeof(float) * ((size_t)2 * cmax * AT + AT * AT + 8 * AT + AT + STAGE_FLOATS);
    int grid = a->mb < 148 ? a->mb : 148;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(HC)                                                                                           \
    do {                                                                                                     \
        cudaFuncSetAttribute(relgcn_fwd_kernel<HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        relgcn_fwd_kernel<HC><<<grid, NTHREADS, smem, st>>>(*a, cmax);                                       \
    } while (0)
    if (cmax <= 64) LAUNCH(1);
    else if (cmax <= 128) LAUNCH(2);
    else LAUNCH(4);
#undef LAUNCH
    count_launch();
    return check_launch("relgcn_fwd_kernel");
}

static int relgcn_backward_impl(const bmp_relgcn_bwd_t *a, void *stream) {
    if (a && a->mode == BMP_MODE_BF16) {
        if (!a->adj) { set_error("bmp_relgcn_backward: null argument"); return BMP_EINVAL; }
        if (a->mb <= 0 || a->n_atoms <= 0 || a->n_atoms > BMP_MAX_ATOMS || !bmp_relgcn_tc_supported(a->ch, a->n_layers, a->n_edge)) {
            set_error("BMP_MODE_BF16 RelGCN: needs one channel count in {64,128} for all layers, 4 bond types, N <= %d", BMP_MAX_ATOMS);
            return BMP_ESHAPE;
        }
        return bmp_relgcn_backward_tc(a, stream);
    }
    if (a && a->adj_u8) { set_error("bmp_relgcn_backward: a byte adjacency needs BMP_MODE_BF16"); return BMP_EINVAL; }
    // the tensor-core path (more than BMP_MAX_ATOMS atoms) keeps its temporaries in tc_workspace: Ds and Ps are not used there
    const bool x3 = a && a->mode == BMP_MODE_F32 && a->n_atoms > BMP_MAX_ATOMS;
    if (!a || !a->adj || !a->Hs || !a->d_h_out || (!x3 && (!a->Ds || !a->Ps))) {
        set_error("bmp_relgcn_backward: null argument");
        return BMP_EINVAL;
    }
    int cmax = 0;
    int rc = relgcn_check(a->mb, a->n_atoms, a->n_edge, a->n_layers, a->ch, &cmax, x3 ? BMP_X3_MAX_ATOMS : BMP_MAX_ATOMS);
    if (rc) return rc;
    const int L = a->n_layers, E = a->n_edge;
    for (int l = 0; l < L; ++l)
        if (!a->self_W[l] || !a->edge_W[l] || !aligned16({a->self_W[l], a->edge_W[l]})) {
            set_error("bmp_relgcn_backward: null or misaligned (16 B) weights at layer %d", l);
            return BMP_EINVAL;
        }
    if (!aligned16({a->Hs, a->d_h_out, a->Ds, a->Ps, a->d_h0})) { set_error("bmp_relgcn_backward: buffers must be 16-byte aligned"); return BMP_EINVAL; }
    if (x3) {
        const char *why = bmp_relgcn_x3_refusal(a->mb, a->n_atoms, a->n_edge, a->n_layers, a->ch, a->act, a->tc_workspace, a->tc_workspace_bytes);
        if (*why) { set_error("relgcn: %s", why); return BMP_ESHAPE; }
        return bmp_relgcn_backward_x3(a, stream);
    }
    size_t smem = sizeof(float) * ((size_t)2 * cmax * AT + AT * AT + AT + STAGE_FLOATS);
    int grid = a->mb < 148 ? a->mb : 148;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(HC)                                                                                           \
    do {                                                                                                     \
        cudaFuncSetAttribute(relgcn_bwd_kernel<HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        relgcn_bwd_kernel<HC><<<grid, NTHREADS, smem, st>>>(*a, cmax);                                       \
    } while (0)
    if (cmax <= 64) LAUNCH(1);
    else if (cmax <= 128) LAUNCH(2);
    else LAUNCH(4);
#undef LAUNCH
    count_launch();
    if ((rc = check_launch("relgcn_bwd_kernel"))) return rc;
    const long rows = (long)a->mb * a->n_atoms;
    long hs_off = 0, ds_off = 0, ps_off = 0;
    for (int l = 0; l < L; ++l) {
        const int Cin = a->ch[l], Cout = a->ch[l + 1];
        const float *Hl = a->Hs + hs_off, *Dl = a->Ds + ds_off, *Pl = a->Ps + ps_off;
        if (a->d_self_W[l] && (rc = bmp_wgrad(Dl, Cout, Hl, Cin, a->d_self_W[l], Cin, rows, Cout, Cin, stream))) return rc;
        if (a->d_self_b[l] && (rc = bmp_colsum(Dl, Cout, a->d_self_b[l], 1, rows, Cout, stream))) return rc;
        for (int e = 0; e < E; ++e) {
            if (a->d_edge_W[l] &&
                (rc = bmp_wgrad(Pl + (long)e * Cout, E * Cout, Hl, Cin, a->d_edge_W[l] + (long)e * Cin, E * Cin, rows, Cout, Cin, stream)))
                return rc;
            if (a->d_edge_b[l] && (rc = bmp_colsum(Pl + (long)e * Cout, E * Cout, a->d_edge_b[l] + e, E, rows, Cout, stream)))
                return rc;
        }
        hs_off += rows * Cin;
        ds_off += rows * Cout;
        ps_off += rows * E * Cout;
    }
    return BMP_OK;
}

// Bytes of det_scratch (deterministic mode, det.cuh) that bmp_relgcn_backward needs for this filled-in struct; 0 = no shape to cover.
extern "C" size_t bmp_relgcn_backward_det_bytes(const bmp_relgcn_bwd_t *a) {
    if (!a) return 0;
    if (a->mb <= 0 || a->n_atoms <= 0 || a->n_layers <= 0 || a->n_layers > BMP_MAX_STEPS) return 0;
    int c = 0;
    for (int l = 0; l <= a->n_layers; ++l) c = a->ch[l] > c ? a->ch[l] : c;
    if (c <= 0) return 0;
    c = c <= 64 ? 64 : (c <= 128 ? 128 : 256 > c ? 256 : c);     // the tensor-core row path pads every layer
    size_t n = det_max({det_wgrad_bytes(c, c), det_wgrad_tc_bytes(c, c), det_colsum_bytes(c)});
    return a->mode == BMP_MODE_BF16 ? det_max({n, det_panels_bytes()}) : n;
}
extern "C" int bmp_relgcn_backward(const bmp_relgcn_bwd_t *a, void *stream) {
    if (a && a->det_scratch) {
        int rc = det_check("bmp_relgcn_backward", a->det_scratch, a->det_scratch_bytes, bmp_relgcn_backward_det_bytes(a));
        if (rc) return rc;
    }
    DetScope ds(a ? a->det_scratch : nullptr, a ? a->det_scratch_bytes : 0);
    return relgcn_backward_impl(a, stream);
}
