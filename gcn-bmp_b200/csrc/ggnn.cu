// ggnn.cu -- fused GGNN encoder, fp32 mode (BMP_MODE_F32).
//
// Forward: one CTA owns one padded molecule for ALL T message-passing steps
// (embed -> T x [message, GRU gate]); hidden state, message and r*state stay in
// shared memory, weights stream from L2 through cp.async double-buffered tiles.
// Replaces models/models/ggnn.py:72-106 + models/update/ggnn_update.py:31-63 and the
// inlined copies models/ggnn_att.py:220-268,589-660, models/ggnn_dev.py:69-111.
//
// The message is re-associated as  m = sum_e (A_e h) W_e^T + deg_e b_e^T  with
// W_e = W_m[e::E] (the c*E+e interleave of ggnn_update.py:35-39 becomes a row
// stride), so the (mb,E,N,H) tensors of the reference never exist.
#include "common.cuh"

namespace bmp {

struct GgnnSmem {
    float *hs, *xs, *rs, *ss, *adj, *deg, *stage;
};

__device__ __forceinline__ GgnnSmem carve_fwd(float *base, int H, bool sep_state, int E) {
    GgnnSmem s;
    s.hs = base;                    // [H][64]
    s.xs = s.hs + H * AT;           // [H][64]   A_e h, then the message m  (must follow hs: K = 2H GEMMs)
    s.rs = s.xs + H * AT;           // [H][64]   r * state
    s.ss = sep_state ? s.rs + H * AT : s.hs;
    s.adj = (sep_state ? s.ss : s.rs) + H * AT;   // [64][64]
    s.deg = s.adj + AT * AT;        // [E][64]
    s.stage = s.deg + E * AT;
    return s;
}

static size_t fwd_smem_bytes(int H, bool sep_state, int E) {
    return sizeof(float) * ((size_t)(sep_state ? 4 : 3) * H * AT + AT * AT + E * AT + STAGE_FLOATS);
}

template <int HC>
__global__ void __launch_bounds__(NTHREADS, 1) ggnn_fwd_kernel(const bmp_ggnn_fwd_t a) {
    extern __shared__ __align__(16) float smem[];
    const int H = a.hidden, N = a.n_atoms, E = a.n_edge, T = a.n_steps;
    const int n_mol = a.mb;
    const bool sep_state = a.state_in != nullptr;
    GgnnSmem S = carve_fwd(smem, H, sep_state, E);
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int i0 = tx * 4;
    const long rows_total = (long)n_mol * N;
    const int K4 = (N + 3) & ~3;

    for (int mol = blockIdx.x; mol < n_mol; mol += gridDim.x) {
        const long row0 = (long)mol * N;
        __syncthreads();
        if (a.atoms) load_embed_cm(S.hs, a.atoms + row0, a.embed_W, N, H, a.n_atom_types);
        else load_cm(S.hs, a.h_in + row0 * H, N, H);
        if (sep_state) load_cm(S.ss, a.state_in + row0 * H, N, H);
        __syncthreads();
        if (a.Hs) store_cm(a.Hs + row0 * H, H, S.hs, N, H);
        if (a.h0_out) store_cm(a.h0_out + row0 * H, H, S.hs, N, H);

        for (int t = 0; t < T; ++t) {
            const bool stateful = a.stateful[t] != 0;
            const float *state = (t == 0 && sep_state) ? S.ss : S.hs;
            const bmp_gru_t &G = a.gru[t];
            // ---------------- message ----------------
            float accm[HC][4][4];
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) zero_acc(accm[oc]);
            for (int e = 0; e < E; ++e) {
                load_adj<true>(S.adj, a.adj + ((long)mol * E + e) * N * N, N);
                __syncthreads();
                if (tid < AT) {
                    float d = 0.f;
                    for (int j = 0; j < N; ++j) d += S.adj[j * AT + tid];
                    S.deg[e * AT + tid] = d;
                }
                // xs[c][i] = sum_j hs[c][j] * adjT[j][i]
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 < H) {
                        float acc[4][4];
                        zero_acc(acc);
                        if (oc * 64 + ty * 4 < H) gemm64_s(acc, S.hs, AT, oc * 64, K4, S.adj);
                        if (oc * 64 + ty * 4 < H) tile_store_s(S.xs, oc * 64, acc);
                    }
                }
                __syncthreads();
                // accm[c][i] += sum_c' W_e[c][c'] xs[c'][i]
#pragma unroll
                for (int oc = 0; oc < HC; ++oc)
                    if (oc * 64 < H)
                        gemm64_g<false>(accm[oc], a.msg_W[t] + (long)e * H, (long)E * H, oc * 64, H, H, S.xs, S.stage);
            }
            // bias rides through the adjacency: + sum_e b[c*E+e] * deg_e[i]
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                const int o0 = oc * 64 + ty * 4;
                if (o0 < H) {
                    for (int e = 0; e < E; ++e) {
                        float4 d = *reinterpret_cast<const float4 *>(S.deg + e * AT + i0);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            float bb = a.msg_b[t][(long)(o0 + q) * E + e];
                            accm[oc][q][0] += bb * d.x; accm[oc][q][1] += bb * d.y;
                            accm[oc][q][2] += bb * d.z; accm[oc][q][3] += bb * d.w;
                        }
                    }
                    tile_store_s(S.xs, oc * 64, accm[oc]);
                    if (a.Ms) tile_store_g(a.Ms + ((long)t * rows_total + row0) * H, H, oc * 64, H, N, accm[oc]);
                }
            }
            __syncthreads();
            // ---------------- reset gate ----------------
            if (stateful) {
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 >= H) continue;
                    float acc[4][4];
                    zero_acc(acc);
                    gemm64_g<false>(acc, G.W_r, 2 * H, oc * 64, H, 2 * H, S.hs, S.stage);
                    gemm64_g<false>(acc, G.U_r, H, oc * 64, H, H, state, S.stage);
                    const int o0 = oc * 64 + ty * 4;
                    if (o0 < H) {
                        float sv[4][4];
                        tile_load_s(state, oc * 64, sv);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            float bb = G.b_Wr[o0 + q] + G.b_Ur[o0 + q];
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                acc[q][b] = sigmoidf_(acc[q][b] + bb);
                                sv[q][b] *= acc[q][b];
                            }
                        }
                        tile_store_s(S.rs, oc * 64, sv);
                        if (a.Gs) tile_store_g(a.Gs + ((long)t * rows_total + row0) * 3 * H, 3 * H, oc * 64, H, N, acc);
                        if (a.RSs) tile_store_g(a.RSs + ((long)t * rows_total + row0) * H, H, oc * 64, H, N, sv);
                    }
                }
                __syncthreads();
            }
            // ---------------- update gate + candidate ----------------
            float hnew[HC][4][4];
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= H) continue;
                float az[4][4], ah[4][4];
                zero_acc(az);
                zero_acc(ah);
                gemm64_g<false>(az, G.W_z, 2 * H, oc * 64, H, 2 * H, S.hs, S.stage);
                gemm64_g<false>(ah, G.W, 2 * H, oc * 64, H, 2 * H, S.hs, S.stage);
                if (stateful) {
                    gemm64_g<false>(az, G.U_z, H, oc * 64, H, H, state, S.stage);
                    gemm64_g<false>(ah, G.U, H, oc * 64, H, H, S.rs, S.stage);
                }
                const int o0 = oc * 64 + ty * 4;
                if (o0 < H) {
                    float sv[4][4];
                    if (stateful) tile_load_s(state, oc * 64, sv);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float bz = G.b_Wz[o0 + q] + (stateful ? G.b_Uz[o0 + q] : 0.f);
                        float bh = G.b_W[o0 + q] + (stateful ? G.b_U[o0 + q] : 0.f);
#pragma unroll
                        for (int b = 0; b < 4; ++b) {
                            float z = sigmoidf_(az[q][b] + bz);
                            float hb = tanhf(ah[q][b] + bh);
                            az[q][b] = z;
                            ah[q][b] = hb;
                            hnew[oc][q][b] = stateful ? z * hb + (1.f - z) * sv[q][b] : z * hb;
                        }
                    }
                    if (a.Gs) {
                        float *g = a.Gs + ((long)t * rows_total + row0) * 3 * H;
                        if (!stateful) {   // r slot of a stateless step: zeros (keeps merged wgrad GEMMs exact)
                            float zr[4][4];
                            zero_acc(zr);
                            tile_store_g(g, 3 * H, oc * 64, H, N, zr);
                            if (a.RSs) tile_store_g(a.RSs + ((long)t * rows_total + row0) * H, H, oc * 64, H, N, zr);
                        }
                        tile_store_g(g + H, 3 * H, oc * 64, H, N, az);
                        tile_store_g(g + 2 * H, 3 * H, oc * 64, H, N, ah);
                    }
                }
            }
            __syncthreads();
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                const int o0 = oc * 64 + ty * 4;
                if (oc * 64 < H && o0 < H) {
                    tile_store_s(S.hs, oc * 64, hnew[oc]);
                    if (a.Hs) tile_store_g(a.Hs + ((long)(t + 1) * rows_total + row0) * H, H, oc * 64, H, N, hnew[oc]);
                    if (t == T - 1 && a.h_out) tile_store_g(a.h_out + row0 * H, H, oc * 64, H, N, hnew[oc]);
                }
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// Backward (data part).  One CTA per molecule walks the steps in reverse, reading
// the stash.  Writes the pre-activation gradients over Gs and A_e^T dm into Ps;
// parameter gradients are then plain  C += A^T B  contractions over all atoms
// (bmp_wgrad), issued by bmp_ggnn_backward below.
// ---------------------------------------------------------------------------
struct GgnnBwdSmem {
    float *g, *s, *dr, *dz, *dh, *adj, *stage;
};

static size_t bwd_smem_bytes(int H) {
    return sizeof(float) * ((size_t)5 * H * AT + AT * AT + STAGE_FLOATS);
}

template <int HC>
__global__ void __launch_bounds__(NTHREADS, 1) ggnn_bwd_kernel(const bmp_ggnn_bwd_t a) {
    extern __shared__ __align__(16) float smem[];
    const int H = a.hidden, N = a.n_atoms, E = a.n_edge, T = a.n_steps;
    GgnnBwdSmem S;
    S.g = smem;                 // running dL/dh_{t+1}
    S.s = S.g + H * AT;         // state of the step, later dm
    S.dr = S.s + H * AT;        // [dr | dz | dh] contiguous: Y operand of the K = 3H... (kept separate GEMMs)
    S.dz = S.dr + H * AT;
    S.dh = S.dz + H * AT;
    S.adj = S.dh + H * AT;
    S.stage = S.adj + AT * AT;
    const int tid = threadIdx.x;
    const int ty = tid >> 4;
    const long rows_total = (long)a.mb * N;
    const int K4 = (N + 3) & ~3;

    for (int mol = blockIdx.x; mol < a.mb; mol += gridDim.x) {
        const long row0 = (long)mol * N;
        __syncthreads();
        load_cm(S.g, a.dHs + ((long)T * rows_total + row0) * H, N, H);
        for (int t = T - 1; t >= 0; --t) {
            const bool stateful = a.stateful[t] != 0;
            const bool ext_state = (t == 0 && a.state_in != nullptr);
            const bmp_gru_t &G = a.gru[t];
            float *Gt = a.Gs + ((long)t * rows_total + row0) * 3 * H;
            if (stateful)
                load_cm(S.s, ext_state ? a.state_in + row0 * H : a.Hs + ((long)t * rows_total + row0) * H, N, H);
            __syncthreads();
            // ---- gate derivatives (thread-owned elements) ----
            float dsacc[HC][4][4];
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                zero_acc(dsacc[oc]);
                const int o0 = oc * 64 + ty * 4;
                if (oc * 64 >= H || o0 >= H) continue;
                float g[4][4], z[4][4], hb[4][4], sv[4][4];
                tile_load_s(S.g, oc * 64, g);
                tile_load_g(Gt + H, 3 * H, oc * 64, H, N, z);
                tile_load_g(Gt + 2 * H, 3 * H, oc * 64, H, N, hb);
                if (stateful) tile_load_s(S.s, oc * 64, sv);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        float s_ = stateful ? sv[q][b] : 0.f;
                        float dzv = g[q][b] * (hb[q][b] - s_);
                        float dhv = g[q][b] * z[q][b];
                        if (stateful) dsacc[oc][q][b] = g[q][b] * (1.f - z[q][b]);
                        hb[q][b] = dhv * (1.f - hb[q][b] * hb[q][b]);       // delta_h
                        z[q][b] = dzv * z[q][b] * (1.f - z[q][b]);          // delta_z
                    }
                tile_store_s(S.dz, oc * 64, z);
                tile_store_s(S.dh, oc * 64, hb);
                tile_store_g(Gt + H, 3 * H, oc * 64, H, N, z);
                tile_store_g(Gt + 2 * H, 3 * H, oc * 64, H, N, hb);
            }
            __syncthreads();
            // ---- through U and the reset gate ----
            if (stateful) {
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 >= H) continue;
                    float q_[4][4];
                    zero_acc(q_);
                    gemm64_g<true>(q_, G.U, H, oc * 64, H, H, S.dh, S.stage);   // q = U^T delta_h
                    const int o0 = oc * 64 + ty * 4;
                    if (o0 < H) {
                        float r[4][4], sv[4][4];
                        tile_load_g(Gt, 3 * H, oc * 64, H, N, r);
                        tile_load_s(S.s, oc * 64, sv);
#pragma unroll
                        for (int q = 0; q < 4; ++q)
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                float dr = q_[q][b] * sv[q][b];
                                dsacc[oc][q][b] += q_[q][b] * r[q][b];
                                r[q][b] = dr * r[q][b] * (1.f - r[q][b]);   // delta_r
                            }
                        tile_store_s(S.dr, oc * 64, r);
                        tile_store_g(Gt, 3 * H, oc * 64, H, N, r);
                    }
                }
                __syncthreads();
            }
            // ---- dx = [dh_x | dm], ds ----
            float dhx[HC][4][4];
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                zero_acc(dhx[oc]);
                if (oc * 64 >= H) continue;
                gemm64_g<true>(dhx[oc], G.W_z, 2 * H, oc * 64, H, H, S.dz, S.stage);
                gemm64_g<true>(dhx[oc], G.W, 2 * H, oc * 64, H, H, S.dh, S.stage);
                if (stateful) {
                    gemm64_g<true>(dhx[oc], G.W_r, 2 * H, oc * 64, H, H, S.dr, S.stage);
                    gemm64_g<true>(dsacc[oc], G.U_r, H, oc * 64, H, H, S.dr, S.stage);
                    gemm64_g<true>(dsacc[oc], G.U_z, H, oc * 64, H, H, S.dz, S.stage);
                }
            }
            // dm -> S.s (state no longer needed)
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= H) continue;
                float dm[4][4];
                zero_acc(dm);
                gemm64_g<true>(dm, G.W_z + H, 2 * H, oc * 64, H, H, S.dz, S.stage);
                gemm64_g<true>(dm, G.W + H, 2 * H, oc * 64, H, H, S.dh, S.stage);
                if (stateful) gemm64_g<true>(dm, G.W_r + H, 2 * H, oc * 64, H, H, S.dr, S.stage);
                if (oc * 64 + ty * 4 < H) tile_store_s(S.s, oc * 64, dm);
            }
            __syncthreads();
            // external state: its gradient leaves here; otherwise state == h_t and ds joins dh_t
            if (ext_state && stateful) {
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 < H && a.d_state_in)
                        tile_store_g(a.d_state_in + row0 * H, H, oc * 64, H, N, dsacc[oc]);
                }
            } else if (stateful) {
#pragma unroll
                for (int oc = 0; oc < HC; ++oc)
#pragma unroll
                    for (int q = 0; q < 4; ++q)
#pragma unroll
                        for (int b = 0; b < 4; ++b) dhx[oc][q][b] += dsacc[oc][q][b];
            }
            // ---- message backward: P_e = A_e^T dm ; dh += sum_e W_e^T P_e ----
            for (int e = 0; e < E; ++e) {
                load_adj<false>(S.adj, a.adj + ((long)mol * E + e) * N * N, N);
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 >= H) continue;
                    float p[4][4];
                    zero_acc(p);
                    if (oc * 64 + ty * 4 < H) {
                        gemm64_s(p, S.s, AT, oc * 64, K4, S.adj);   // P^T[c][j] = sum_i dm[c][i] A[i][j]
                        tile_store_s(S.dr, oc * 64, p);             // dr buffer is free now
                        tile_store_g(a.Ps + ((long)t * rows_total + row0) * E * H + (long)e * H, (long)E * H,
                                     oc * 64, H, N, p);
                    }
                }
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc)
                    if (oc * 64 < H)
                        gemm64_g<true>(dhx[oc], a.msg_W[t] + (long)e * H, (long)E * H, oc * 64, H, H, S.dr, S.stage);
            }
            // ---- dh_t = dhx + external dHs[t] -> running gradient ----
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= H || oc * 64 + ty * 4 >= H) continue;
                float ext[4][4];
                tile_load_g(a.dHs + ((long)t * rows_total + row0) * H, H, oc * 64, H, N, ext);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int b = 0; b < 4; ++b) dhx[oc][q][b] += ext[q][b];
                tile_store_s(S.g, oc * 64, dhx[oc]);
                if (t == 0) tile_store_g(a.dHs + row0 * H, H, oc * 64, H, N, dhx[oc]);
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------
// Backward (data part) for 128 < hidden <= 256.  The kernel above keeps five H x 64 fp32 buffers in shared memory (H <= 128);
// here only TWO are resident -- `y`, the pre-activation gradient currently used as a GEMM operand (delta_h, then delta_z,
// then delta_r, re-loaded from the Gs slots they were written to; later the P_e panels), and `s` (dm) -- the running
// gradient dL/dh_{t+1} lives in dHs[t+1] / dHs[t] in global memory, and every contribution to dL/dh_t is accumulated in
// one register tile set per 64-channel block.  Same arithmetic as ggnn_bwd_kernel, a slower schedule; the parity path for
// training at hidden 192 / 256.  state == step input only (no external GRU state).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void load_cm_ld(float *dst, const float *__restrict__ src, long ld, int n, int C) {
    const int nq = C >> 2;
    for (int idx = threadIdx.x; idx < nq * AT; idx += NTHREADS) {
        int i = idx & (AT - 1), cq = idx >> 6;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) v = *reinterpret_cast<const float4 *>(src + (long)i * ld + cq * 4);
        float *d = dst + (cq * 4) * AT + i;
        d[0] = v.x; d[AT] = v.y; d[2 * AT] = v.z; d[3 * AT] = v.w;
    }
}

static size_t bwd_big_smem_bytes(int H) {
    return sizeof(float) * ((size_t)2 * H * AT + AT * AT + STAGE_FLOATS);
}

template <int HC>
__global__ void __launch_bounds__(NTHREADS, 1) ggnn_bwd_big_kernel(const bmp_ggnn_bwd_t a) {
    extern __shared__ __align__(16) float smem[];
    const int H = a.hidden, N = a.n_atoms, E = a.n_edge, T = a.n_steps;
    float *Sy = smem, *Ss = Sy + H * AT, *Sadj = Ss + H * AT, *Sstage = Sadj + AT * AT;
    const int ty = threadIdx.x >> 4;
    const long rows_total = (long)a.mb * N;
    const int K4 = (N + 3) & ~3;

    for (int mol = blockIdx.x; mol < a.mb; mol += gridDim.x) {
        const long row0 = (long)mol * N;
        for (int t = T - 1; t >= 0; --t) {
            const bool stateful = a.stateful[t] != 0;
            const bmp_gru_t &G = a.gru[t];
            float *Gt = a.Gs + ((long)t * rows_total + row0) * 3 * H;
            const float *St = a.Hs + ((long)t * rows_total + row0) * H;                 // state of the step = h_t
            const float *gin = a.dHs + ((long)(t + 1) * rows_total + row0) * H;          // dL/dh_{t+1} (running gradient)
            float acc[HC][4][4], dm[HC][4][4];
            __syncthreads();
            // ---- gate derivatives (thread-owned elements): delta_z, delta_h -> Gs ; acc = g (1 - z)
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                zero_acc(acc[oc]);
                zero_acc(dm[oc]);
                if (oc * 64 + ty * 4 >= H) continue;
                float g[4][4], z[4][4], hb[4][4], sv[4][4];
                tile_load_g(gin, H, oc * 64, H, N, g);
                tile_load_g(Gt + H, 3 * H, oc * 64, H, N, z);
                tile_load_g(Gt + 2 * H, 3 * H, oc * 64, H, N, hb);
                if (stateful) tile_load_g(St, H, oc * 64, H, N, sv);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const float s_ = stateful ? sv[q][b] : 0.f;
                        const float dzv = g[q][b] * (hb[q][b] - s_);
                        const float dhv = g[q][b] * z[q][b];
                        if (stateful) acc[oc][q][b] = g[q][b] * (1.f - z[q][b]);
                        hb[q][b] = dhv * (1.f - hb[q][b] * hb[q][b]);       // delta_h
                        z[q][b] = dzv * z[q][b] * (1.f - z[q][b]);          // delta_z
                    }
                tile_store_g(Gt + H, 3 * H, oc * 64, H, N, z);
                tile_store_g(Gt + 2 * H, 3 * H, oc * 64, H, N, hb);
            }
            __syncthreads();
            // ---- operand delta_h: q = U^T delta_h -> delta_r, ds += q r ; dh_x += W_h^T delta_h ; dm += W_m^T delta_h
            load_cm_ld(Sy, Gt + 2 * H, 3 * H, N, H);
            __syncthreads();
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= H) continue;
                if (stateful) {
                    float q_[4][4];
                    zero_acc(q_);
                    gemm64_g<true>(q_, G.U, H, oc * 64, H, H, Sy, Sstage);
                    if (oc * 64 + ty * 4 < H) {
                        float r[4][4], sv[4][4];
                        tile_load_g(Gt, 3 * H, oc * 64, H, N, r);
                        tile_load_g(St, H, oc * 64, H, N, sv);
#pragma unroll
                        for (int q = 0; q < 4; ++q)
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                const float dr = q_[q][b] * sv[q][b];
                                acc[oc][q][b] += q_[q][b] * r[q][b];
                                r[q][b] = dr * r[q][b] * (1.f - r[q][b]);   // delta_r
                            }
                        tile_store_g(Gt, 3 * H, oc * 64, H, N, r);
                    }
                }
                gemm64_g<true>(acc[oc], G.W, 2 * H, oc * 64, H, H, Sy, Sstage);
                gemm64_g<true>(dm[oc], G.W + H, 2 * H, oc * 64, H, H, Sy, Sstage);
            }
            // ---- operand delta_z
            __syncthreads();
            load_cm_ld(Sy, Gt + H, 3 * H, N, H);
            __syncthreads();
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 >= H) continue;
                gemm64_g<true>(acc[oc], G.W_z, 2 * H, oc * 64, H, H, Sy, Sstage);
                gemm64_g<true>(dm[oc], G.W_z + H, 2 * H, oc * 64, H, H, Sy, Sstage);
                if (stateful) gemm64_g<true>(acc[oc], G.U_z, H, oc * 64, H, H, Sy, Sstage);
            }
            // ---- operand delta_r
            if (stateful) {
                __syncthreads();
                load_cm_ld(Sy, Gt, 3 * H, N, H);
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 >= H) continue;
                    gemm64_g<true>(acc[oc], G.W_r, 2 * H, oc * 64, H, H, Sy, Sstage);
                    gemm64_g<true>(dm[oc], G.W_r + H, 2 * H, oc * 64, H, H, Sy, Sstage);
                    gemm64_g<true>(acc[oc], G.U_r, H, oc * 64, H, H, Sy, Sstage);
                }
            }
            // ---- dm -> shared memory
            __syncthreads();
#pragma unroll
            for (int oc = 0; oc < HC; ++oc)
                if (oc * 64 + ty * 4 < H) tile_store_s(Ss, oc * 64, dm[oc]);
            __syncthreads();
            // ---- message backward: P_e = A_e^T dm ; dh += sum_e W_e^T P_e
            for (int e = 0; e < E; ++e) {
                load_adj<false>(Sadj, a.adj + ((long)mol * E + e) * N * N, N);
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc) {
                    if (oc * 64 + ty * 4 >= H) continue;
                    float p[4][4];
                    zero_acc(p);
                    gemm64_s(p, Ss, AT, oc * 64, K4, Sadj);       // P^T[c][j] = sum_i dm[c][i] A[i][j]
                    tile_store_s(Sy, oc * 64, p);
                    tile_store_g(a.Ps + ((long)t * rows_total + row0) * E * H + (long)e * H, (long)E * H, oc * 64, H, N, p);
                }
                __syncthreads();
#pragma unroll
                for (int oc = 0; oc < HC; ++oc)
                    if (oc * 64 < H)
                        gemm64_g<true>(acc[oc], a.msg_W[t] + (long)e * H, (long)E * H, oc * 64, H, H, Sy, Sstage);
            }
            // ---- dh_t = acc + external dHs[t] -> dHs[t] (the running gradient of the next iteration)
#pragma unroll
            for (int oc = 0; oc < HC; ++oc) {
                if (oc * 64 + ty * 4 >= H) continue;
                float ext[4][4];
                float *gout = a.dHs + ((long)t * rows_total + row0) * H;
                tile_load_g(gout, H, oc * 64, H, N, ext);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[oc][q][b] += ext[q][b];
                tile_store_g(gout, H, oc * 64, H, N, acc[oc]);
            }
            __syncthreads();
        }
    }
}

static int check_common(int mb, int N, int H, int E, int T, int mode, int nmax = BMP_MAX_ATOMS) {
    if (mode != BMP_MODE_F32) { set_error("ggnn fp32 path called with mode %d", mode); return BMP_EINVAL; }
    if (mb <= 0 || T <= 0 || T > BMP_MAX_STEPS) { set_error("ggnn: bad mb=%d or n_steps=%d", mb, T); return BMP_ESHAPE; }
    if (N <= 0 || N > nmax) {
        set_error("ggnn: n_atoms=%d outside 1..%d (more than %d atoms need BMP_MODE_F32 with the tensor-core workspace: hidden 64/128/256, "
                  "4 bond types)", N, nmax, BMP_MAX_ATOMS);
        return BMP_ESHAPE;
    }
    if (H <= 0 || H > BMP_MAX_HIDDEN || (H & 3)) { set_error("ggnn: hidden=%d must be a multiple of 4 in 4..%d", H, BMP_MAX_HIDDEN); return BMP_ESHAPE; }
    if (E <= 0 || E > 8) { set_error("ggnn: n_edge=%d outside 1..8", E); return BMP_ESHAPE; }
    return BMP_OK;
}

}  // namespace bmp

using namespace bmp;

int bmp_ggnn_forward_tc(const bmp_ggnn_fwd_t *a, void *stream);    // ggnn_tc.cu
int bmp_ggnn_backward_tc(const bmp_ggnn_bwd_t *a, void *stream);   // ggnn_tc_bwd.cu (bf16 panel stash)
// ggnn_x3.cu: BMP_MODE_F32 with the contractions on tcgen05 (bf16 hi/lo split, fp32-grade), when a workspace is given
bool bmp_ggnn_x3_usable(int mb, int N, int H, int E, int T, const void *ws, size_t ws_bytes, const void *state_in, bool inference);
int bmp_ggnn_forward_x3(const bmp_ggnn_fwd_t *a, void *stream);
int bmp_ggnn_backward_x3(const bmp_ggnn_bwd_t *a, void *stream);

extern "C" int bmp_ggnn_forward(const bmp_ggnn_fwd_t *a, void *stream) {
    if (!a || !a->adj || (!a->atoms && !a->h_in) || (a->atoms && !a->embed_W)) {
        set_error("bmp_ggnn_forward: null argument");
        return BMP_EINVAL;
    }
    if (a->mode == BMP_MODE_BF16) return bmp_ggnn_forward_tc(a, stream);
    if (a->mol_index) { set_error("bmp_ggnn_forward: mol_index (table indirection) is a BMP_MODE_BF16 feature; gather the rows first"); return BMP_ESHAPE; }
    if (a->adj_u8) { set_error("bmp_ggnn_forward: a byte adjacency needs BMP_MODE_BF16"); return BMP_EINVAL; }
    bool x3 = a->n_steps > 0 && a->n_steps <= BMP_MAX_STEPS &&
              bmp_ggnn_x3_usable(a->mb, a->n_atoms, a->hidden, a->n_edge, a->n_steps, a->tc_workspace, a->tc_workspace_bytes, a->state_in, a->Hs == nullptr);
    for (int t = 0; x3 && t < a->n_steps; ++t) {
        const bmp_gru_t &g = a->gru[t];
        x3 = aligned16({a->msg_b[t], g.b_Wr, g.b_Ur, g.b_Wz, g.b_Uz, g.b_W, g.b_U});
    }
    int rc = check_common(a->mb, a->n_atoms, a->hidden, a->n_edge, a->n_steps, a->mode, x3 ? BMP_X3_MAX_ATOMS : BMP_MAX_ATOMS);
    if (rc) return rc;
    for (int t = 0; t < a->n_steps; ++t) {
        const bmp_gru_t &g = a->gru[t];
        if (!a->msg_W[t] || !a->msg_b[t] || !g.W_z || !g.W) {
            set_error("bmp_ggnn_forward: null parameter at step %d", t);
            return BMP_EINVAL;
        }
        if (!aligned16({a->msg_W[t], g.W_r, g.U_r, g.W_z, g.U_z, g.W, g.U})) {
            set_error("bmp_ggnn_forward: weight matrices must be 16-byte aligned (step %d)", t);
            return BMP_EINVAL;
        }
    }
    if (!aligned16({a->h_in, a->embed_W, a->state_in, a->h_out, a->h0_out, a->Hs, a->Ms, a->Gs, a->RSs})) {
        set_error("bmp_ggnn_forward: activation buffers must be 16-byte aligned");
        return BMP_EINVAL;
    }
    const int H = a->hidden;
    if (x3) return bmp_ggnn_forward_x3(a, stream);
    const bool sep = a->state_in != nullptr;
    size_t smem = fwd_smem_bytes(H, sep, a->n_edge);
    if (smem > 227 * 1024) {
        set_error("bmp_ggnn_forward: hidden=%d with an external state needs %zu B of shared memory", H, smem);
        return BMP_ESHAPE;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int grid = a->mb < sms ? a->mb : sms;
    cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(HC)                                                                                         \
    do {                                                                                                   \
        cudaFuncSetAttribute(ggnn_fwd_kernel<HC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        ggnn_fwd_kernel<HC><<<grid, NTHREADS, smem, st>>>(*a);                                             \
    } while (0)
    if (H <= 64) LAUNCH(1);
    else if (H <= 128) LAUNCH(2);
    else LAUNCH(4);
#undef LAUNCH
    count_launch();
    return check_launch("ggnn_fwd_kernel");
}

extern "C" int bmp_ggnn_backward(const bmp_ggnn_bwd_t *a, void *stream) {
    if (a && (a->stash2 || a->mode == BMP_MODE_BF16)) {
        if (!a->stash2 || a->mode != BMP_MODE_BF16) {
            set_error("bmp_ggnn_backward: BMP_MODE_BF16 trains on the bf16 panel stash: stash2 (written by the forward) is required, "
                      "and only in that mode");
            return BMP_EINVAL;
        }
        if ((a->hidden != 64 && a->hidden != 128) || a->n_edge != 4 || a->state_in || !a->adj || !a->dHs) {
            set_error("bmp_ggnn_backward: the panel stash needs hidden 64/128, 4 bond types and no external state");
            return BMP_EINVAL;
        }
        return bmp_ggnn_backward_tc(a, stream);
    }
    if (!a || !a->adj || !a->Hs || !a->Ms || !a->Gs || !a->Ps || !a->dHs || !a->RSs) {
        set_error("bmp_ggnn_backward: null argument");
        return BMP_EINVAL;
    }
    const bool x3_data = a->mode == BMP_MODE_F32 && a->n_steps > 0 && a->n_steps <= BMP_MAX_STEPS &&
                         bmp_ggnn_x3_usable(a->mb, a->n_atoms, a->hidden, a->n_edge, a->n_steps, a->tc_workspace, a->tc_workspace_bytes, a->state_in, false);
    int rc = check_common(a->mb, a->n_atoms, a->hidden, a->n_edge, a->n_steps, BMP_MODE_F32, x3_data ? BMP_X3_MAX_ATOMS : BMP_MAX_ATOMS);
    if (rc) return rc;
    const int H = a->hidden, T = a->n_steps, E = a->n_edge;
    const bool tc3 = a->mode == BMP_MODE_F32 && (H == 64 || H == 128 || H == 256);
    auto WG = [&](const float *A_, int lda, const float *B_, int ldb, float *C_, int ldc, long r_, float *db, int dbs) -> int {
        // parameter-gradient contractions on tcgen05 with a bf16 hi/lo split (three UMMAs per product): fp32-grade accuracy
        if (tc3) return bmp_wgrad_tc3(A_, lda, B_, ldb, C_, ldc, r_, H, H, db, dbs, stream);
        int e_ = bmp_wgrad(A_, lda, B_, ldb, C_, ldc, r_, H, H, stream);
        if (!e_ && db) e_ = bmp_colsum(A_, lda, db, dbs, r_, H, stream);
        return e_;
    };
    if (a->adj_u8) { set_error("bmp_ggnn_backward: a byte adjacency needs BMP_MODE_BF16"); return BMP_EINVAL; }
    if (H > 128 && a->state_in) {
        set_error("bmp_ggnn_backward: an external GRU state needs hidden <= 128 (hidden=%d)", H);
        return BMP_ESHAPE;
    }
    for (int t = 0; t < T; ++t) {
        const bmp_gru_t &g = a->gru[t];
        if (!aligned16({a->msg_W[t], g.W_r, g.U_r, g.W_z, g.U_z, g.W, g.U})) {
            set_error("bmp_ggnn_backward: weight matrices must be 16-byte aligned (step %d)", t);
            return BMP_EINVAL;
        }
    }
    if (!aligned16({a->Hs, a->Ms, a->RSs, a->Gs, a->Ps, a->dHs, a->state_in, a->d_state_in})) {
        set_error("bmp_ggnn_backward: stash buffers must be 16-byte aligned");
        return BMP_EINVAL;
    }
    if (x3_data) {
        if ((rc = bmp_ggnn_backward_x3(a, stream))) return rc;
    } else {
        size_t smem = bwd_smem_bytes(H);
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        int grid = a->mb < sms ? a->mb : sms;
        cudaStream_t st = (cudaStream_t)stream;
        if (H > 128) {
            smem = bwd_big_smem_bytes(H);
            if (H <= 192) {
                cudaFuncSetAttribute(ggnn_bwd_big_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                ggnn_bwd_big_kernel<3><<<grid, NTHREADS, smem, st>>>(*a);
            } else {
                cudaFuncSetAttribute(ggnn_bwd_big_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                ggnn_bwd_big_kernel<4><<<grid, NTHREADS, smem, st>>>(*a);
            }
        } else if (H <= 64) {
            cudaFuncSetAttribute(ggnn_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            ggnn_bwd_kernel<1><<<grid, NTHREADS, smem, st>>>(*a);
        } else {
            cudaFuncSetAttribute(ggnn_bwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            ggnn_bwd_kernel<2><<<grid, NTHREADS, smem, st>>>(*a);
        }
        count_launch();
        rc = check_launch("ggnn_bwd_kernel");
        if (rc) return rc;
    }

    // ---- parameter gradients: C += A^T B over all atoms of the batch ----
    // Consecutive steps that share parameter pointers are contiguous in every stash,
    // so they collapse into one contraction with rows = (#steps) * mb * N.
    const long rows = (long)a->mb * a->n_atoms;
    int t0 = 0;
    while (t0 < T) {
        int t1 = t0;
        while (t1 + 1 < T && a->d_msg_W[t1 + 1] == a->d_msg_W[t0] && a->d_gru[t1 + 1].W == a->d_gru[t0].W &&
               a->d_gru[t1 + 1].U == a->d_gru[t0].U)
            ++t1;
        const long r = (long)(t1 - t0 + 1) * rows;
        const float *Gs = a->Gs + (long)t0 * rows * 3 * H;
        const float *Hs = a->Hs + (long)t0 * rows * H;
        const float *Ms = a->Ms + (long)t0 * rows * H;
        const float *Ps = a->Ps + (long)t0 * rows * E * H;
        const bmp_gru_grad_t &D = a->d_gru[t0];
        // step 0 with an external state feeds h_in, not the state, to W_*: Hs[0] is h_in in both cases.
        float *Wg[3] = {D.W_r, D.W_z, D.W};
        float *bg[3] = {D.b_Wr, D.b_Wz, D.b_W};
        for (int k = 0; k < 3; ++k) {
            if (!Wg[k]) continue;
            if ((rc = WG(Gs + k * H, 3 * H, Hs, H, Wg[k], 2 * H, r, bg[k], 1))) return rc;
            if ((rc = WG(Gs + k * H, 3 * H, Ms, H, Wg[k] + H, 2 * H, r, nullptr, 1))) return rc;
        }
        if (a->d_msg_W[t0]) {
            // dW_m[c*E+e][c'] += sum_rows P[row][e*H+c] * h[row][c']  (row stride E*H in dW_m -> ldc);
            // db_m[c*E+e] += column sums of P_e, scattered with stride E
            for (int e = 0; e < E; ++e)
                if ((rc = WG(Ps + e * H, E * H, Hs, H, a->d_msg_W[t0] + (long)e * H, E * H, r,
                             a->d_msg_b[t0] ? a->d_msg_b[t0] + e : nullptr, E)))
                    return rc;
        }
        // U-type gradients only over stateful steps
        int s0 = t0;
        while (s0 <= t1) {
            if (!a->stateful[s0]) { ++s0; continue; }
            int s1 = s0;
            const bool ext = (s0 == 0 && a->state_in);   // state of step 0 lives outside the stash
            while (!ext && s1 + 1 <= t1 && a->stateful[s1 + 1]) ++s1;
            const float *Gss = a->Gs + (long)s0 * rows * 3 * H;
            const float *St = ext ? a->state_in : a->Hs + (long)s0 * rows * H;
            const float *RS = a->RSs + (long)s0 * rows * H;
            const long rs2 = (long)(s1 - s0 + 1) * rows;
            if (D.U_r && (rc = WG(Gss, 3 * H, St, H, D.U_r, H, rs2, D.b_Ur, 1))) return rc;
            if (D.U_z && (rc = WG(Gss + H, 3 * H, St, H, D.U_z, H, rs2, D.b_Uz, 1))) return rc;
            if (D.U && (rc = WG(Gss + 2 * H, 3 * H, RS, H, D.U, H, rs2, D.b_U, 1))) return rc;
            s0 = s1 + 1;
        }
        t0 = t1 + 1;
    }
    return BMP_OK;
}
