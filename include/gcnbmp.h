/* gcnbmp.h -- C-ABI of the B200-native GCN-BMP message-passing hot path.
 *
 * The reference (Minys233/GCN-BMP) has no FFI layer: its hot path sits behind
 * Chainer `Link.__call__` and every FLOP runs inside Chainer/CuPy.  This header
 * is the boundary a maintainer binds with ctypes (see INTEGRATION.md): plain
 * device pointers (CuPy `arr.data.ptr`, Torch `t.data_ptr()`), sizes and a
 * caller-supplied `cudaStream_t` (passed as void*).  All entry points are
 * asynchronous on that stream, never allocate, never synchronise, and return an
 * int status (0 = ok).  `bmp_last_error()` is thread-local.
 *
 * Layouts are the reference's: atoms int32 (mb, N), 0 = padding (still embedded);
 * adj fp32 (mb, E, N, N); atom features fp32 (mb, N, H) row-major; `Linear.W`
 * is (out, in); the message GraphLinear's W is (E*H, H) with row index c*E+e
 * (channel-major / edge-minor, models/update/ggnn_update.py:35-39).
 *
 * Each entry point cites the reference code it replaces (paths relative to the
 * reference repository root).
 */
#ifndef GCNBMP_H_
#define GCNBMP_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMP_OK       0
#define BMP_EINVAL  -1   /* null pointer / bad enum                       */
#define BMP_ESHAPE  -2   /* shape outside what the kernels are built for  */
#define BMP_EARCH   -3   /* device is not sm_100                          */
#define BMP_ECUDA   -4   /* a CUDA runtime call failed                    */

#define BMP_MAX_STEPS   16
#define BMP_MAX_ATOMS   64   /* padded atoms per molecule handled by one CTA */
#define BMP_X3_MAX_ATOMS 256 /* GGNN and RelGCN encoders in BMP_MODE_F32 with the tensor-core workspace (bmp_ggnn_x3_workspace_bytes,
                               bmp_relgcn_x3_workspace_bytes): their row GEMMs never see molecule boundaries; n_atoms * hidden * 4
                               bytes <= 160 KB.  Also the limit of bmp_rescale_adj, bmp_gin_aggregate and bmp_nfp_gather */
#define BMP_MAX_HIDDEN 256

/* activations (chainer.functions.{identity,tanh,relu,sigmoid}) */
enum { BMP_ACT_IDENTITY = 0, BMP_ACT_TANH = 1, BMP_ACT_RELU = 2, BMP_ACT_SIGMOID = 3 };
/* readout variants: R1 = models/readout/ggnn_readout.py:42-58 (i and j see [h|h0]);
 * R2 = models/ggnn_att.py:338-346 (j sees h only); SUM = models/ggnn_dev.py:167 */
enum { BMP_READOUT_R1 = 1, BMP_READOUT_R2 = 2, BMP_READOUT_SUM = 3 };
/* co-attention variants: NIE/VQA = nie_coattention.py:312-396 /
 * vqa_parallel_coattention.py:13-103 (same math); POOL = PoolingFineCoattention.py:13-83 */
enum { BMP_COATTN_FINE = 0, BMP_COATTN_POOL = 1 };
/* arithmetic mode of the encoder kernels */
enum { BMP_MODE_F32 = 0,    /* fp32 FFMA everywhere: parity <= 1e-4 vs the oracle */
       BMP_MODE_BF16 = 1 }; /* tcgen05 bf16 operands, fp32 accumulate/state       */

/* One chainer links.GRU (= StatefulGRU): six Linear sub-links, W (out,in). */
typedef struct {
    const float *W_r, *b_Wr, *U_r, *b_Ur;   /* (H,2H),(H),(H,H),(H) */
    const float *W_z, *b_Wz, *U_z, *b_Uz;
    const float *W,   *b_W,  *U,   *b_U;
} bmp_gru_t;

typedef struct {                             /* gradients, same shapes; accumulated (+=) */
    float *W_r, *b_Wr, *U_r, *b_Ur;
    float *W_z, *b_Wz, *U_z, *b_Uz;
    float *W,   *b_W,  *U,   *b_U;
} bmp_gru_grad_t;

/* ---- GGNN encoder: embed -> T x GGNNUpdate --------------------------------
 * replaces models/models/ggnn.py:72-106 (loop), models/update/ggnn_update.py:31-63
 * (one step), models/ggnn_att.py:220-268,589-660, models/ggnn_dev.py:69-111,135-168.
 * Step t uses msg_W[t]/msg_b[t] and gru[t]; `stateful[t]` != 0 means the GRU has a
 * state at that call (the StatefulGRU "h is not None" branch); the state is
 * `state_in` for t == 0 and the step's own input h for t > 0 (which is what every
 * reference GGNN feeds it).  Tied weights = the same pointers at every t.
 * Stash buffers (needed by the BMP_MODE_F32 bmp_ggnn_backward, NULL for inference):
 *   Hs (T+1, mb*N, H)  h_0 .. h_T           Ms (T, mb*N, H)   messages
 *   Gs (T, mb*N, 3H)   r | z | h_bar        RSs (T, mb*N, H)  r*state
 * BMP_MODE_BF16 trains on stash2 instead: Ms / Gs / RSs must be NULL there, and Hs
 * (only with stash2) receives h_0 .. h_T as an output the backward does not read.   */
typedef struct {
    int mb, n_atoms, hidden, n_edge, n_steps, n_atom_types, mode;
    const int32_t *atoms;        /* (mb,N) or NULL when h_in is given              */
    const float   *h_in;         /* (mb,N,H) or NULL                                */
    const float   *embed_W;      /* (n_atom_types,H); used when atoms != NULL       */
    const float   *adj;          /* (mb,E,N,N)                                      */
    const float   *state_in;     /* (mb,N,H) or NULL (= after reset_state)          */
    const float   *msg_W[BMP_MAX_STEPS];   /* (E*H,H) */
    const float   *msg_b[BMP_MAX_STEPS];   /* (E*H)   */
    bmp_gru_t      gru[BMP_MAX_STEPS];
    int            stateful[BMP_MAX_STEPS];
    float *h_out;                /* (mb,N,H) final atom states (get_atom_array)     */
    float *h0_out;               /* (mb,N,H) copy of h_0 for the readout, or NULL   */
    float *Hs, *Ms, *Gs, *RSs;   /* stash or NULL (BMP_MODE_BF16: Hs only, see above) */
    void  *tc_workspace;         /* BMP_MODE_BF16 only: packed bf16 weight tiles    */
    size_t tc_workspace_bytes;   /* >= bmp_ggnn_tc_workspace_bytes(hidden, n_steps) */
    void  *stash2;               /* BMP_MODE_BF16 training: bf16 panel stash of      */
                                 /* bmp_ggnn_stash2_bytes() bytes, the only tape     */
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
    int    adj_u8;               /* BMP_MODE_BF16 only, storage of `adj`: 0 = fp32 (mb,E,N,N) as the reference; 1 = the same
                                   array as bytes (exact for 0/1 bonds; 1/4 of the PCIe / HBM traffic); 2 = bit-packed rows
                                   (mb,E,N,ceil(N/8)), bit j&7 of byte j>>3 = adj[i][j] (numpy.packbits little; 1/32)  */
    const int32_t *mol_index;    /* BMP_MODE_BF16 only, or NULL.  (mb,) int32: `atoms` (U,N) and `adj` (U,E,N,N) are a device-resident
                                   drug TABLE and molecule b of this call is its row mol_index[b] (train_binary.py:285-294 builds the
                                   per-pair copies this replaces); read inside the kernels, no gather copy              */
} bmp_ggnn_fwd_t;

int bmp_ggnn_forward(const bmp_ggnn_fwd_t *a, void *stream);
/* Bytes of device workspace the BMP_MODE_BF16 (tcgen05) encoder needs; 0 = shape unsupported. */
size_t bmp_ggnn_tc_workspace_bytes(int hidden, int n_steps);
/* BMP_MODE_F32 on the tensor cores (csrc/ggnn_x3.cu): when tc_workspace / tc_workspace_bytes of a BMP_MODE_F32 call hold at
 * least this many bytes (and state_in is NULL), every H x H contraction of the encoder runs on tcgen05 with a bf16 hi/lo
 * operand split -- three UMMAs per product, fp32 accumulate: the <= 1e-4 parity of the mode is kept -- instead of the FFMA
 * kernels; same stash, same results up to fp32 rounding order.  `inference` != 0: the call passes no stash (adds a one-step
 * stash to the workspace).  The backward must be given a workspace sized with inference = 0; dHs[t] is then updated in
 * place for every t (the FFMA path only writes dHs[0]).  0 = shape not covered (hidden 64/128/256, 4 bond types).          */
size_t bmp_ggnn_x3_workspace_bytes(int mb, int n_atoms, int hidden, int n_edge, int n_steps, int inference);
/* Bytes of the bf16 panel stash (forward operand panels + gate values + backward delta/P panels). */
size_t bmp_ggnn_stash2_bytes(int mb, int hidden, int n_steps);

/* Backward of the above (Chainer autograd through the same lines).
 * dHs (T+1, mb*N, H): on entry the external gradient w.r.t. every h_t (zero where
 * none; dHs[T] = grad of h_out, dHs[0] += grad of h0 from the readout); on exit
 * dHs[0] holds the total gradient w.r.t. h_0 (feed it to bmp_embed_backward or
 * return it as d h_in).  Gs is overwritten with dr|dz|dh_bar pre-activation
 * gradients, Ps (T, mb*N, E*H) receives A_e^T dm.  Parameter gradients are
 * accumulated (+=) into the per-step pointers (tied = same pointers).
 * d_state_in (mb,N,H) or NULL.                                                  */
typedef struct {
    int mb, n_atoms, hidden, n_edge, n_steps, mode;
    const float *adj, *state_in;
    const float *msg_W[BMP_MAX_STEPS];
    bmp_gru_t    gru[BMP_MAX_STEPS];
    int          stateful[BMP_MAX_STEPS];
    const float *Hs, *Ms, *RSs;
    float *Gs, *Ps, *dHs;
    float *d_msg_W[BMP_MAX_STEPS], *d_msg_b[BMP_MAX_STEPS];
    bmp_gru_grad_t d_gru[BMP_MAX_STEPS];
    float *d_state_in;
    void  *tc_workspace;         /* BMP_MODE_BF16 only (same size rule as the forward) */
    size_t tc_workspace_bytes;
    void  *stash2;               /* BMP_MODE_BF16: the forward's panel stash (required there); Hs/Ms/RSs/Gs/Ps are
                                    unused and dHs is laid out as dHs_every_step says                          */
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
    int    adj_u8;               /* BMP_MODE_BF16 only, storage of `adj`: 0 = fp32 (mb,E,N,N) as the reference; 1 = the same
                                   array as bytes (exact for 0/1 bonds; 1/4 of the PCIe / HBM traffic); 2 = bit-packed rows
                                   (mb,E,N,ceil(N/8)), bit j&7 of byte j>>3 = adj[i][j] (numpy.packbits little; 1/32)  */
    const int32_t *mol_index;    /* the forward's mol_index: adjacency table rows, or NULL                          */
    int    dHs_every_step;       /* BMP_MODE_BF16 only.  0: dHs has TWO slices, [0] = gradient w.r.t. h_0, [1] = gradient
                                    w.r.t. h_T.  Nonzero: dHs (T+1, mb*N, H) as in BMP_MODE_F32, an external gradient for
                                    every h_t.  Either way dHs[0] holds the total gradient w.r.t. h_0 on exit    */
} bmp_ggnn_bwd_t;

int bmp_ggnn_backward(const bmp_ggnn_bwd_t *a, void *stream);

/* EmbedAtomID (models/models/ggnn.py:55,89-92): forward gather is fused into the
 * encoders; this is its backward: d_embed_W[atoms[r], :] += dh[r, :].            */
int bmp_embed_backward(const int32_t *atoms, const float *dh, float *d_embed_W,
                       int rows, int hidden, int n_atom_types, void *stream);

/* ---- RelGCN encoder: embed -> [rescale_adj] -> L x tanh(RelGCNUpdate) ------
 * replaces models/relgcn.py:61-73, :20-28 and models/update/relgcn_update.py:24-44.
 * ch[0..L] are the channel sizes.  Hs stash: concatenation over l = 0..L of
 * (mb*N, ch[l]) activations (h_0 = embedding, h_l = tanh(conv_l)).  `scale_adj`
 * applies the column-degree normalisation inside the kernel.                     */
typedef struct {
    int mb, n_atoms, n_edge, n_layers, n_atom_types, scale_adj;
    int act;               /* per-layer activation: BMP_ACT_TANH (RelGCN) or BMP_ACT_IDENTITY (bare RelGCNUpdate) */
    int ch[BMP_MAX_STEPS + 1];
    const int32_t *atoms;  const float *h_in;  const float *embed_W;
    const float *adj;
    const float *self_W[BMP_MAX_STEPS], *self_b[BMP_MAX_STEPS];   /* (Cout,Cin),(Cout)     */
    const float *edge_W[BMP_MAX_STEPS], *edge_b[BMP_MAX_STEPS];   /* (Cout*E,Cin),(Cout*E) */
    float *h_out;      /* (mb,N,ch[L]) */
    float *Hs;         /* stash or NULL */
    /* BMP_MODE_BF16 (tcgen05): every ch[l] equal and in {64,128}, n_edge = 4; stash2 (bmp_ggnn_stash2_bytes(mb, ch[0],
     * n_layers) bytes, or NULL for inference) replaces Hs. */
    int    mode;
    void  *tc_workspace;         /* >= bmp_relgcn_tc_workspace_bytes(ch[0], n_layers) */
    size_t tc_workspace_bytes;
    void  *stash2;
    int    tc_images_ready;      /* as in bmp_ggnn_fwd_t */
    int    adj_u8;               /* BMP_MODE_BF16 only, storage of `adj`: 0 = fp32 (mb,E,N,N) as the reference; 1 = the same
                                   array as bytes (exact for 0/1 bonds; 1/4 of the PCIe / HBM traffic); 2 = bit-packed rows
                                   (mb,E,N,ceil(N/8)), bit j&7 of byte j>>3 = adj[i][j] (numpy.packbits little; 1/32)  */
} bmp_relgcn_fwd_t;

int bmp_relgcn_forward(const bmp_relgcn_fwd_t *a, void *stream);
size_t bmp_relgcn_tc_workspace_bytes(int channels, int n_layers);   /* 0 = channel count not on the tcgen05 path */
/* BMP_MODE_F32 with 65 <= n_atoms <= BMP_X3_MAX_ATOMS (csrc/ggnn_x3.cu): bmp_relgcn_forward / bmp_relgcn_backward take the
 * tensor-core row path -- per layer one adjacency product over bit masks and one split-bf16 GEMM (three UMMAs per product, fp32
 * accumulate: the <= 1e-4 parity of the mode is kept) -- when tc_workspace / tc_workspace_bytes hold at least this many bytes.
 * ch_max = the largest ch[l]: every layer runs zero-padded to it rounded up to 64, 128 or 256, which with n_atoms must satisfy
 * n_atoms * padded channels * 4 bytes <= 160 KB; n_edge must be 4 and act identity or tanh.  Same Hs stash as the FFMA kernels;
 * the backward takes a workspace of the same size (its contents need not be the forward's) and leaves Ds / Ps unused (they may
 * be NULL).  Host-only; the size does not depend on `inference`.  0 = shape not covered (the FFMA kernels take n_atoms <= 64). */
size_t bmp_relgcn_x3_workspace_bytes(int mb, int n_atoms, int ch_max, int n_layers, int inference);
/* adj_out[b,e,i,j] = adj[b,e,i,j] / (sum_{e',i'} adj[b,e',i',j] or 1)   (rescale_adj, models/relgcn.py:20-28) */
int bmp_rescale_adj(const float *adj, float *adj_out, int mb, int n_edge, int n_atoms, void *stream);

/* Ds: workspace, concatenation over l of (mb*N, ch[l+1]) pre-tanh gradients;
 * Ps: workspace, concatenation over l of (mb*N, E*ch[l+1]) (A_e^T delta);
 * d_h0 (mb*N, ch[0]) receives the gradient w.r.t. h_0.                           */
typedef struct {
    int mb, n_atoms, n_edge, n_layers, scale_adj, act;
    int ch[BMP_MAX_STEPS + 1];
    const float *adj;
    const float *self_W[BMP_MAX_STEPS], *edge_W[BMP_MAX_STEPS];
    const float *Hs;
    const float *d_h_out;   /* (mb,N,ch[L]) */
    float *Ds, *Ps, *d_h0;
    float *d_self_W[BMP_MAX_STEPS], *d_self_b[BMP_MAX_STEPS];
    float *d_edge_W[BMP_MAX_STEPS], *d_edge_b[BMP_MAX_STEPS];
    /* BMP_MODE_BF16: stash2 written by the forward (Hs, Ds, Ps unused), adj = the adjacency the forward saw */
    int    mode;
    void  *tc_workspace;
    size_t tc_workspace_bytes;
    void  *stash2;
    int    tc_images_ready;
    int    adj_u8;               /* BMP_MODE_BF16 only, storage of `adj`: 0 = fp32 (mb,E,N,N) as the reference; 1 = the same
                                   array as bytes (exact for 0/1 bonds; 1/4 of the PCIe / HBM traffic); 2 = bit-packed rows
                                   (mb,E,N,ceil(N/8)), bit j&7 of byte j>>3 = adj[i][j] (numpy.packbits little; 1/32)  */
} bmp_relgcn_bwd_t;

int bmp_relgcn_backward(const bmp_relgcn_bwd_t *a, void *stream);

/* ---- gated readout ---------------------------------------------------------
 * replaces models/readout/ggnn_readout.py:42-58 (R1), models/ggnn_att.py:338-346
 * (R2), models/ggnn_dev.py:167 (SUM).  h0 may be NULL (R1 on h alone, relgcn.py:72).
 * is_real_node (mb,N) fp32 or NULL.  W_i (O, Kin), W_j (O, Kin or H); b may be NULL. */
typedef struct {
    int mb, n_atoms, hidden, out_dim, variant, act, act_agg;
    const float *h, *h0, *is_real_node;
    const float *W_i, *b_i, *W_j, *b_j;
    float *g;                          /* (mb,O) ; (mb,H) for SUM */
    int    mode;                       /* BMP_MODE_BF16: tcgen05 kernel when H,O in {64,128} (else fp32 kernel) */
    void  *tc_workspace;               /* >= bmp_readout_tc_workspace_bytes(hidden, out_dim) in BF16 mode      */
    size_t tc_workspace_bytes;
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
} bmp_readout_fwd_t;

int bmp_readout_forward(const bmp_readout_fwd_t *a, void *stream);
size_t bmp_readout_tc_workspace_bytes(int hidden, int out_dim);   /* 0 = shape not on the tcgen05 path */
/* BMP_MODE_F32 forward on the tensor cores (both linears as split-bf16 row GEMMs, csrc/ggnn_x3.cu): taken when tc_workspace holds at
 * least this many bytes; hidden and out_dim in {64,128,256}, variants R1 / R2, mb * n_atoms >= 128; 0 = not covered (FFMA kernel).  */
size_t bmp_readout_x3_workspace_bytes(int mb, int n_atoms, int hidden, int out_dim, int variant, int has_h0);

/* DU/DV: workspaces (mb*N, O) receiving the pre-activation gradients of the i and
 * j linears; dh/dh0 are ACCUMULATED (+=) so they can point into bmp_ggnn dHs.     */
typedef struct {
    int mb, n_atoms, hidden, out_dim, variant, act, act_agg;
    const float *h, *h0, *is_real_node;
    const float *W_i, *b_i, *W_j, *b_j;
    const float *g, *dg;
    float *DU, *DV, *dh, *dh0;
    float *d_W_i, *d_b_i, *d_W_j, *d_b_j;
    int    mode;
    void  *tc_workspace;
    size_t tc_workspace_bytes;
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
} bmp_readout_bwd_t;

int bmp_readout_backward(const bmp_readout_bwd_t *a, void *stream);

/* ---- fine-grained co-attention ---------------------------------------------
 * replaces models/coattention/nie_coattention.py:335-396,
 * vqa_parallel_coattention.py:42-103 (variant FINE) and
 * PoolingFineCoattention.py:31-83 (variant POOL).  The tile-materialised
 * (mb*N2*N1, H) bilinear operands of the reference never exist here.
 * W (H,H) [= Bilinear.W[:,:,0]], V1 (H), V2 (H), b (1), lt_k (head,H), wa_k (head),
 * W_j (O,H), b_j (O).                                                            */
typedef struct {
    int mb, n1, n2, hidden, out_dim, head, variant, act;
    const float *atoms_1, *atoms_2;    /* (mb,N1,H), (mb,N2,H) */
    const float *W, *V1, *V2, *b, *lt_1, *lt_2, *wa_1, *wa_2, *W_j, *b_j;
    float *compact_1, *compact_2;      /* (mb,O) */
    int    mode;                       /* BMP_MODE_BF16: contractions on tcgen05 (FINE variant, hidden 64/128, head <= 15) */
    void  *tc_workspace;               /* BMP_MODE_BF16: >= bmp_coattn_tc_workspace_bytes(hidden) bytes, 16-byte aligned */
    size_t tc_workspace_bytes;
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
} bmp_coattn_fwd_t;

int bmp_coattn_forward(const bmp_coattn_fwd_t *a, void *stream);

/* R (mb*N1, H), P1/P2 (mb, H) and DL1/DL2 (mb*N1 / mb*N2, head) are workspaces the
 * parameter-gradient GEMMs read (the tcgen05 kernel leaves R and DL untouched: it contracts
 * d W, d lt_k and d V_k on chip).  d_atoms_k are OVERWRITTEN (every live element is written);
 * parameter gradients d_* are ACCUMULATED (+=).                                           */
typedef struct {
    int mb, n1, n2, hidden, out_dim, head, variant, act;
    const float *atoms_1, *atoms_2;
    const float *W, *V1, *V2, *b, *lt_1, *lt_2, *wa_1, *wa_2, *W_j, *b_j;
    const float *d_compact_1, *d_compact_2;
    float *R, *P1, *P2, *DL1, *DL2;
    float *d_atoms_1, *d_atoms_2;
    float *d_W, *d_V1, *d_V2, *d_b, *d_lt_1, *d_lt_2, *d_wa_1, *d_wa_2, *d_W_j, *d_b_j;
    int    mode;   /* BMP_MODE_BF16: data contractions and the (H,H) / (O,H) weight gradients run on tcgen05 */
    void  *tc_workspace;
    size_t tc_workspace_bytes;
    int    tc_images_ready;      /* nonzero: tc_workspace already holds the images packed by an earlier call of the same
                                   kind with exactly these parameter values -- skip packing             */
} bmp_coattn_bwd_t;

int bmp_coattn_backward(const bmp_coattn_bwd_t *a, void *stream);
/* packed bf16 weight images of the tcgen05 co-attention kernels; 0 when hidden is not 64 or 128 */
size_t bmp_coattn_tc_workspace_bytes(int hidden);

/* ---- HolE circular correlation ----------------------------------------------
 * replaces models/link_prediction/hole.py:28-50 (= models/mlp.py:128-151):
 * c[b,k] = sum_i l[b,i] r[b,(i+k) mod D], computed directly (no FFT).            */
int bmp_hole_corr_forward(const float *left, const float *right, float *out,
                          int mb, int dim, void *stream);
int bmp_hole_corr_backward(const float *left, const float *right, const float *d_out,
                           float *d_left, float *d_right, int mb, int dim, void *stream);

/* ---- dense layers of the heads (links.Linear; hole.py:21-26) ----------------
 * y = act(x W^T + b); W (out,in), b NULL allowed.                                */
int bmp_linear_forward(const float *x, const float *W, const float *b, float *y,
                       int rows, int in_dim, int out_dim, int act, void *stream);
/* dy is overwritten with the pre-activation gradient; dx (=), dW/db (+=). dx may be NULL. */
int bmp_linear_backward(const float *x, const float *W, const float *y, float *dy,
                        float *dx, float *dW, float *db,
                        int rows, int in_dim, int out_dim, int act, void *stream);

/* C (M,N) += A^T B with A (rows,M; lda), B (rows,N; ldb): the parameter-gradient
 * contraction over all atoms of a batch (split over CTAs, fp32 atomics at the end). */
int bmp_wgrad(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
              int64_t rows, int M, int N, void *stream);
/* Same contraction on tcgen05 (bf16 operands, fp32 accumulate; used by BMP_MODE_BF16): N in {64,128,256},
 * 16-byte aligned operands, else BMP_ESHAPE.  dbias[m*bias_stride] += column sums of A when non-NULL. */
int bmp_wgrad_tc(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                 int64_t rows, int M, int N, float *dbias, int bias_stride, void *stream);
/* The same contraction at fp32-grade accuracy on the tensor cores: bf16 hi/lo split of both operands, three UMMAs per product,
 * fp32 TMEM accumulate (relative error ~1e-5); what BMP_MODE_F32 uses for the GGNN parameter gradients at hidden 64/128/256.   */
int bmp_wgrad_tc3(const float *A, int lda, const float *B, int ldb, float *C, int ldc,
                 int64_t rows, int M, int N, float *dbias, int bias_stride, void *stream);
/* out[n * out_stride] += sum_r B[r*ldb + n] */
int bmp_colsum(const float *B, int ldb, float *out, int out_stride, int64_t rows, int N, void *stream);

/* ---- loss (train_binary.py:524: F.sigmoid_cross_entropy, mean over t != -1) --
 * `count` = number of non-ignored elements the mean divides by (pass the GLOBAL
 * count under data parallelism); loss_sum[0] += sum of per-element losses / count;
 * d_logits = (sigmoid(x) - t) / count.                                            */
int bmp_sigmoid_ce(const float *logits, const int32_t *labels, float *loss_sum,
                   float *d_logits, int n, float count, void *stream);

/* Adam as chainer.optimizers.Adam (alpha, beta1, beta2, eps, weight_decay_rate):
 * train_binary.py:533-536.  step = t (1-based).                                   */
int bmp_adam_step(float *param, const float *grad, float *m, float *v, int n,
                  float alpha, float beta1, float beta2, float eps,
                  float weight_decay_rate, int step, void *stream);

/* ---- one training step of a drug PAIR batch in ONE call ------------------------
 * replaces GraphConvPredictorForPair.__call__ + the loss and Chainer's backward through them (train_binary.py:84-118,524)
 * for the headline composition: the SAME GGNN encoder on both drugs (its final atom states; the co-attention ignores the
 * graph vectors, nie_coattention.py:335) -> fine-grained co-attention (Nie / VQA; variant POOL with head = 0) -> HolE
 * (circular correlation, hidden_dims = (), l_out) -> sigmoid cross-entropy (mean over labels != -1).
 * Writes `logits` (mb, n_classes), ADDS the loss into loss[0] and every parameter gradient into its d_* pointer (the layout
 * a flat gradient buffer wants: tied steps pass the same pointers).  The caller owns everything, including ONE workspace of
 * bmp_pair_workspace_bytes(): both encoder stashes (fp32, or the bf16 panel stash in BMP_MODE_BF16), the weight images, the
 * co-attention temporaries.  BMP_MODE_F32 runs the encoders on the fp32 tensor-core path when the shape is covered.       */
typedef struct {
    int mb, n1, n2, hidden, out_dim, head, n_classes, n_steps, n_atom_types, mode;
    int coattn_variant, coattn_act;
    const int32_t *atoms_1, *atoms_2;      /* (mb,N1), (mb,N2) */
    const void    *adj_1, *adj_2;          /* (mb,4,N1,N1), (mb,4,N2,N2): fp32, or the storage `adj_u8` names (BMP_MODE_BF16 only) */
    const int32_t *labels;                 /* (mb,n_classes), -1 = ignored */
    float count;                           /* what the loss mean divides by (the GLOBAL count of labels != -1 under data parallelism) */
    const float *embed_W;
    const float *msg_W[BMP_MAX_STEPS], *msg_b[BMP_MAX_STEPS];
    bmp_gru_t    gru[BMP_MAX_STEPS];
    int          stateful[BMP_MAX_STEPS];
    const float *W, *V1, *V2, *b, *lt_1, *lt_2, *wa_1, *wa_2, *W_j, *b_j;     /* co-attention, as bmp_coattn_fwd_t */
    const float *out_W, *out_b;            /* HolE l_out: (n_classes, out_dim), (n_classes) */
    float *d_embed_W;
    float *d_msg_W[BMP_MAX_STEPS], *d_msg_b[BMP_MAX_STEPS];
    bmp_gru_grad_t d_gru[BMP_MAX_STEPS];
    float *d_W, *d_V1, *d_V2, *d_b, *d_lt_1, *d_lt_2, *d_wa_1, *d_wa_2, *d_W_j, *d_b_j;
    float *d_out_W, *d_out_b;
    float *logits, *loss;
    void  *workspace;
    size_t workspace_bytes;
    int    adj_u8;                         /* storage of adj_1 / adj_2 as in bmp_ggnn_fwd_t: 0 fp32, 1 bytes, 2 bit-packed rows (BF16 mode) */
} bmp_pair_t;

size_t bmp_pair_workspace_bytes(int mb, int n1, int n2, int hidden, int out_dim, int head, int n_classes, int n_steps, int mode);
int bmp_pair_forward_backward(const bmp_pair_t *a, void *stream);

/* ---- remaining link-prediction heads (SURVEY 8 f-4) --------------------------------
 * Pair features feeding a Linear stack:
 *   BMP_PAIR_SYM    out (rows, 2*dim) = [l + r | l * r]     SymMLP, models/mlp.py:104-105
 *   BMP_PAIR_PROD   out (rows, dim)   = l * r               DistMult: BilinearDiag (models/mlp.py:154-197) is Linear(l * r)
 *   BMP_PAIR_CONCAT out (rows, 2*dim) = [l | r]             MLP head, train_binary.py:98-100 (F.concat)            */
enum { BMP_PAIR_SYM = 0, BMP_PAIR_PROD = 1, BMP_PAIR_CONCAT = 2 };
int bmp_pair_features_forward(const float *left, const float *right, float *out, int rows, int dim, int kind, void *stream);
int bmp_pair_features_backward(const float *left, const float *right, const float *d_out, float *d_left, float *d_right,
                               int rows, int dim, int kind, void *stream);

/* chainer.links.Bilinear(left, right, out) as the NTN head uses it (models/mlp.py:47-74):
 *   y[b,k] = sum_ij e1[b,i] W[i,j,k] e2[b,j] + e1 V1 + e2 V2 + b      W (left,right,out), V1 (left,out), V2 (right,out), b (out)
 * u (rows, right*out) = e1 W_flat is caller-owned scratch kept for the backward; du (same size) is backward scratch.
 * V1/V2/b may be NULL together (nobias).  Parameter gradients ACCUMULATE (+=); de1/de2 are overwritten.               */
int bmp_bilinear_forward(const float *e1, const float *e2, const float *W, const float *V1, const float *V2, const float *b,
                         float *u, float *y, int rows, int left, int right, int out, void *stream);
int bmp_bilinear_backward(const float *e1, const float *e2, const float *W, const float *V1, const float *V2, const float *u,
                          const float *dy, float *du, float *de1, float *de2, float *dW, float *dV1, float *dV2, float *db,
                          int rows, int left, int right, int out, void *stream);

/* ---- atom-wise primitives of the vector-query co-attentions (`--attn alter | para | circ`) -------------------------
 * models/coattention/alternating_coattention.py:34-80, parallel_coattention.py:33-80 (ParallelCoattention) and :107-160
 * (CircularParallelCoattention): a (mb, O) query vector against (mb, N, C) atom arrays.
 *   bcast_add_act   y[b,n,c] = act(x[b,n,c] + v[b,c]); x NULL = F.tile of v over the atoms, v NULL = plain activation.
 *                   backward: dx = dy * act'(y) (NULL: skipped), dv[b,c] = sum over atoms of the same (NULL: skipped)
 *   softmax         F.softmax(x, axis=1) over the atoms of each (b, c)
 *   pool            out[b,c] = sum_n a[b,n,(a_ch == 1 ? 0 : c)] * z[b,n,c]  = F.sum(F.tile(attn) * z, axis=1)              */
int bmp_atoms_bcast_add_act_forward(const float *x, const float *v, float *y, int mb, int n_atoms, int ch, int act, void *stream);
int bmp_atoms_bcast_add_act_backward(const float *y, const float *dy, float *dx, float *dv, int mb, int n_atoms, int ch, int act, void *stream);
int bmp_atoms_softmax_forward(const float *x, float *y, int mb, int n_atoms, int ch, void *stream);
int bmp_atoms_softmax_backward(const float *y, const float *dy, float *dx, int mb, int n_atoms, int ch, void *stream);
int bmp_atoms_pool_forward(const float *a, int a_ch, const float *z, float *out, int mb, int n_atoms, int ch, void *stream);
int bmp_atoms_pool_backward(const float *a, int a_ch, const float *z, const float *d_out, float *da, float *dz,
                            int mb, int n_atoms, int ch, void *stream);

/* GIN aggregation, models/gin.py:88-94: out[b,i,:] = h[b,i,:] + sum_e sum_j adj[b,e,i,j] h[b,j,:]; `transpose` != 0 uses
 * adj[b,e,j,i] instead -- the same call is the backward with respect to h (pass d_out as h).  fp32, N <= 256 with
 * N * hidden * 4 bytes well inside the 227 KB of shared memory of a block.                                              */
int bmp_gin_aggregate(const float *adj, const float *h, float *out, int mb, int n_edge, int n_atoms, int hidden,
                      int transpose, void *stream);

/* Optimizer hooks of train_binary.py:537-543 on the flat gradient, in the order the reference adds them:
 * GradientClipping(threshold) (g *= threshold/||g||_2 when that is < 1; off when threshold <= 0), WeightDecay(l2_rate)
 * (g += l2 * p), Lasso(l1_rate) (g += l1 * sign(p)).  norm_ws: one float of device scratch (needed when clipping).     */
int bmp_grad_hooks(float *grad, const float *param, int n, float clip_threshold, float l2_rate, float l1_rate,
                   float *norm_ws, void *stream);

/* ---- housekeeping ------------------------------------------------------------ */
const char *bmp_last_error(void);
int         bmp_version(void);
int         bmp_device_check(void);           /* BMP_OK iff current device is sm_100 */
uint64_t    bmp_launch_count(void);           /* kernels launched by this library    */
void        bmp_reset_launch_count(void);

/* ---- BiMPM matching co-attention ---------------------------------------------
 * replaces models/coattention/bimpm.py:17-197 (`--attn bimpm`, train_binary.py:253-256) with all three matchings on
 * (max-pooling, attentive, max-attentive) and aggr = F.sum: out_k (mb, 3*head) = [max-pool | att-mean | att-max] matching
 * vectors summed over the atoms of drug k.  As in the reference, mp_matching_func keeps column 0 of its head x head product
 * (perspective k of an atom against perspective 0 of its attentive vector).  fp32; N1, N2 <= 64; head * hidden <= 16384.
 * backward: d_atoms_k are overwritten, the three weight gradients accumulated (+=).  `workspace`: bmp_bimpm_workspace_bytes. */
typedef struct {
    int mb, n1, n2, hidden, head;
    const float *atoms_1, *atoms_2;                              /* (mb,N1,H), (mb,N2,H) */
    const float *max_pooling_W, *att_mean_W, *att_max_W;         /* (head,H) each        */
    float *out_1, *out_2;                                        /* forward: (mb,3*head) */
    const float *d_out_1, *d_out_2;                              /* backward inputs      */
    float *d_atoms_1, *d_atoms_2;
    float *d_max_pooling_W, *d_att_mean_W, *d_att_max_W;         /* may be NULL          */
    void  *workspace;
    size_t workspace_bytes;
} bmp_bimpm_t;
size_t bmp_bimpm_workspace_bytes(int mb, int n1, int n2, int hidden, int head);
int bmp_bimpm_forward(const bmp_bimpm_t *a, void *stream);
int bmp_bimpm_backward(const bmp_bimpm_t *a, void *stream);

/* ---- NFP encoder pieces (models/models/nfp.py) ------------------------------
 * EmbedAtomID forward (the GGNN / RelGCN encoders fuse this gather): out[r,:] = embed_W[clamp(atoms[r]), :].
 * bmp_nfp_gather, NFPUpdate (nfp.py:35-59) on the (mb,N,N) adjacency of the NFP preprocessor:
 *   forward  (backward == 0): src = h (mb,N,C) -> dst = X (mb,N,D*C), X[b,i,(d-1)C+c] = (adj[b] h[b])[i,c] if degree(b,i) == d
 *            (degree = column sums of adj, nfp.py:152; d = 1..D), else 0; the D degree-specific GraphLinears are then one
 *            Linear over X with their weights concatenated along the input axis and their biases summed;
 *   backward (backward != 0): src = dX -> dst = dh = adj[b]^T (degree block of dX).  fp32, N <= 256.                       */
int bmp_embed_forward(const int32_t *atoms, const float *embed_W, float *out, int rows, int hidden, int n_atom_types, void *stream);
int bmp_nfp_gather(const float *adj, const float *src, float *dst, int mb, int n_atoms, int ch, int n_degree, int backward,
                   void *stream);

/* ---- per-kernel timing (measurement aid, no reference counterpart) ----------
 * With profiling enabled every launch of the hot tcgen05 kernels is bracketed by two CUDA events recorded on the
 * launching stream; bmp_profile_read synchronises on them, adds the elapsed milliseconds and launch counts per kind
 * into ms[] / launches[] (n_kinds entries, BMP_PROF_* order) and forgets them.  Off by default.                    */
enum { BMP_PROF_GGNN_FWD = 0, BMP_PROF_GGNN_BWD = 1, BMP_PROF_WGRAD = 2, BMP_PROF_COATTN_FWD = 3, BMP_PROF_COATTN_BWD = 4,
       BMP_PROF_READOUT = 5, BMP_PROF_KINDS = 6 };
void bmp_profile_enable(int on);
int  bmp_profile_read(double *ms, long long *launches, int n_kinds);

#ifdef __cplusplus
}
#endif
#endif /* GCNBMP_H_ */
