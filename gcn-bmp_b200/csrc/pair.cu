// pair.cu -- bmp_pair_forward_backward: one training step of a drug-pair batch as ONE C call.
//
// Host-side composition of the library's own entry points for the headline model (train_binary.py:84-118 with a GGNN encoder, a
// fine-grained co-attention and HolE; loss :524): encoder on drug 1 and drug 2 (same weights) -> co-attention on the final atom
// states -> circular correlation -> l_out -> sigmoid cross-entropy, then the backward chain in reverse.  Every launch goes to the
// caller's stream; nothing is allocated: the caller's workspace is carved here.  A CuPy / Chainer process needs nothing but this
// call (INTEGRATION.md); the Torch host (gcnbmp/train.py) composes the same calls itself because it also serves the other heads,
// encoders and attention variants.
#include <cstring>
#include "common.cuh"

using namespace bmp;

namespace {

struct Carve {
    uint8_t *p;
    size_t used;
    explicit Carve(void *base) : p((uint8_t *)(((uintptr_t)base + 1023) & ~(uintptr_t)1023)), used(1024) {}
    template <class T>
    T *take(size_t n) {
        const size_t bytes = (n * sizeof(T) + 1023) & ~(size_t)1023;
        T *r = p ? reinterpret_cast<T *>(p) : nullptr;
        if (p) p += bytes;
        used += bytes;
        return r;
    }
};

struct Enc {            // per-drug encoder buffers
    float *Hs, *Ms, *Gs, *RSs, *Ps, *dHs;      // fp32 stash (BMP_MODE_F32)
    float *out2, *dout2;                       // BMP_MODE_BF16: [h_0, h_T] and their gradients
    uint8_t *stash2;
    float *R, *DL;                             // co-attention backward workspaces of this side
};

struct Plan {
    Enc e[2];
    void *x3_ws, *tc_fwd, *tc_bwd, *co_ws;
    size_t x3_bytes, tc_bytes, co_bytes;
    float *c1, *c2, *dc1, *dc2, *P1, *P2, *corr, *dcorr, *dlogits;
    size_t total;
};

Plan make_plan(void *base, int mb, int n1, int n2, int H, int O, int head, int K, int T, int mode) {
    Plan pl;
    memset(&pl, 0, sizeof(pl));
    Carve c(base);
    const int N[2] = {n1, n2};
    const bool bf16 = mode == BMP_MODE_BF16;
    for (int s = 0; s < 2; ++s) {
        const size_t R = (size_t)mb * N[s], RH = R * H;
        Enc &e = pl.e[s];
        if (bf16) {
            e.out2 = c.take<float>(2 * RH);
            e.dout2 = c.take<float>(2 * RH);
            e.stash2 = c.take<uint8_t>(bmp_ggnn_stash2_bytes(mb, H, T));
        } else {
            e.Hs = c.take<float>((size_t)(T + 1) * RH);
            e.Ms = c.take<float>((size_t)T * RH);
            e.Gs = c.take<float>((size_t)T * 3 * RH);
            e.RSs = c.take<float>((size_t)T * RH);
            e.Ps = c.take<float>((size_t)T * 4 * RH);
            e.dHs = c.take<float>((size_t)(T + 1) * RH);
        }
        e.R = c.take<float>(RH);
        e.DL = c.take<float>(R * (size_t)(head > 0 ? head : 1));
    }
    if (bf16) {
        pl.tc_bytes = bmp_ggnn_tc_workspace_bytes(H, T);
        pl.tc_fwd = c.take<uint8_t>(pl.tc_bytes);
        pl.tc_bwd = c.take<uint8_t>(pl.tc_bytes);
        pl.co_bytes = bmp_coattn_tc_workspace_bytes(H);
        pl.co_ws = c.take<uint8_t>(pl.co_bytes ? pl.co_bytes : 16);
    } else {
        const size_t b1 = bmp_ggnn_x3_workspace_bytes(mb, n1, H, 4, T, 0), b2 = bmp_ggnn_x3_workspace_bytes(mb, n2, H, 4, T, 0);
        pl.x3_bytes = (b1 && b2) ? (b1 > b2 ? b1 : b2) : 0;          // both drugs or neither: one image set serves both
        pl.x3_ws = pl.x3_bytes ? c.take<uint8_t>(pl.x3_bytes) : nullptr;
        pl.co_bytes = bmp_coattn_large_workspace_bytes(n1, n2, H, head);     // 0 unless a molecule has more than 64 atoms
        pl.co_ws = pl.co_bytes ? c.take<uint8_t>(pl.co_bytes) : nullptr;
    }
    pl.c1 = c.take<float>((size_t)mb * O); pl.c2 = c.take<float>((size_t)mb * O);
    pl.dc1 = c.take<float>((size_t)mb * O); pl.dc2 = c.take<float>((size_t)mb * O);
    pl.P1 = c.take<float>((size_t)mb * H); pl.P2 = c.take<float>((size_t)mb * H);
    pl.corr = c.take<float>((size_t)mb * O); pl.dcorr = c.take<float>((size_t)mb * O);
    pl.dlogits = c.take<float>((size_t)mb * K);
    pl.total = c.used;
    return pl;
}

bool shape_bad(int mb, int n1, int n2, int H, int O, int head, int K, int T) {
    return mb <= 0 || n1 <= 0 || n2 <= 0 || H <= 0 || O <= 0 || head < 0 || K <= 0 || T <= 0 || T > BMP_MAX_STEPS;
}

}  // namespace

extern "C" size_t bmp_pair_workspace_bytes(int mb, int n1, int n2, int hidden, int out_dim, int head, int n_classes, int n_steps, int mode) {
    if (shape_bad(mb, n1, n2, hidden, out_dim, head, n_classes, n_steps)) return 0;
    if (mode == BMP_MODE_BF16 && bmp_ggnn_stash2_bytes(mb, hidden, n_steps) == 0) return 0;
    return make_plan(nullptr, mb, n1, n2, hidden, out_dim, head, n_classes, n_steps, mode).total;
}

extern "C" int bmp_pair_forward_backward(const bmp_pair_t *a, void *stream) {
    if (!a || !a->atoms_1 || !a->atoms_2 || !a->adj_1 || !a->adj_2 || !a->labels || !a->embed_W || !a->out_W || !a->logits || !a->loss ||
        !a->workspace) {
        set_error("bmp_pair_forward_backward: null argument");
        return BMP_EINVAL;
    }
    const int mb = a->mb, H = a->hidden, O = a->out_dim, K = a->n_classes, T = a->n_steps, head = a->head;
    if (shape_bad(mb, a->n1, a->n2, H, O, head, K, T)) { set_error("bmp_pair_forward_backward: bad shape"); return BMP_ESHAPE; }
    const size_t need = bmp_pair_workspace_bytes(mb, a->n1, a->n2, H, O, head, K, T, a->mode);
    if (need == 0 || a->workspace_bytes < need) {
        set_error("bmp_pair_forward_backward: workspace of %zu bytes, %zu needed", a->workspace_bytes, need);
        return BMP_EINVAL;
    }
    if (!(a->count > 0.f)) { set_error("bmp_pair_forward_backward: count must be positive"); return BMP_EINVAL; }
    const bool bf16 = a->mode == BMP_MODE_BF16;
    cudaStream_t st = (cudaStream_t)stream;
    Plan pl = make_plan(a->workspace, mb, a->n1, a->n2, H, O, head, K, T, a->mode);
    const int N[2] = {a->n1, a->n2};
    const int32_t *atoms[2] = {a->atoms_1, a->atoms_2};
    const void *adj[2] = {a->adj_1, a->adj_2};
    if (a->adj_u8 && !bf16 && !pl.x3_ws) {
        set_error("bmp_pair_forward_backward: adj_u8=%d in BMP_MODE_F32 needs both encoders on the tensor-core row path (hidden "
                  "64/128/256, mb * n_atoms >= 128 on each side)", a->adj_u8);
        return BMP_EINVAL;
    }
    const float *hT[2];
    float *d_hT[2];
    int rc;

    // ---------------------------------------------------------------- forward: the encoder on both drugs
    for (int s = 0; s < 2; ++s) {
        const size_t RH = (size_t)mb * N[s] * H;
        Enc &e = pl.e[s];
        bmp_ggnn_fwd_t f;
        memset(&f, 0, sizeof(f));
        f.mb = mb; f.n_atoms = N[s]; f.hidden = H; f.n_edge = 4; f.n_steps = T; f.n_atom_types = a->n_atom_types; f.mode = a->mode;
        f.atoms = atoms[s]; f.embed_W = a->embed_W; f.adj = reinterpret_cast<const float *>(adj[s]); f.adj_u8 = a->adj_u8;
        for (int t = 0; t < T; ++t) { f.msg_W[t] = a->msg_W[t]; f.msg_b[t] = a->msg_b[t]; f.gru[t] = a->gru[t]; f.stateful[t] = a->stateful[t]; }
        if (bf16) {
            f.h0_out = e.out2; f.h_out = e.out2 + RH; f.stash2 = e.stash2;
            f.tc_workspace = pl.tc_fwd; f.tc_workspace_bytes = pl.tc_bytes; f.tc_images_ready = s;      // drug 2 reuses drug 1's images
            hT[s] = e.out2 + RH; d_hT[s] = e.dout2 + RH;
        } else {
            f.Hs = e.Hs; f.Ms = e.Ms; f.Gs = e.Gs; f.RSs = e.RSs;
            f.tc_workspace = pl.x3_ws; f.tc_workspace_bytes = pl.x3_bytes; f.tc_images_ready = s;
            hT[s] = e.Hs + (size_t)T * RH; d_hT[s] = e.dHs + (size_t)T * RH;
        }
        if ((rc = bmp_ggnn_forward(&f, stream))) return rc;
    }
    // ---------------------------------------------------------------- co-attention, HolE, loss
    bmp_coattn_fwd_t cf;
    memset(&cf, 0, sizeof(cf));
    cf.mb = mb; cf.n1 = a->n1; cf.n2 = a->n2; cf.hidden = H; cf.out_dim = O; cf.head = head; cf.variant = a->coattn_variant; cf.act = a->coattn_act;
    cf.atoms_1 = hT[0]; cf.atoms_2 = hT[1];
    cf.W = a->W; cf.V1 = a->V1; cf.V2 = a->V2; cf.b = a->b; cf.lt_1 = a->lt_1; cf.lt_2 = a->lt_2; cf.wa_1 = a->wa_1; cf.wa_2 = a->wa_2;
    cf.W_j = a->W_j; cf.b_j = a->b_j;
    cf.compact_1 = pl.c1; cf.compact_2 = pl.c2;
    cf.mode = a->mode; cf.tc_workspace = pl.co_ws; cf.tc_workspace_bytes = pl.co_bytes;
    if ((rc = bmp_coattn_forward(&cf, stream))) return rc;
    if ((rc = bmp_hole_corr_forward(pl.c1, pl.c2, pl.corr, mb, O, stream))) return rc;
    if ((rc = bmp_linear_forward(pl.corr, a->out_W, a->out_b, a->logits, mb, O, K, BMP_ACT_IDENTITY, stream))) return rc;
    if ((rc = bmp_sigmoid_ce(a->logits, a->labels, a->loss, pl.dlogits, mb * K, a->count, stream))) return rc;
    // ---------------------------------------------------------------- backward
    if ((rc = bmp_linear_backward(pl.corr, a->out_W, a->logits, pl.dlogits, pl.dcorr, a->d_out_W, a->d_out_b, mb, O, K, BMP_ACT_IDENTITY, stream)))
        return rc;
    if ((rc = bmp_hole_corr_backward(pl.c1, pl.c2, pl.dcorr, pl.dc1, pl.dc2, mb, O, stream))) return rc;
    for (int s = 0; s < 2; ++s) {       // gradients w.r.t. h_0 .. h_{T-1} start at zero; the co-attention overwrites the h_T slice
        const size_t RH = (size_t)mb * N[s] * H;
        if (bf16) cudaMemsetAsync(pl.e[s].dout2, 0, RH * sizeof(float), st);
        else cudaMemsetAsync(pl.e[s].dHs, 0, (size_t)T * RH * sizeof(float), st);
    }
    bmp_coattn_bwd_t cb;
    memset(&cb, 0, sizeof(cb));
    cb.mb = mb; cb.n1 = a->n1; cb.n2 = a->n2; cb.hidden = H; cb.out_dim = O; cb.head = head; cb.variant = a->coattn_variant; cb.act = a->coattn_act;
    cb.atoms_1 = hT[0]; cb.atoms_2 = hT[1];
    cb.W = a->W; cb.V1 = a->V1; cb.V2 = a->V2; cb.b = a->b; cb.lt_1 = a->lt_1; cb.lt_2 = a->lt_2; cb.wa_1 = a->wa_1; cb.wa_2 = a->wa_2;
    cb.W_j = a->W_j; cb.b_j = a->b_j;
    cb.d_compact_1 = pl.dc1; cb.d_compact_2 = pl.dc2;
    cb.R = pl.e[0].R; cb.P1 = pl.P1; cb.P2 = pl.P2; cb.DL1 = pl.e[0].DL; cb.DL2 = pl.e[1].DL;
    cb.d_atoms_1 = d_hT[0]; cb.d_atoms_2 = d_hT[1];
    cb.d_W = a->d_W; cb.d_V1 = a->d_V1; cb.d_V2 = a->d_V2; cb.d_b = a->d_b; cb.d_lt_1 = a->d_lt_1; cb.d_lt_2 = a->d_lt_2;
    cb.d_wa_1 = a->d_wa_1; cb.d_wa_2 = a->d_wa_2; cb.d_W_j = a->d_W_j; cb.d_b_j = a->d_b_j;
    cb.mode = a->mode; cb.tc_workspace = pl.co_ws; cb.tc_workspace_bytes = pl.co_bytes; cb.tc_images_ready = 1;
    if ((rc = bmp_coattn_backward(&cb, stream))) return rc;
    for (int s = 0; s < 2; ++s) {
        Enc &e = pl.e[s];
        bmp_ggnn_bwd_t g;
        memset(&g, 0, sizeof(g));
        g.mb = mb; g.n_atoms = N[s]; g.hidden = H; g.n_edge = 4; g.n_steps = T; g.mode = a->mode;
        g.adj = reinterpret_cast<const float *>(adj[s]); g.adj_u8 = a->adj_u8;
        for (int t = 0; t < T; ++t) {
            g.msg_W[t] = a->msg_W[t]; g.gru[t] = a->gru[t]; g.stateful[t] = a->stateful[t];
            g.d_msg_W[t] = a->d_msg_W[t]; g.d_msg_b[t] = a->d_msg_b[t]; g.d_gru[t] = a->d_gru[t];
        }
        if (bf16) {
            g.stash2 = e.stash2; g.dHs = e.dout2;
            g.tc_workspace = pl.tc_bwd; g.tc_workspace_bytes = pl.tc_bytes; g.tc_images_ready = s;
        } else {
            g.Hs = e.Hs; g.Ms = e.Ms; g.RSs = e.RSs; g.Gs = e.Gs; g.Ps = e.Ps; g.dHs = e.dHs;
            g.tc_workspace = pl.x3_ws; g.tc_workspace_bytes = pl.x3_bytes; g.tc_images_ready = 1;       // packed by the forward
        }
        if ((rc = bmp_ggnn_backward(&g, stream))) return rc;
        if (a->d_embed_W &&
            (rc = bmp_embed_backward(atoms[s], bf16 ? e.dout2 : e.dHs, a->d_embed_W, mb * N[s], H, a->n_atom_types, stream)))
            return rc;
    }
    return BMP_OK;
}
