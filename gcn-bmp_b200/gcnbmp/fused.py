"""The whole pair training step as ONE C call (`bmp_pair_forward_backward`, csrc/pair.cu): what a host without an autograd
engine binds (INTEGRATION.md).  This module is the Torch-side caller of that entry for the headline composition
-- `GraphConvPredictorForPair(GGNNMono, NieFineCoattention | VQAParallelCoattention | PoolingFineCoattention, HolE(hidden_dims=()))`,
train_binary.py:84-118,524 -- and the cross-check of the composed autograd path in train.PairTrainer."""
import ctypes as C

import torch

from . import _capi as K
from . import functional as Fn
from . import links


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def supported(model):
    enc, attn, head = model.graph_conv, model.attn, model.mlp
    return (isinstance(enc, links.GGNNMono) and not enc.concat_hidden and
            isinstance(attn, (links.NieFineCoattention, links.PoolingFineCoattention)) and
            not isinstance(attn, (links.FourierFineCoattention,)) and
            isinstance(head, links.HolE) and all(len(list(c)) == 0 for n, c in head._children.items() if n != "l_out") and
            not getattr(model, "first_last_atoms", False))


def pair_forward_backward(model, atoms_1, adj_1, atoms_2, adj_2, labels, count=None):
    """One fwd+bwd of the pair model in a single library call.  Adds every parameter gradient into `p.grad` (created as zeros
    when absent), returns (loss, logits).  `count`: what the loss mean divides by (default: this batch's labels != -1)."""
    Fn.no_deterministic("gcnbmp.fused.pair_forward_backward (the one-call step reduces with atomics)")
    if not supported(model):
        raise ValueError("gcnbmp.fused: the one-call step covers GGNNMono + fine / pooling co-attention + HolE(hidden_dims=())")
    enc, attn, head = model.graph_conv, model.attn, model.mlp
    dev = torch.device("cuda")
    a1 = torch.as_tensor(atoms_1).to(dev, torch.int32).contiguous()
    a2 = torch.as_tensor(atoms_2).to(dev, torch.int32).contiguous()
    mode = model.graph_conv.__dict__.get("mode", K.MODE_F32)
    A1, u8 = Fn._adj(torch.as_tensor(adj_1).to(dev), mode)          # BF16 mode keeps a uint8 / bit-packed adjacency as it is
    A2, u8_2 = Fn._adj(torch.as_tensor(adj_2).to(dev), mode)
    if u8 != u8_2:
        raise ValueError("gcnbmp.fused: both adjacencies must use the same storage")
    y = torch.as_tensor(labels).to(dev, torch.int32).contiguous()
    mb, n1, n2 = a1.shape[0], a1.shape[1], a2.shape[1]
    H, O, T, Kc = enc.hidden_dim, attn.out_dim, enc.n_layers, y.shape[1]
    pool = isinstance(attn, links.PoolingFineCoattention)
    hd = 0 if pool else attn.head
    if count is None:
        count = float((y != -1).sum().item())

    def grad_of(p):
        if p is None:
            return None
        if p.grad is None:
            p.grad = torch.zeros_like(p)
        return p.grad

    a = K.Pair()
    a.mb, a.n1, a.n2, a.hidden, a.out_dim, a.head, a.n_classes, a.n_steps = mb, n1, n2, H, O, hd, Kc, T
    a.n_atom_types, a.mode, a.adj_u8 = enc.embed.W.shape[0], mode, u8
    a.coattn_variant, a.coattn_act = (K.COATTN_POOL if pool else K.COATTN_FINE), Fn.act_code(attn.activation)
    a.atoms_1, a.atoms_2, a.adj_1, a.adj_2, a.labels, a.count = _p(a1), _p(a2), _p(A1), _p(A2), _p(y), count
    a.embed_W, a.d_embed_W = _p(enc.embed.W), _p(grad_of(enc.embed.W))
    gru = enc.update_layer.tensors()
    for t in range(T):
        m = enc.message_layers[0 if enc.weight_tying else t]
        a.msg_W[t], a.msg_b[t] = _p(m.W), _p(m.b)
        a.d_msg_W[t], a.d_msg_b[t] = _p(grad_of(m.W)), _p(grad_of(m.b))
        Fn._fill_gru(a.gru[t], gru)
        Fn._fill_gru(a.d_gru[t], [grad_of(p) for p in gru])
        a.stateful[t] = int(t > 0)
    e = attn.energy_layer
    names = [("W", e.W), ("V1", e.V1), ("V2", e.V2), ("b", e.b), ("W_j", attn.j_layer.W), ("b_j", attn.j_layer.b)]
    if not pool:
        names += [("lt_1", attn.lt_layer_1.W), ("lt_2", attn.lt_layer_2.W), ("wa_1", attn.attention_layer_1.W),
                  ("wa_2", attn.attention_layer_2.W)]
    for n, p in names:
        setattr(a, n, _p(p))
        setattr(a, "d_" + n, _p(grad_of(p)))
    lo = head.l_out.ensure(O)
    a.out_W, a.out_b, a.d_out_W, a.d_out_b = _p(lo.W), _p(lo.b), _p(grad_of(lo.W)), _p(grad_of(lo.b))
    logits = torch.empty((mb, Kc), device=dev, dtype=torch.float32)
    loss = torch.zeros((1,), device=dev, dtype=torch.float32)
    nbytes = int(K.lib.bmp_pair_workspace_bytes(mb, n1, n2, H, O, hd, Kc, T, mode))
    if nbytes == 0:
        raise ValueError("gcnbmp.fused: shape not covered (hidden=%d, steps=%d, mode=%d)" % (H, T, mode))
    ws = torch.empty((nbytes,), device=dev, dtype=torch.uint8)
    a.logits, a.loss, a.workspace, a.workspace_bytes = _p(logits), _p(loss), _p(ws), nbytes
    K.check(K.lib.bmp_pair_forward_backward(C.byref(a), Fn._stream()))
    return loss[0], logits
