"""RelGCN, GIN and NFP on molecules with more than 64 atoms (fp32 mode), against the fp64 NumPy oracle.

The reference pads every batch to its largest molecule with no atom cap (ggnn_preprocessor.py:41, max_atoms=-1), so one large
drug in a batch takes the whole batch past 64 atoms.  RelGCN runs such batches on the tensor-core row path of csrc/ggnn_x3.cu,
GIN's aggregation and NFP's gather on their per-molecule kernels tiled over adjacency rows."""
import numpy as np
import pytest
import torch

import cases
import product
from product import rel_err
from oracle import minichainer as F
from oracle import reference_path as R

pytestmark = pytest.mark.gpu
TOL = 1e-4

# (N, ch_list, mb): ragged molecules inside the padding; mb = 1 at N = 100 is fewer rows than one 128-row GEMM tile
RELGCN_CASES = [
    (65, [64] * 5, 3),
    (100, [64] * 5, 3),
    (128, [16, 128, 64], 2),
    (256, [128, 128], 2),
    (100, [16, 128, 64], 1),
]


def _molecules(seed, mb, N, n_max=None):
    """mb molecules of up to n_max (default N) atoms, padded to N atoms"""
    from gcnbmp import synthetic
    return synthetic.random_molecules(np.random.default_rng(seed), mb, n_max or N, pad_to=N)


def _check_grads(got, want, tol=TOL):
    assert set(got) == set(want)
    for k in sorted(want):
        if want[k] is None:                 # a parameter the oracle's graph never reached (GIN's unused read-outs)
            assert not np.any(got[k]), k
            continue
        assert got[k].shape == want[k].shape, k
        err = rel_err(got[k], want[k], floor=1e-7)
        assert err <= tol, (k, err)


def _relgcn_step(atoms, adj, ch, scale_adj, params, mode=None):
    """graph vector, atom states and parameter gradients of loss = sum(g * wg) + sum(atoms * wa): oracle and product."""
    import gcnbmp
    rng = np.random.default_rng(1)
    O = 32
    mb, N = atoms.shape
    wg, wa = rng.standard_normal((mb, O)), rng.standard_normal((mb, N, ch[-1]))
    tab = R.wrap_params(params)
    onet = R.RelGCN(R.P(tab), O, ch_list=ch, scale_adj=scale_adj)
    og = onet(atoms, adj.astype(np.float64))
    F.add(F.sum_(F.mul(og, F.const(wg))), F.sum_(F.mul(onet.get_atom_array(), F.const(wa)))).backward()
    net = gcnbmp.RelGCN(O, ch_list=ch, scale_adj=scale_adj)
    net.load_params({k: np.asarray(v, np.float32) for k, v in params.items()})
    if mode is not None:
        net.mode = mode
    net.cleargrads()
    pg = net(atoms, adj)
    pa = net.get_atom_array()
    loss = (pg * torch.tensor(wg, dtype=torch.float32, device="cuda")).sum() + \
        (pa * torch.tensor(wa, dtype=torch.float32, device="cuda")).sum()
    loss.backward()
    torch.cuda.synchronize()
    return dict(g=(pg.detach().cpu().numpy(), og.data), atoms=(pa.detach().cpu().numpy(), onet.get_atom_array().data),
                grads=(net.grad_dict(), {k: tab[k].grad for k in params}))


@pytest.mark.parametrize("scale_adj", [False, True])
@pytest.mark.parametrize("N,ch,mb", RELGCN_CASES)
def test_relgcn_stack_above_64_atoms_matches_oracle(N, ch, mb, scale_adj):
    atoms, adj = _molecules(N + mb, mb, N, n_max=N - 7)     # ragged: every molecule smaller than the padding
    params = R.init_params(R.relgcn_shapes(32, ch), np.random.default_rng(N), dtype=np.float64)
    r = _relgcn_step(atoms, adj, ch, scale_adj, params)
    assert rel_err(*r["g"]) <= TOL
    assert rel_err(*r["atoms"]) <= TOL
    _check_grads(*r["grads"])


def test_bare_relgcn_update_at_100_atoms_with_fractional_adjacency():
    """General (non-0/1) edge weights: the adjacency products read the dense values, not only the bit masks."""
    import gcnbmp
    rng = np.random.default_rng(8)
    mb, N, cin, cout = 3, 100, 16, 40
    _, adj = _molecules(3, mb, N)
    adj = adj * rng.random(adj.shape).astype(np.float32)
    h = rng.standard_normal((mb, N, cin))
    shapes = {"graph_linear_self/W": (cout, cin), "graph_linear_self/b": (cout,),
              "graph_linear_edge/W": (cout * 4, cin), "graph_linear_edge/b": (cout * 4,)}
    params = R.init_params(shapes, rng, dtype=np.float64)
    tab = R.wrap_params(params)
    hv = F.param(h)
    o = R.RelGCNUpdate(R.P(tab), cin, cout)(hv, adj.astype(np.float64))
    F.sum_(F.mul(o, o)).backward()
    link = gcnbmp.RelGCNUpdate(cin, cout)
    link.load_params(params)
    ht = torch.tensor(h, dtype=torch.float32, device="cuda", requires_grad=True)
    p = link(ht, adj)
    (p * p).sum().backward()
    assert rel_err(p.detach().cpu().numpy(), o.data) <= TOL
    assert rel_err(ht.grad.cpu().numpy(), hv.grad) <= TOL
    _check_grads(link.grad_dict(), {k: tab[k].grad for k in params})


def _relgcn_pair_case(attn, seed):
    rng = np.random.default_rng(seed)
    sp = dict(enc="relgcn", ch=[16, 64, 64], O=32, scale_adj=True, attn=attn, head=4 if attn else None, hole_hidden=(), K=1,
              mb=3, N1=100, N2=70)
    a1, A1 = _molecules(seed, sp["mb"], 100)
    a2, A2 = _molecules(seed + 1, sp["mb"], 70)
    shapes = {"graph_conv/" + k: v for k, v in R.relgcn_shapes(sp["O"], sp["ch"]).items()}
    d_in = sp["O"]
    if attn:
        shapes.update({"attn/" + k: v for k, v in R.coattn_shapes(sp["ch"][-1], sp["O"], sp["head"]).items()})
    shapes.update({"mlp/" + k: v for k, v in R.hole_shapes(d_in, 1, ()).items()})
    y = (rng.random((sp["mb"], 1)) < 0.4).astype(np.int32)
    return dict(name="relgcn-large", spec=sp, params=R.init_params(shapes, rng, dtype=np.float64),
                inputs=(a1, A1.astype(np.float64), a2, A2.astype(np.float64)), labels=y)


@pytest.mark.parametrize("attn", [None, "nie"])
def test_relgcn_pair_step_at_100_and_70_atoms_matches_oracle(attn):
    case = _relgcn_pair_case(attn, 21)
    o = cases.oracle_eval(case)
    p = product.product_eval(case)
    assert rel_err(p["logits"], o["logits"]) <= TOL
    assert abs(p["loss"] - float(o["loss"])) <= TOL * max(1.0, abs(float(o["loss"])))
    for k in sorted(o["grads"]):
        err = rel_err(p["grads"][k], o["grads"][k], floor=1e-3 if o["grads"][k].size == 1 else 1e-30)
        assert err <= TOL, (k, err)


def test_bf16_mode_relgcn_takes_batches_past_64_atoms_through_the_fp32_path():
    """A RelGCN model in BF16 mode does not fail on a batch padded past 64 atoms: that batch runs the fp32 tensor-core row path
    (inside the fp32 bound), also when the adjacency arrives as bytes."""
    import gcnbmp
    case = _relgcn_pair_case("nie", 33)
    o = cases.oracle_eval(case)
    p = product.product_eval(case, mode=gcnbmp.MODE_BF16)
    assert rel_err(p["logits"], o["logits"]) <= TOL
    for k in sorted(o["grads"]):
        assert rel_err(p["grads"][k], o["grads"][k], floor=1e-3 if o["grads"][k].size == 1 else 1e-30) <= TOL, k
    model = product.product_model(case["spec"], case["params"])
    model.graph_conv.mode = model.attn.mode = gcnbmp.MODE_BF16
    a1, A1, a2, A2 = case["inputs"]
    with torch.no_grad():
        y8 = model(a1, A1.astype(np.uint8), a2, A2.astype(np.uint8)).cpu().numpy()
    assert rel_err(y8, o["logits"]) <= TOL


@pytest.mark.parametrize("tied,concat", [(True, False), (False, False), (True, True), (False, True)])
def test_gin_at_100_atoms_matches_oracle(tied, concat):
    import gcnbmp
    mb, N, H, O, T = 3, 100, 16, 12, 3
    atoms, adj = _molecules(40, mb, N)
    params = R.init_params(R.gin_shapes(O, H, T, concat_hidden=concat, weight_tying=tied), np.random.default_rng(41), dtype=np.float64)
    tab = R.wrap_params(params)
    og = R.GIN(R.P(tab), O, H, T, concat_hidden=concat, weight_tying=tied)(atoms, adj.astype(np.float64))
    w = np.random.default_rng(42).standard_normal(og.data.shape)
    F.sum_(F.mul(og, F.const(w))).backward()
    net = gcnbmp.GIN(O, hidden_dim=H, n_layers=T, dropout_ratio=0.0, concat_hidden=concat, weight_tying=tied)
    net.load_params({k: np.asarray(v, np.float32) for k, v in params.items()})
    net.cleargrads()
    pg = net(atoms, adj)
    (pg * torch.tensor(w, dtype=torch.float32, device="cuda")).sum().backward()
    assert rel_err(pg.detach().cpu().numpy(), og.data) <= TOL
    _check_grads(net.grad_dict(), {k: tab[k].grad for k in params})


def test_nfp_at_100_atoms_matches_oracle():
    import gcnbmp
    mb, N, H, O, T = 3, 100, 16, 12, 3
    atoms, adj4 = _molecules(50, mb, N)
    adj = (adj4.sum(axis=1) + np.eye(N, dtype=np.float32)[None] * (atoms > 0)[:, :, None]).astype(np.float32)
    params = R.init_params(R.nfp_shapes(O, H, T), np.random.default_rng(51), dtype=np.float64)
    w = np.random.default_rng(52).standard_normal((mb, O))
    tab = R.wrap_params(params)
    onet = R.NFP(R.P(tab), O, H, T)
    og = onet(atoms, adj.astype(np.float64))
    F.sum_(F.mul(og, F.const(w))).backward()
    net = gcnbmp.NFP(O, hidden_dim=H, n_layers=T)
    net.load_params({k: np.asarray(v, np.float32) for k, v in params.items()})
    net.cleargrads()
    pg = net(atoms, adj)
    (pg * torch.tensor(w, dtype=torch.float32, device="cuda")).sum().backward()
    assert rel_err(pg.detach().cpu().numpy(), og.data) <= TOL
    assert rel_err(net.get_atom_array().detach().cpu().numpy(), onet.get_atom_array().data) <= TOL
    want = {k: tab[k].grad for k in params if tab[k].grad is not None and np.abs(tab[k].grad).max() > 1e-9}
    got = net.grad_dict()
    for k in want:
        assert rel_err(got[k], want[k]) <= TOL, k


@pytest.mark.parametrize("scale_adj", [False, True])
def test_relgcn_same_molecules_padded_to_64_100_and_128_agree(scale_adj):
    """Padded atoms carry no bonds, so the real atoms' states and the parameter gradients of a loss over them do not depend on the
    padding.  Padded to 100 and to 128 atoms (both on the tensor-core row path: the same per-row arithmetic) they agree to fp32
    rounding of the gradient sums.  Padded to 64 atoms (FFMA kernels) they agree within the fp32-mode bound: the row GEMMs carry
    each fp32 operand as a bf16 hi / lo pair (about 2^-17 relative), which at these pre-activations (|x| up to 11 before tanh)
    moves the states by a few 1e-5, where the FFMA kernels stay near 1e-6."""
    import gcnbmp
    mb, ch = 4, [16, 64, 64, 64]
    a64, A64 = _molecules(60, mb, 64, n_max=60)
    n = (a64 > 0).sum(axis=1)
    params = {k: np.asarray(v, np.float32) for k, v in
              R.init_params(R.relgcn_shapes(32, ch), np.random.default_rng(61), dtype=np.float64).items()}
    live = np.arange(64)[None, :] < n[:, None]
    w = np.random.default_rng(62).standard_normal((mb, 64, ch[-1])) * live[:, :, None]
    out = []
    for N in (64, 100, 128):
        atoms, adj = np.zeros((mb, N), np.int32), np.zeros((mb, 4, N, N), np.float32)
        atoms[:, :64], adj[:, :, :64, :64] = a64, A64
        net = gcnbmp.RelGCN(32, ch_list=ch, scale_adj=scale_adj)
        net.load_params(params)
        net.cleargrads()
        net(atoms, adj)
        h = net.get_atom_array()[:, :64]
        (h * torch.tensor(w, dtype=torch.float32, device="cuda")).sum().backward()
        g = net.grad_dict()
        out.append((h.detach().cpu().numpy() * live[:, :, None], {k: v for k, v in g.items() if not k.startswith("rgcn_readout")}))
    ffma, x100, x128 = out
    assert rel_err(x128[0], x100[0]) <= 1e-6
    for k in x100[1]:
        assert rel_err(x128[1][k], x100[1][k], floor=1e-7) <= 1e-5, k
    assert rel_err(x100[0], ffma[0]) <= TOL
    for k in ffma[1]:
        assert rel_err(x100[1][k], ffma[1][k], floor=1e-7) <= TOL, k


def test_relgcn_above_64_atoms_outside_the_covered_shapes_fails_loudly():
    import gcnbmp
    atoms, adj = _molecules(70, 2, 257)
    with pytest.raises(ValueError, match="n_atoms=257"):
        gcnbmp.RelGCN(16, ch_list=[64, 64])(atoms, adj)
    atoms, adj = _molecules(71, 2, 200)
    with pytest.raises(ValueError, match="n_atoms=200"):           # 200 x 256 fp32 channels do not fit the adjacency tile
        gcnbmp.RelGCN(16, ch_list=[256, 256])(atoms, adj)
    atoms, adj = _molecules(72, 2, 100)
    with pytest.raises(ValueError, match="n_atoms=100"):           # three bond types
        gcnbmp.RelGCN(16, ch_list=[64, 64], num_edge_type=3)(atoms, adj[:, :3])
