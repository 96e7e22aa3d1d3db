"""Deterministic mode (include/gcnbmp.h "Deterministic reductions"): C exports, version and size queries, no GPU needed."""
import ctypes as C
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gcn-bmp_b200"))

K = pytest.importorskip("gcnbmp._capi")

NEW = ["bmp_ggnn_backward_det_bytes", "bmp_relgcn_backward_det_bytes", "bmp_readout_backward_det_bytes",
       "bmp_coattn_backward_det_bytes", "bmp_linear_backward_det", "bmp_linear_backward_det_bytes", "bmp_embed_backward_det",
       "bmp_embed_backward_det_bytes", "bmp_sigmoid_ce_det", "bmp_sigmoid_ce_det_bytes", "bmp_grad_hooks_det",
       "bmp_grad_hooks_det_bytes", "bmp_bilinear_backward_det", "bmp_bilinear_backward_det_bytes"]


def test_exports_and_version():
    assert K.lib.bmp_version() >= 101
    for name in NEW:
        assert hasattr(K.lib, name) and name in K.EXPORTS


@pytest.mark.parametrize("cls", [K.GgnnBwd, K.RelgcnBwd, K.ReadoutBwd, K.CoattnBwd])
def test_struct_ends_with_det_fields(cls):
    names = [f[0] for f in cls._fields_]
    assert names[-2:] == ["det_scratch", "det_scratch_bytes"]
    header = open(os.path.join(ROOT, "include", "gcnbmp.h")).read()
    assert header.count("size_t det_scratch_bytes;") == 4


def test_struct_size_queries():
    g = K.GgnnBwd()
    assert K.lib.bmp_ggnn_backward_det_bytes(C.byref(g)) == 0            # empty struct: nothing to cover
    g.mb, g.n_atoms, g.hidden, g.n_edge, g.n_steps, g.mode = 8288, 64, 128, 4, 6, K.MODE_BF16
    bf16 = K.lib.bmp_ggnn_backward_det_bytes(C.byref(g))
    # one wgrad2 launch: at most one 192 KB slot per SM (148 on a B200, the fallback without a device)
    assert 148 * 192 * 1024 <= bf16 <= 256 * 200 * 1024
    g.mode = K.MODE_F32
    assert 0 < K.lib.bmp_ggnn_backward_det_bytes(C.byref(g)) <= bf16 * 4
    r = K.RelgcnBwd()
    r.mb, r.n_atoms, r.n_edge, r.n_layers = 64, 100, 4, 2
    for l, c in enumerate((64, 64, 64)):
        r.ch[l] = c
    assert K.lib.bmp_relgcn_backward_det_bytes(C.byref(r)) > 0
    ro = K.ReadoutBwd()
    ro.mb, ro.n_atoms, ro.hidden, ro.out_dim = 4096, 64, 128, 128
    assert K.lib.bmp_readout_backward_det_bytes(C.byref(ro)) > 0
    co = K.CoattnBwd()
    assert K.lib.bmp_coattn_backward_det_bytes(C.byref(co)) == 0
    co.mb, co.n1, co.n2, co.hidden, co.out_dim, co.head = 8288, 64, 64, 128, 128, 8
    assert K.lib.bmp_coattn_backward_det_bytes(C.byref(co)) >= 148 * (128 * 128 + 34 * 128) * 4


def test_plain_size_queries():
    assert K.lib.bmp_linear_backward_det_bytes(0, 128, 86) == 0
    assert K.lib.bmp_linear_backward_det_bytes(4096, 128, 86) >= 128 * 86 * 4
    assert K.lib.bmp_embed_backward_det_bytes(1000, 128, 100) >= 148 * 100 * 128 * 4
    # a table wider than the owner kernel's shared memory runs as column tiles: one tile's slots at a time
    assert 148 * 117 * 216 * 4 <= K.lib.bmp_embed_backward_det_bytes(1000, 256, 117) < 148 * 117 * 256 * 4
    assert K.lib.bmp_sigmoid_ce_det_bytes(0) == 0 and K.lib.bmp_sigmoid_ce_det_bytes(10 ** 6) >= 4
    assert K.lib.bmp_grad_hooks_det_bytes(10 ** 6) >= 4


def test_null_scratch_is_refused():
    rc = K.lib.bmp_sigmoid_ce_det(None, None, None, None, 10, 1.0, None, None, 0)
    assert rc == K.EINVAL and b"scratch" in K.lib.bmp_last_error()


# ---- each struct query against the scratch every call of that entry point takes, with the sites' own split rules
SMS = 148


def _wgrad(M, N, rows=10 ** 8):          # gemm.cu bmp_wgrad: take(split * M * N)
    tiles = ((M + 63) // 64) * ((N + 63) // 64)
    split = max(1, min((4 * SMS + tiles - 1) // tiles, (rows + 127) // 128))
    return split * M * N * 4 + 512


def _colsum(N, rows=10 ** 8):
    tiles = (N + 63) // 64
    return max(1, min((2 * SMS + tiles - 1) // tiles, (rows + 255) // 256)) * N * 4 + 512


def _wgrad_tc(M, N, rows=10 ** 8):       # wgrad_tc.cu: C and bias partials
    mt = (M + 127) // 128
    split = max(1, min((SMS + mt - 1) // mt, (rows + 511) // 512))
    return split * M * N * 4 + 256 + split * M * 4 + 512


@pytest.mark.parametrize("H", [16, 32, 64, 96, 128, 192, 256])
@pytest.mark.parametrize("O", [16, 24, 64, 86, 100, 128, 200, 256])
def test_coattn_and_readout_queries_cover_their_calls(H, O):
    co = K.CoattnBwd()
    co.mb, co.n1, co.n2, co.hidden, co.out_dim, co.head = 8288, 64, 64, H, O, 8
    have = K.lib.bmp_coattn_backward_det_bytes(C.byref(co))
    for M in (H, O, 8):                  # d W (M = H), d W_j (M = O), d lt_k (M = head); all N = H
        assert have >= _wgrad(M, H) and have >= _wgrad_tc(M, H), (M, H)
    assert have >= _colsum(O)
    ro = K.ReadoutBwd()
    ro.mb, ro.n_atoms, ro.hidden, ro.out_dim = 8288, 64, H, O
    have = K.lib.bmp_readout_backward_det_bytes(C.byref(ro))
    for N in (H, 2 * H):
        assert have >= _wgrad(O, N) and have >= _wgrad_tc(O, N)
    assert have >= _colsum(O)


@pytest.mark.parametrize("ch", [[16, 128, 64], [128, 192], [64, 64, 64], [256, 256], [16, 32, 32], [100, 70, 256]])
def test_relgcn_query_covers_its_calls(ch):
    r = K.RelgcnBwd()
    r.mb, r.n_atoms, r.n_edge, r.n_layers = 4096, 100, 4, len(ch) - 1
    for l, c in enumerate(ch):
        r.ch[l] = c
    have = K.lib.bmp_relgcn_backward_det_bytes(C.byref(r))
    pad = lambda c: 64 if c <= 64 else 128 if c <= 128 else 256
    for l in range(len(ch) - 1):
        cin, cout = ch[l], ch[l + 1]
        assert have >= _wgrad(cout, cin) and have >= _colsum(cout)
        assert have >= _wgrad_tc(pad(cout), pad(cin))


@pytest.mark.parametrize("H", [16, 32, 64, 128, 256])
def test_ggnn_query_covers_its_calls(H):
    g = K.GgnnBwd()
    g.mb, g.n_atoms, g.hidden, g.n_edge, g.n_steps, g.mode = 8288, 64, H, 4, 3, K.MODE_F32
    have = K.lib.bmp_ggnn_backward_det_bytes(C.byref(g))
    assert have >= _wgrad(H, H) and have >= _wgrad_tc(H, H) and have >= _colsum(H)


@pytest.mark.parametrize("L,R,O", [(32, 32, 8), (64, 100, 86), (128, 16, 4)])
def test_bilinear_query_covers_its_calls(L, R, O):
    have = K.lib.bmp_bilinear_backward_det_bytes(20000, L, R, O)
    assert have >= _wgrad(L, R * O) and have >= _wgrad(L, O) and have >= _wgrad(R, O) and have >= _colsum(O)
