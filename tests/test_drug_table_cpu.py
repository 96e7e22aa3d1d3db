"""Host side of the drug table on the fp32 tensor-core encoder: which calls read the table in place and which keep gathering,
the storage the encoder is handed, and the header's description of the relaxed BMP_MODE_F32 fields."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fwd(mb, N, H, E, T, state=False, bias_off=0):
    """a GgnnFwd as the host fills it before deciding (pointer values only: the decision never dereferences them)"""
    import ctypes as C
    from gcnbmp import _capi as K, functional as Fn
    a = K.GgnnFwd()
    a.mb, a.n_atoms, a.hidden, a.n_edge, a.n_steps, a.mode = mb, N, H, E, T, K.MODE_F32
    a.state_in = C.c_void_p(1 << 20) if state else None
    for t in range(T):
        a.msg_W[t] = C.c_void_p(1 << 16)
        a.msg_b[t] = C.c_void_p((1 << 17) + bias_off)
        for i, name in enumerate(Fn.GRU_FIELDS):
            setattr(a.gru[t], name, C.c_void_p((1 << 18) + 4096 * i))
    return a


def test_row_path_decision_names_the_calls_that_read_the_table_in_place(monkeypatch):
    """the host asks the library (bmp_ggnn_x3_forward_bytes), which applies the test bmp_ggnn_forward itself applies"""
    from gcnbmp import _capi as K, functional as Fn
    assert Fn.x3_row_path(_fwd(12, 100, 64, 4, 3), False)
    assert Fn.x3_row_path(_fwd(2, 64, 128, 4, 6), True)             # 128 rows: one full row tile
    assert Fn.x3_row_path(_fwd(1, 256, 128, 4, 2), False)
    assert not Fn.x3_row_path(_fwd(1, 100, 64, 4, 3), False)         # fewer than 128 rows: FFMA kernels, gathered rows
    assert not Fn.x3_row_path(_fwd(12, 100, 64, 4, 3, state=True), False)   # an external GRU state
    assert not Fn.x3_row_path(_fwd(12, 100, 96, 4, 3), False)        # hidden not 64 / 128 / 256
    assert not Fn.x3_row_path(_fwd(12, 100, 64, 3, 3), False)        # 3 bond types
    assert not Fn.x3_row_path(_fwd(4, 256, 256, 4, 3), False)        # 256 x 256 fp32 tile does not fit shared memory
    assert not Fn.x3_row_path(_fwd(12, 100, 64, 4, 3, bias_off=4), False)   # a bias vector not 16-byte aligned
    a = _fwd(12, 100, 64, 4, 3)
    assert K.lib.bmp_ggnn_x3_forward_bytes(C.byref(a), 0) == K.lib.bmp_ggnn_x3_workspace_bytes(12, 100, 64, 4, 3, 0)
    monkeypatch.setattr(Fn, "F32_TENSOR_CORES", False)
    assert not Fn.x3_row_path(_fwd(12, 100, 64, 4, 3), False)


def test_row_path_keeps_the_table_storage_and_the_ffma_route_widens_it():
    from gcnbmp import _capi as K, functional as Fn
    rng = np.random.default_rng(0)
    adj = torch.tensor((rng.random((3, 4, 100, 100)) < 0.05).astype(np.float32))
    packed = Fn.pack_adjacency(adj)
    t, code = Fn._adj(packed, K.MODE_F32, keep=True)
    assert code == 2 and t.dtype == torch.uint8 and tuple(t.shape) == (3, 4, 100, 13)
    t, code = Fn._adj(adj.to(torch.bool), K.MODE_F32, keep=True)
    assert code == 1 and t.dtype == torch.uint8 and torch.equal(t.float(), adj)
    t, code = Fn._adj(packed, K.MODE_F32)
    assert code == 0 and t.dtype == torch.float32 and torch.equal(t, adj)
    t, code = Fn._adj(adj.to(torch.uint8), K.MODE_F32)
    assert code == 0 and torch.equal(t, adj)


def test_header_documents_the_fp32_table_fields():
    text = open(os.path.join(ROOT, "include", "gcnbmp.h")).read()
    fwd = text[text.index("typedef struct {\n    int mb, n_atoms, hidden, n_edge, n_steps, n_atom_types, mode;"):text.index("} bmp_ggnn_fwd_t;")]
    bwd = text[text.index("} bmp_ggnn_fwd_t;"):text.index("} bmp_ggnn_bwd_t;")]
    pair = text[text.index("int mb, n1, n2, hidden"):text.index("} bmp_pair_t;")]
    flat = lambda s: re.sub(r"\s+", " ", s)
    for block in (fwd, bwd):
        assert "BMP_MODE_BF16 only, storage" not in block and "BMP_MODE_BF16 only, or NULL" not in block
        assert "tensor-core row path" in flat(block) and "BMP_ESHAPE" in block and "BMP_EINVAL" in block
    assert "mb is the length of the index" in flat(fwd)
    assert "BMP_MODE_F32 takes 1 / 2 when both encoders run on the tensor-core row path" in flat(pair)
