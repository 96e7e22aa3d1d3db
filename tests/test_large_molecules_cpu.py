"""Host-side checks of the RelGCN tensor-core row path for molecules with more than 64 atoms (no GPU needed)."""


def test_relgcn_x3_workspace_query_is_host_only_and_covers_65_to_256_atoms():
    q = __import__("gcnbmp")._capi.lib.bmp_relgcn_x3_workspace_bytes
    covered = [(100, 64), (65, 16), (128, 128), (256, 128), (160, 256), (100, 200)]
    for N, ch in covered:
        n = q(8, N, ch, 4, 0)
        assert n > 0, (N, ch)
        assert q(16, N, ch, 4, 0) > n                       # grows with the batch
        assert q(8, N, ch, 4, 1) == n                       # same size for inference
        assert n > 8 * N * 4 * ch * 4                       # at least the A_e h temporaries of one layer
    assert q(1, 100, 64, 4, 0) > 0                          # fewer rows than one 128-row GEMM tile
    assert q(8, 64, 64, 4, 0) == 0 and q(8, 10, 64, 4, 0) == 0       # <= 64 atoms: the FFMA kernels
    assert q(8, 257, 64, 4, 0) == 0
    assert q(8, 200, 256, 4, 0) == 0                        # 200 x 256 fp32 channels exceed the 160 KB adjacency tile
    assert q(8, 100, 257, 4, 0) == 0
    assert q(0, 100, 64, 4, 0) == 0 and q(8, 100, 64, 0, 0) == 0 and q(8, 100, 64, 17, 0) == 0
