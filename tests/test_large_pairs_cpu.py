"""Host-only sizing of the co-attention scratch for molecules of 65..256 atoms (csrc/coattn_big.cu) and of the one-call pair
step that carves it."""


def test_large_coattention_workspace_query_is_host_only():
    q = __import__("gcnbmp")._capi.lib.bmp_coattn_large_workspace_bytes
    assert q(64, 64, 128, 8) == 0 and q(20, 64, 64, 8) == 0          # both sides fit the shared-memory-resident kernels
    assert q(100, 70, 196, 8) == 0 and q(100, 70, 256, 8) == 0       # atoms wider than 192
    assert q(257, 20, 64, 8) == 0 and q(20, 257, 64, 8) == 0
    assert q(100, 70, 66, 8) == 0 and q(100, 70, 64, 17) == 0
    for n1, n2, H, head in [(65, 64, 64, 8), (100, 70, 128, 8), (128, 128, 192, 16), (256, 33, 64, 0), (33, 256, 64, 1),
                            (256, 256, 192, 8)]:
        n = q(n1, n2, H, head)
        assert n >= 148 * n1 * n2 * 4, (n1, n2, H)                   # one energy slice per CTA of the persistent grid
    assert q(256, 256, 192, 8) > q(100, 70, 192, 8)


def test_pair_step_workspace_grows_by_the_coattention_scratch_above_64_atoms():
    lib = __import__("gcnbmp")._capi.lib
    q = lib.bmp_pair_workspace_bytes
    mb, H, O, hd, K, T = 64, 64, 24, 8, 3, 3
    big = q(mb, 100, 70, H, O, hd, K, T, 0)
    scratch = lib.bmp_coattn_large_workspace_bytes(100, 70, H, hd)
    assert scratch > 0 and big >= scratch
    # on top of the per-row buffers (here just the fp32 stash of h_0 .. h_T of both drugs) the plan carves one co-attention scratch
    assert big >= scratch + mb * (100 + 70) * H * 4 * (T + 1)
    assert big > q(mb, 64, 64, H, O, hd, K, T, 0) + scratch
