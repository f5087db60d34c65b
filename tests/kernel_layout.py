"""Shared-memory sizes of the solve kernels restated from fcc_qp_b200/csrc/fccqp_kernel.cuh, so that tests can tell from
fccqp_last_launch_info which kernel ran."""


def up8(v):
    return (v + 7) & ~7


def layout_bytes(n, m, nc):
    """fccqp::Layout::bytes(): shared memory of one QP on the general kernel."""
    up2 = lambda v: (v + 1) & ~1
    N8 = up8(n) + up8(m)
    NB, NT = N8 >> 3, ((N8 + 31) >> 5) * 32
    return 8 * (NB * (NB + 1) // 2 * 64 + 4 * NT + up8(n) + 8 + 2 * up2(nc + 2) + up2(nc // 3 + 2) + 4 * 32 + 32)
