"""CPU checks of the pruned passes' workspace size now that the work list holds 128-point boxes: a pure function of
(n, W), monotone in both, and large enough for the worst case in which the cull lists every box of every tile."""
import pytest


@pytest.fixture(scope="module")
def L():
    from trajectory_optimization_b200 import _lib
    return _lib.lib()


NS = [1, 127, 128, 1023, 1024, 1025, 65_536, 65_537, 300_037, 1_000_000, 25_600_000, 100_000_000]
WS = [1, 31, 32, 33, 64, 100, 320, 1000, 2048]


def _mask_words(W):  # mask_stride_words: pose words rounded up to a 16-byte multiple
    return (((W + 31) >> 5) + 3) & ~3


def test_workspace_is_a_pure_function_and_monotone(L):
    for W in WS:
        sizes = [L.cov_traj_workspace_bytes(n, W) for n in NS]
        assert sizes == [L.cov_traj_workspace_bytes(n, W) for n in NS]
        assert all(a <= b for a, b in zip(sizes, sizes[1:])), (W, sizes)
    for n in NS:
        sizes = [L.cov_traj_workspace_bytes(n, W) for W in WS]
        assert all(a <= b for a, b in zip(sizes, sizes[1:])), (n, sizes)
        assert all(s % 256 == 0 for s in sizes)


def test_workspace_holds_every_box_listed(L):
    for n in NS:
        for W in WS:
            items = ((n + 1023) // 1024) * 8                 # every box of every 1024-point tile
            need = (items * 4                                 # work list (box indices)
                    + items * _mask_words(W) * 4              # one pose mask per listed box
                    + L.cov_tile_boxes_count(n) * 32          # the boxes built into the workspace when none are given
                    + W * 6 * 16)                             # pose table
            assert L.cov_traj_workspace_bytes(n, W) >= need, (n, W)


def test_sweep_workspaces_cover_the_trajectory_workspace(L):
    for n in (65_536, 1_000_000, 25_600_000):
        for n_traj, per in ((1, 1), (16, 64), (200, 10), (3, 2048)):
            W = min(n_traj * per, 2048)
            assert L.cov_sweep_workspace_bytes(n, n_traj, per) >= L.cov_traj_workspace_bytes(n, W)
            assert L.cov_sweep_fused_workspace_bytes(n, n_traj, per, None) >= L.cov_traj_workspace_bytes(n, min(W, 2048))
