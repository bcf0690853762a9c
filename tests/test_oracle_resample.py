"""CPU: the numpy restatement of monai._C.grid_pull (oracle/resample.py) against the reference's golden rows and against outputs
of the reference's own C++ sources (compiled into oracle/_ref by oracle/build_ref.py; fixtures in tests/golden/grid_pull.npz)."""
import os

import numpy as np

from oracle import resample as ors

INTERP = ["nearest", "linear", "quadratic", "cubic", "fourth", "fifth", "sixth", "seventh"]


def test_oracle_reproduces_1d_bp_fwd_rows(golden_dir):
    """tests/testing_data/1D_BP_fwd.txt (56 rows = 7 bounds x 8 orders), the vectors of tests/networks/layers/test_grid_pull.py."""
    g = np.load(os.path.join(golden_dir, "grid_pull.npz"))
    x = np.arange(10, dtype=np.float32).reshape(1, 1, 10, 1, 1)
    grid = np.zeros((1, 20, 1, 1, 3), dtype=np.float32)
    grid[0, :, 0, 0, 0] = np.arange(20, dtype=np.float32) + 0.5
    assert len(g["bp1d.labels"]) == 56
    for row, lab in zip(g["bp1d.rows"], g["bp1d.labels"]):
        it, bt = str(lab).split()
        o, b = INTERP.index(it.split(".")[1]), ors.BOUNDS[bt.split(".")[1]]
        got = ors.grid_pull(x, grid, [b, 0, 0], [o, 0, 0]).reshape(-1)
        np.testing.assert_allclose(got, row, rtol=1e-4, atol=1e-4, err_msg=str(lab))


def test_oracle_matches_compiled_reference_3d(golden_dir):
    g = np.load(os.path.join(golden_dir, "grid_pull.npz"))
    for bn, b in ors.BOUNDS.items():
        for o in range(8):
            got = ors.grid_pull(g["x"], g["grid"], [b] * 3, [o] * 3)
            np.testing.assert_allclose(got, g[f"y.{bn}.{o}"], rtol=2e-4, atol=2e-5, err_msg=f"{bn} order {o}")
    np.testing.assert_allclose(ors.grid_pull(g["x"], g["grid"], [2, 5, 3], [3, 1, 2]), g["y.mixed"], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(ors.grid_pull(g["x"], g["grid"], [0, 0, 0], [1, 1, 1], extrapolate=False), g["y.noextrap"], rtol=2e-4, atol=2e-5)


def test_oracle_matches_the_stored_compiled_reference_dst2_cubic(golden_dir):
    """monai._C.grid_pull of the reference's own C++ (dst2, cubic; fixture of make_golden.py grid_pull_ref_dst2) against the
    restatement.  Where oracle/_ref has been built, the compiled module must also import and reproduce the stored output."""
    g = np.load(os.path.join(golden_dir, "grid_pull_dst2_cubic.npz"))
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 2, 5, 4, 6)).astype(np.float32)
    grid = (rng.random((1, 3, 4, 5, 3)) * 9 - 2).astype(np.float32)
    np.testing.assert_array_equal(x, g["x"])
    np.testing.assert_array_equal(grid, g["grid"])
    np.testing.assert_allclose(ors.grid_pull(x, grid, [4] * 3, [3] * 3), g["y"], rtol=2e-4, atol=2e-5)

    from oracle import build_ref

    C = build_ref.load()
    if C is not None:
        import torch

        ref = C.grid_pull(torch.from_numpy(x), torch.from_numpy(grid), [C.BoundType(4)] * 3, [C.InterpolationType(3)] * 3, True).numpy()
        np.testing.assert_allclose(ref, g["y"], rtol=1e-6, atol=1e-6)


def test_oracle_push_and_count_match_the_compiled_reference(golden_dir):
    """monai._C.grid_push / grid_count outputs of the reference's own C++ (tests/golden/make_golden.py grid_push_ref)."""
    g = np.load(os.path.join(golden_dir, "grid_push.npz"))
    for i in range(int(g["n"])):
        bound, order, extrap, *shape = (int(v) for v in g[f"c{i}.cfg"])
        got = ors.grid_push(g[f"c{i}.x"], g[f"c{i}.grid"], shape, [bound] * 3, [order] * 3, bool(extrap))
        np.testing.assert_allclose(got, g[f"c{i}.y"], rtol=1e-5, atol=2e-6, err_msg=f"case {i}: bound {bound} order {order} extrapolate {extrap}")
    np.testing.assert_allclose(ors.grid_count(g["count.grid"], (5, 6, 7), [2] * 3, [1] * 3), g["count.y"], rtol=1e-5, atol=2e-6)


def test_oracle_grad_matches_the_compiled_reference(golden_dir):
    """monai._C.grid_grad outputs of the reference's own C++ (make_golden.py grid_push_ref)."""
    g = np.load(os.path.join(golden_dir, "grid_push.npz"))
    assert int(g["n_grad"]) >= 30
    for i in range(int(g["n_grad"])):
        bound, order, extrap = (int(v) for v in g[f"g{i}.cfg"])
        got = ors.grid_grad(g[f"g{i}.x"], g[f"g{i}.grid"], [bound] * 3, [order] * 3, bool(extrap))
        np.testing.assert_allclose(got, g[f"g{i}.y"], rtol=1e-4, atol=1e-5, err_msg=f"case {i}: bound {bound} order {order} extrapolate {extrap}")


def test_oracle_count_and_grad_reproduce_1d_bp_bwd_rows(golden_dir):
    """tests/testing_data/1D_BP_bwd.txt: the gradients of grid_pull(arange(10), arange(20) + 0.5).sum() that
    tests/networks/layers/test_grid_pull.py checks.  d/d input = grid_count of the grid into the input's shape (grid_push of ones),
    d/d grid = grid_grad of the input: 56 golden rows (7 bounds x 8 orders) for the push / count / grad restatements."""
    g = np.load(os.path.join(golden_dir, "grid_push.npz"))
    x = np.arange(10, dtype=np.float32).reshape(1, 1, 10, 1, 1)
    grid = np.zeros((1, 20, 1, 1, 3), dtype=np.float32)
    grid[0, :, 0, 0, 0] = np.arange(20, dtype=np.float32) + 0.5
    assert len(g["bp1d_bwd.labels"]) == 56
    for row, lab in zip(g["bp1d_bwd.rows"], g["bp1d_bwd.labels"]):
        it, bt = str(lab).split()
        o, b = INTERP.index(it.split(".")[1]), ors.BOUNDS[bt.split(".")[1]]
        cnt = ors.grid_count(grid, (10, 1, 1), [b, 0, 0], [o, 0, 0]).reshape(-1)
        np.testing.assert_allclose(cnt, row[:10], rtol=1e-4, atol=1e-4, err_msg=f"count {lab}")
        grd = ors.grid_grad(x, grid, [b, 0, 0], [o, 0, 0])[..., 0].reshape(-1)
        np.testing.assert_allclose(grd, row[10:], rtol=1e-4, atol=1e-4, err_msg=f"grad {lab}")


def test_backward_compositions_match_the_compiled_reference(golden_dir):
    """monai._C.grid_pull_backward / grid_push_backward / grid_count_backward (fixtures of make_golden.py grid_push_ref): the backward
    passes monai_b200 attaches to grid_pull / grid_push / grid_count are compositions of the FORWARD operators --
    pull: (push(grad), sum_c grad * grad_op(input)); push: (pull(grad), sum_c input * grad_op(grad)); count: grad_op(grad)."""
    g = np.load(os.path.join(golden_dir, "grid_push.npz"))
    assert int(g["n_bwd"]) >= 16
    for i in range(int(g["n_bwd"])):
        bound, order, extrap = (int(v) for v in g[f"b{i}.cfg"])
        bb, oo, ex = [bound] * 3, [order] * 3, bool(extrap)
        x, grid, gout, xin, gvol, gcnt = (g[f"b{i}.{k}"] for k in ("x", "grid", "gout", "xin", "gvol", "gcnt"))
        tol = dict(rtol=1e-4, atol=1e-5, err_msg=f"case {i}: bound {bound} order {order} extrapolate {extrap}")
        np.testing.assert_allclose(ors.grid_push(gout, grid, x.shape[2:], bb, oo, ex), g[f"b{i}.pull_dx"], **tol)
        np.testing.assert_allclose((ors.grid_grad(x, grid, bb, oo, ex) * gout[..., None]).sum(1), g[f"b{i}.pull_dg"], **tol)
        np.testing.assert_allclose(ors.grid_pull(gvol, grid, bb, oo, ex), g[f"b{i}.push_dx"], **tol)
        np.testing.assert_allclose((ors.grid_grad(gvol, grid, bb, oo, ex) * xin[..., None]).sum(1), g[f"b{i}.push_dg"], **tol)
        np.testing.assert_allclose(ors.grid_grad(gcnt, grid, bb, oo, ex)[:, 0], g[f"b{i}.count_dg"], **tol)
