"""Generate the golden fixtures in this directory from the REAL reference (Project-MONAI/MONAI at /root/reference).

Run in the build container only (the reference does not exist on the GPU box):
    PYTHONPATH=/root/reference python tests/golden/make_golden.py
Everything is seeded; fixtures are small .npz files that are committed.
"""
from __future__ import annotations

import itertools
import os
import sys

import numpy as np
import torch

sys.path.insert(0, "/root/reference")
import monai  # noqa: E402
from monai.data.utils import compute_importance_map, dense_patch_slices, get_valid_patch_size  # noqa: E402
from monai.inferers import sliding_window_inference  # noqa: E402
from monai.inferers.utils import _get_scan_interval  # noqa: E402
from monai.networks.nets import BasicUNet, SwinUNETR, UNet  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def save(name, **arrays):
    np.savez_compressed(os.path.join(HERE, name), **arrays)
    print("wrote", name, {k: getattr(v, "shape", None) for k, v in arrays.items() if not k.startswith("sd.")})


def sd_arrays(net):
    return {"sd." + k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}


def planner():
    cases = []
    for image, roi, ov in [
        ((64, 64, 64), (32, 32, 32), 0.25), ((256, 256, 256), (96, 96, 96), 0.5), ((512, 512, 1024), (96, 96, 96), 0.5),
        ((33, 47, 21), (16, 16, 16), 0.6), ((20, 20, 20), (32, 16, 8), 0.0), ((50, 17, 9), (7, 17, 4), 0.9),
        ((100, 100), (33, 44), (0.1, 0.7)), ((7,), (3,), 0.5), ((96, 96, 96), (96, 96, 96), 0.5),
    ]:
        image_p = tuple(max(i, r) for i, r in zip(image, roi))
        ovt = ov if isinstance(ov, tuple) else (ov,) * len(image)
        interval = _get_scan_interval(image_p, roi, len(image), ovt)
        sl = dense_patch_slices(image_p, roi, interval)
        starts = np.array([[s.start for s in w] for w in sl], dtype=np.int64)
        cases.append((np.array(image), np.array(roi), np.array(ovt), np.array(interval), starts))
    out = {}
    for i, (im, roi, ov, iv, st) in enumerate(cases):
        out[f"c{i}.image"], out[f"c{i}.roi"], out[f"c{i}.overlap"], out[f"c{i}.interval"], out[f"c{i}.starts"] = im, roi, ov, iv, st
    out["n"] = np.array(len(cases))
    for j, (ps, mode, sig) in enumerate([((96, 96, 96), "gaussian", 0.125), ((8, 5, 3), "gaussian", (0.2, 0.125, 0.5)), ((4, 4), "constant", 0.125), ((32, 32, 32), "gaussian", 0.125)]):
        out[f"imp{j}.map"] = compute_importance_map(ps, mode=mode, sigma_scale=sig).numpy()
        out[f"imp{j}.patch"] = np.array(ps)
        out[f"imp{j}.sigma"] = np.atleast_1d(np.array(sig, dtype=np.float64))
        out[f"imp{j}.mode"] = np.array(mode)
    out["n_imp"] = np.array(4)
    save("planner.npz", **out)


def _cheap_predictor(x):
    """deterministic, resolution-preserving, 2 output channels: depends on values and on the window-local position."""
    ramp = torch.arange(x.shape[-1], dtype=x.dtype, device=x.device) * 0.01
    a = x.mean(dim=1, keepdim=True) * 1.5 + ramp
    b = torch.tanh(x[:, :1]) - 0.25
    return torch.cat([a, b], dim=1)


def sliding():
    torch.manual_seed(0)
    out = {}
    cases = [
        # name, shape, roi, sw_bs, overlap, mode, padding_mode, cval
        ("a", (1, 1, 64, 64, 64), (32, 32, 32), 4, 0.25, "constant", "constant", 0.0),
        ("b", (2, 2, 30, 26, 34), (12, 16, 10), 3, 0.5, "gaussian", "constant", 0.0),
        ("c", (1, 1, 20, 20, 20), (32, 16, 24), 2, 0.25, "gaussian", "constant", -1.0),
        ("d", (1, 3, 30, 30), (16, 16), 4, (0.5, 0.25), "gaussian", "replicate", 0.0),
        ("e", (1, 1, 50), (16,), 5, 0.6, "constant", "constant", 0.0),
        ("f", (1, 1, 24, 40, 40), (-1, 16, 24), 8, 0.5, "gaussian", "constant", 0.0),
    ]
    for name, shape, roi, bs, ov, mode, pm, cval in cases:
        x = torch.randn(shape)
        y = sliding_window_inference(x, roi, bs, _cheap_predictor, ov, mode, 0.125, pm, cval)
        out[f"{name}.x"], out[f"{name}.y"] = x.numpy(), y.numpy()
        out[f"{name}.roi"], out[f"{name}.bs"] = np.array(roi), np.array(bs)
        out[f"{name}.overlap"] = np.atleast_1d(np.array(ov, dtype=np.float64))
        out[f"{name}.mode"], out[f"{name}.pad"], out[f"{name}.cval"] = np.array(mode), np.array(pm), np.array(cval)
    out["names"] = np.array([c[0] for c in cases])

    # multi-resolution tuple / dict outputs (test_multioutput, tests/inferers/test_sliding_window_inference.py:314-377)
    def multi(x):
        return {"1": x + 1.0, "2": torch.nn.functional.avg_pool3d(x, 2) * 2.0, "3": x[..., ::4, ::4, ::4] - 3.0}

    x = torch.randn(1, 1, 32, 32, 32)
    r = sliding_window_inference(x, (16, 16, 16), 3, multi, 0.5, "gaussian")
    out["multi.x"] = x.numpy()
    for k, v in r.items():
        out[f"multi.y{k}"] = v.numpy()
    save("sliding_window.npz", **out)


def _load_named(net, seed):
    from weights import fill_state_dict

    net.load_state_dict(fill_state_dict(net.state_dict(), seed))
    return net.eval()


def nets():
    import contextlib
    import io

    sys.path.insert(0, HERE)
    net = _load_named(UNet(3, 1, 2, (4, 8, 16), (2, 2)), 0)
    x = torch.randn(2, 1, 16, 16, 16, generator=torch.Generator().manual_seed(10))
    with torch.no_grad():
        y = net(x)
    save("unet_tiny.npz", x=x.numpy(), y=y.numpy())

    net = _load_named(UNet(3, 1, 2, (16, 32, 64, 128, 256), (2, 2, 2, 2)), 1)  # config C2 topology
    x = torch.randn(1, 1, 32, 32, 32, generator=torch.Generator().manual_seed(11))
    with torch.no_grad():
        y = net(x)
    save("unet_c2_32.npz", x=x.numpy(), y=y.numpy())

    net = _load_named(UNet(3, 2, 3, (4, 8, 8), (2, 1), num_res_units=2), 2)
    x = torch.randn(1, 2, 12, 10, 8, generator=torch.Generator().manual_seed(12))
    with torch.no_grad():
        y = net(x)
    save("unet_res.npz", x=x.numpy(), y=y.numpy())

    with contextlib.redirect_stdout(io.StringIO()):
        net = _load_named(BasicUNet(3, 1, 2, features=(4, 4, 8, 8, 16, 4)), 3)
    x = torch.randn(1, 1, 32, 32, 32, generator=torch.Generator().manual_seed(13))
    with torch.no_grad():
        y = net(x)
    save("basic_unet_tiny.npz", x=x.numpy(), y=y.numpy())

    # feature_size=48 (config C3 architecture); 64^3 is the smallest legal input (InstanceNorm at 1/32 scale needs >1 voxel)
    net = _load_named(SwinUNETR(in_channels=1, out_channels=2, feature_size=48), 4)
    for tag, shape, seed in (("64", (64, 64, 64), 15), ("96x64x64", (96, 64, 64), 16)):
        x = torch.randn(1, 1, *shape, generator=torch.Generator().manual_seed(seed)).half().float()
        with torch.no_grad():
            hs = net.swinViT(x, True)
            y = net(x)
        save(f"swin_unetr_fs48_{tag}.npz", x=x.numpy().astype(np.float16), y_sub=y.numpy()[..., ::4, ::4, ::4],
             h0_sub=hs[0].numpy()[..., ::4, ::4, ::4], h1_sub=hs[1].numpy()[..., ::2, ::2, ::2], h2=hs[2].numpy()[:, ::4],
             h4=hs[4].numpy()[:, ::8], y_mean=np.array(float(y.double().mean())), y_absmean=np.array(float(y.double().abs().mean())))


def nets_r2():
    """Round-2 additions: the 96^3 window every C3 / C5 window has, and the SwinUNETR variants of the reference's
    constructor surface (default feature_size=24, multi-channel input, use_v2)."""
    def dump(tag, net, x):
        with torch.no_grad():
            hs = net.swinViT(x, True)
            y = net(x)
        save(f"swin_unetr_{tag}.npz", x=x.numpy().astype(np.float16), y_sub=y.numpy()[..., ::4, ::4, ::4],
             h0_sub=hs[0].numpy()[..., ::4, ::4, ::4], h4=hs[4].numpy()[:, ::8],
             y_mean=np.array(float(y.double().mean())), y_absmean=np.array(float(y.double().abs().mean())))

    net = _load_named(SwinUNETR(in_channels=1, out_channels=2, feature_size=48), 4)
    dump("fs48_96", net, torch.randn(1, 1, 96, 96, 96, generator=torch.Generator().manual_seed(17)).half().float())
    net = _load_named(SwinUNETR(in_channels=1, out_channels=2, feature_size=24), 5)
    dump("fs24_64", net, torch.randn(1, 1, 64, 64, 64, generator=torch.Generator().manual_seed(18)).half().float())
    net = _load_named(SwinUNETR(in_channels=4, out_channels=3, feature_size=48, use_v2=True), 6)
    dump("fs48_in4_v2_64", net, torch.randn(1, 4, 64, 64, 64, generator=torch.Generator().manual_seed(19)).half().float())


from dynunet_cases import DYNUNET_CASES  # noqa: E402  (shared with the tests)


def dynunet():
    """DynUNet (eval mode) of the real reference on name-keyed deterministic weights: outputs and state_dict key / shape lists."""
    import json

    from monai.networks.nets import DynUNet

    out, keys = {}, {}
    for i, (kw, shape, seed) in enumerate(DYNUNET_CASES):
        net = _load_named(DynUNet(**kw), seed)
        x = torch.randn(shape, generator=torch.Generator().manual_seed(40 + i))
        with torch.no_grad():
            y = net(x)
        out[f"c{i}.x"], out[f"c{i}.y"] = x.numpy(), y.numpy()
        keys[f"c{i}"] = {k: list(v.shape) for k, v in net.state_dict().items()}
    save("dynunet.npz", **out)
    with open(os.path.join(HERE, "dynunet_state_dict_keys.json"), "w") as f:
        json.dump(keys, f)


def segresnet():
    """SegResNet (eval mode) of the real reference on name-keyed deterministic weights: outputs and state_dict key / shape lists."""
    import json

    from monai.networks.nets import SegResNet
    from segresnet_cases import SEGRESNET_CASES

    out, keys = {}, {}
    for i, (kw, _, shape, seed) in enumerate(SEGRESNET_CASES):
        net = _load_named(SegResNet(**kw), seed)
        x = torch.randn(shape, generator=torch.Generator().manual_seed(50 + i))
        with torch.no_grad():
            y = net(x)
        out[f"c{i}.x"], out[f"c{i}.y"] = x.numpy(), y.numpy()
        keys[f"c{i}"] = {k: list(v.shape) for k, v in net.state_dict().items()}
    save("segresnet.npz", **out)
    with open(os.path.join(HERE, "segresnet_state_dict_keys.json"), "w") as f:
        json.dump(keys, f)


def unetr():
    """UNETR (eval mode) of the real reference on name-keyed deterministic weights: outputs and state_dict key / shape lists."""
    import json

    from monai.networks.nets import UNETR
    from unetr_cases import UNETR_CASES

    out, keys = {}, {}
    for i, (kw, _, shape, seed) in enumerate(UNETR_CASES):
        net = _load_named(UNETR(**kw), seed)
        x = torch.randn(shape, generator=torch.Generator().manual_seed(70 + i))
        with torch.no_grad():
            y = net(x)
        out[f"c{i}.x"], out[f"c{i}.y"] = x.numpy(), y.numpy()
        keys[f"c{i}"] = {k: list(v.shape) for k, v in net.state_dict().items()}
    save("unetr.npz", **out)
    with open(os.path.join(HERE, "unetr_state_dict_keys.json"), "w") as f:
        json.dump(keys, f)


def buffered():
    """Window order / batching the predictor observes in the reference's buffered mode (with_coord=True), plus the result."""
    out = {}
    cases = [((2, 3, 10, 11, 12), (7, 8, 10), 0.2, 2, 3, 1), ((1, 2, 20, 9, 14), (6, 9, 5), 0.5, 3, 2, -1), ((2, 1, 30, 17), (8, 6), 0.4, 4, 4, 0)]
    for ci, (img_size, roi, ov, swb, steps, dim) in enumerate(cases):
        x = torch.rand(img_size, generator=torch.Generator().manual_seed(70 + ci))
        seen = []

        def pred(patch, coords):
            seen.append(np.asarray([[c[0].start] + [s.start for s in c[2:]] for c in coords], dtype=np.int64))
            return 2.0 * patch + 1.0

        y = sliding_window_inference(x, roi, swb, pred, ov, mode="gaussian", buffer_steps=steps, buffer_dim=dim, with_coord=True)
        out[f"c{ci}.x"], out[f"c{ci}.y"] = x.numpy(), y.numpy()
        out[f"c{ci}.cfg"] = np.asarray(list(roi) + [swb, steps, dim], dtype=np.int64)
        out[f"c{ci}.ov"] = np.asarray(ov, dtype=np.float64)
        out[f"c{ci}.batch_sizes"] = np.asarray([len(a) for a in seen], dtype=np.int64)
        out[f"c{ci}.coords"] = np.concatenate(seen, 0)
    out["n"] = np.array(len(cases))
    save("buffered.npz", **out)


def resampler():
    """Dense-grid Resample of the real reference (torch path): its own unit-test cases (tests/transforms/test_resampler.py) run
    through the class, plus random deformation grids for every (mode, padding_mode, align_corners, norm_coords)."""
    from monai.transforms import Resample
    from monai.transforms.utils import create_grid

    out, n = {}, 0
    for pad, gsz, isz, mode in [("zeros", (2, 2), (1, 2, 2), None), ("zeros", (4, 4), (1, 2, 2), None), ("border", (4, 4), (1, 2, 2), None),
                                ("zeros", (4, 4, 4), (1, 2, 2, 2), "bilinear"), ("border", (4, 4, 4), (1, 2, 2, 2), "bilinear")]:
        img = torch.arange(int(np.prod(isz)), dtype=torch.float32).reshape(isz)
        grid = torch.as_tensor(create_grid(gsz))
        kw = {} if mode is None else {"mode": mode}
        y = Resample(padding_mode=pad)(img=img, grid=grid, **kw)
        out[f"c{n}.img"], out[f"c{n}.grid"], out[f"c{n}.y"] = img.numpy(), grid.numpy(), np.asarray(y)
        out[f"c{n}.cfg"] = np.asarray([str(mode or "bilinear"), pad, "0", "1"])
        n += 1
    g = torch.Generator().manual_seed(41)
    for mode in ("bilinear", "nearest"):
        for pad in ("zeros", "border", "reflection"):
            for align in (False, True):
                for norm in (True, False):
                    img = torch.rand((2, 9, 7, 11), generator=g)
                    osz = (8, 10, 6)
                    base = torch.as_tensor(create_grid(osz, dtype=np.float64))[:3]          # centred voxel coordinates
                    grid = base * (torch.tensor([9, 7, 11.0]) / torch.tensor(osz, dtype=torch.float64)).reshape(3, 1, 1, 1)
                    grid = grid + (torch.rand(grid.shape, generator=g, dtype=torch.float64) - 0.5) * 5.0   # incl. samples outside the image
                    if not norm:
                        grid = grid / (torch.tensor([9, 7, 11.0], dtype=torch.float64).reshape(3, 1, 1, 1) / 2.0)
                    if mode == "nearest":   # keep clear of the .5 ties whose rounding is round-off dependent
                        pass
                    y = Resample(mode=mode, padding_mode=pad, norm_coords=norm, align_corners=align)(img=img, grid=grid)
                    out[f"c{n}.img"], out[f"c{n}.grid"], out[f"c{n}.y"] = img.numpy(), grid.numpy(), np.asarray(y)
                    out[f"c{n}.cfg"] = np.asarray([mode, pad, str(int(align)), str(int(norm))])
                    n += 1
    out["n"] = np.array(n)
    save("resampler.npz", **out)


def grid_pull_ref():
    """monai._C.grid_pull of the REAL reference (its own C++ sources compiled into oracle/_ref, CPU): every bound x every spline
    order on a random 3-D volume with samples far outside the field of view, the per-axis mixed case, extrapolate=False, and the
    56 rows of tests/testing_data/1D_BP_fwd.txt (transcribed mechanically and re-checked against the compiled reference)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import build_ref

    C = build_ref.load()
    assert C is not None, "run python oracle/build_ref.py first"
    out = {}
    rows, labels = [], []
    for line in open("/root/reference/tests/testing_data/1D_BP_fwd.txt"):
        if "#" not in line:
            continue
        vals, lab = line.split("#")
        rows.append([float(v) for v in vals.split(",") if v.strip()])
        labels.append(lab.strip())
    out["bp1d.rows"], out["bp1d.labels"] = np.asarray(rows, dtype=np.float64), np.asarray(labels)
    bnames = {"replicate": 0, "dct1": 1, "dct2": 2, "dst1": 3, "dst2": 4, "dft": 5, "zero": 7}
    inames = ["nearest", "linear", "quadratic", "cubic", "fourth", "fifth", "sixth", "seventh"]
    x1 = torch.arange(10, dtype=torch.float32).reshape(1, 1, 10)
    g1 = (torch.arange(20, dtype=torch.float32) + 0.5).reshape(1, 20, 1)
    for r, lab in zip(rows, labels):
        it, bt = lab.split()
        o, b = inames.index(it.split(".")[1]), bnames[bt.split(".")[1]]
        got = C.grid_pull(x1, g1, [C.BoundType(b)], [C.InterpolationType(o)], True).reshape(-1).numpy()
        np.testing.assert_allclose(got, np.asarray(r), rtol=1e-4, atol=1e-4, err_msg=lab)
    g = torch.Generator().manual_seed(51)
    x = torch.randn((2, 2, 6, 7, 5), generator=g)
    grid = torch.rand((2, 4, 5, 6, 3), generator=g) * torch.tensor([14.0, 15.0, 13.0]) - 4.0
    out["x"], out["grid"] = x.numpy(), grid.numpy()
    for bn, b in bnames.items():
        for o in range(8):
            out[f"y.{bn}.{o}"] = C.grid_pull(x, grid, [C.BoundType(b)] * 3, [C.InterpolationType(o)] * 3, True).numpy()
    out["y.mixed"] = C.grid_pull(x, grid, [C.BoundType(2), C.BoundType(5), C.BoundType(3)], [C.InterpolationType(3), C.InterpolationType(1), C.InterpolationType(2)], True).numpy()
    out["y.noextrap"] = C.grid_pull(x, grid, [C.BoundType(0)] * 3, [C.InterpolationType(1)] * 3, False).numpy()
    save("grid_pull.npz", **out)


def grid_pull_ref_dst2():
    """monai._C.grid_pull of the REAL reference (oracle/_ref, CPU), dst2 bound, cubic order, samples outside the field of view:
    the inputs of tests/test_oracle_resample.py::test_oracle_matches_the_stored_compiled_reference_dst2_cubic (seeded the same way)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import build_ref

    C = build_ref.load()
    assert C is not None, "run python oracle/build_ref.py first"
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 2, 5, 4, 6)).astype(np.float32)
    grid = (rng.random((1, 3, 4, 5, 3)) * 9 - 2).astype(np.float32)
    y = C.grid_pull(torch.from_numpy(x), torch.from_numpy(grid), [C.BoundType(4)] * 3, [C.InterpolationType(3)] * 3, True).numpy()
    save("grid_pull_dst2_cubic.npz", x=x, grid=grid, y=y)


def grid_push_ref():
    """monai._C.grid_push / grid_count of the REAL reference (oracle/_ref, CPU): random coordinates reaching outside the field of
    view, the seven bounds, orders 0-3, extrapolate on / off; the numpy restatement (oracle/resample.py) is checked on all 56
    combinations while the subset stored here keeps the fixture small."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import build_ref, resample as orr

    C = build_ref.load()
    assert C is not None, "run python oracle/build_ref.py first"
    rng = np.random.default_rng(3)
    out, n = {}, 0
    shape = (6, 5, 8)
    for bound in (0, 1, 2, 3, 4, 5, 7):
        for order in (0, 1, 2, 3):
            for extrap in (True, False):
                x = rng.standard_normal((1, 2, 5, 6, 7)).astype(np.float32)
                grid = (rng.random((1, 5, 6, 7, 3)) * np.array(shape) * 1.4 - 1.2).astype(np.float32)
                r = C.grid_push(torch.from_numpy(x), torch.from_numpy(grid), list(shape), [C.BoundType(bound)] * 3, [C.InterpolationType(order)] * 3, extrap).numpy()
                np.testing.assert_allclose(orr.grid_push(x, grid, shape, [bound] * 3, [order] * 3, extrap), r, rtol=1e-5, atol=2e-6)
                if order in (1, 3) or (order == 0 and bound in (0, 7)):
                    out[f"c{n}.x"], out[f"c{n}.grid"], out[f"c{n}.y"] = x, grid, r
                    out[f"c{n}.cfg"] = np.array([bound, order, int(extrap), *shape], dtype=np.int64)
                    n += 1
    g = (rng.random((2, 4, 5, 6, 3)) * np.array((5, 6, 7)) * 1.2 - 0.5).astype(np.float32)
    out["count.grid"] = g
    out["count.y"] = C.grid_count(torch.from_numpy(g), [5, 6, 7], [C.BoundType(2)] * 3, [C.InterpolationType(1)] * 3, True).numpy()
    out["n"] = np.array(n)
    # monai._C.grid_grad: all 7 bounds x 8 orders x extrapolate checked against the restatement, a subset stored
    m = 0
    for bound in (0, 1, 2, 3, 4, 5, 7):
        for order in range(8):
            for extrap in (True, False):
                x = rng.standard_normal((1, 2, 6, 5, 7)).astype(np.float32)
                grid = (rng.random((1, 4, 5, 6, 3)) * np.array((6, 5, 7)) * 1.4 - 1.2).astype(np.float32)
                r = C.grid_grad(torch.from_numpy(x), torch.from_numpy(grid), [C.BoundType(bound)] * 3, [C.InterpolationType(order)] * 3, extrap).numpy()
                np.testing.assert_allclose(orr.grid_grad(x, grid, [bound] * 3, [order] * 3, extrap), r, rtol=1e-4, atol=1e-5)
                if (extrap and order in (1, 2, 3, 5)) or (not extrap and order == 1) or (order in (0, 7) and bound == 2):
                    out[f"g{m}.x"], out[f"g{m}.grid"], out[f"g{m}.y"] = x, grid, r
                    out[f"g{m}.cfg"] = np.array([bound, order, int(extrap)], dtype=np.int64)
                    m += 1
    out["n_grad"] = np.array(m)
    # tests/testing_data/1D_BP_bwd.txt: gradients of grid_pull(arange(10), arange(20) + 0.5).sum() (tests/networks/layers/test_grid_pull.py).
    # d/d input is grid_push of ones (= grid_count into the input's shape), d/d grid is grid_grad of the input: the 30-value rows
    # (input and grid both require grad) are golden vectors for exactly these operators.  Transcribed mechanically, keyed by label.
    rows, labels = [], []
    for line in open("/root/reference/tests/testing_data/1D_BP_bwd.txt"):
        if "#" not in line:
            continue
        vals, lab = line.split("#")
        v = [float(t) for t in vals.split(",") if t.strip()]
        if len(v) == 30:
            rows.append(v)
            labels.append(lab.strip())
    assert len(rows) == 56, len(rows)
    out["bp1d_bwd.rows"], out["bp1d_bwd.labels"] = np.asarray(rows, dtype=np.float64), np.asarray(labels)
    # all 224 rows in file order (per (bound, interpolation): input+grid, input only, grid only, none), ragged -> padded with NaN
    allrows, alllabels = [], []
    for line in open("/root/reference/tests/testing_data/1D_BP_bwd.txt"):
        if "#" not in line:
            continue
        vals, lab = line.split("#")
        v = [float(t) for t in vals.split(",") if t.strip()]
        allrows.append(v + [np.nan] * (30 - len(v)))
        alllabels.append(lab.strip())
    assert len(allrows) == 224
    out["bp1d_bwd.all_rows"], out["bp1d_bwd.all_labels"] = np.asarray(allrows, dtype=np.float64), np.asarray(alllabels)
    # monai._C.grid_pull_backward / grid_push_backward / grid_count_backward of the compiled reference on 3-D data: the backward passes of
    # monai_b200's grid_pull / grid_push / grid_count are compositions of the forward operators (checked here on all bounds x orders 0-3 x
    # extrapolate; a subset stored)
    k = 0
    for bound in (0, 1, 2, 3, 4, 5, 7):
        for order in (0, 1, 2, 3):
            for extrap in (True, False):
                B_, I_ = [C.BoundType(bound)] * 3, [C.InterpolationType(order)] * 3
                x = rng.standard_normal((1, 2, 6, 5, 7)).astype(np.float32)
                grid = (rng.random((1, 4, 5, 6, 3)) * np.array((6, 5, 7)) * 1.3 - 1.0).astype(np.float32)
                gout = rng.standard_normal((1, 2, 4, 5, 6)).astype(np.float32)
                xin = rng.standard_normal((1, 2, 4, 5, 6)).astype(np.float32)
                gvol = rng.standard_normal((1, 2, 6, 5, 7)).astype(np.float32)
                gcnt = rng.standard_normal((1, 1, 6, 5, 7)).astype(np.float32)
                tg = lambda a: torch.from_numpy(a).requires_grad_()   # noqa: E731
                pb = C.grid_pull_backward(torch.from_numpy(gout), tg(x), tg(grid), B_, I_, extrap)
                sb = C.grid_push_backward(torch.from_numpy(gvol), tg(xin), tg(grid), B_, I_, extrap)
                cb = C.grid_count_backward(torch.from_numpy(gcnt), tg(grid), B_, I_, extrap)
                bb, oo = [bound] * 3, [order] * 3
                np.testing.assert_allclose(orr.grid_push(gout, grid, x.shape[2:], bb, oo, extrap), pb[0].numpy(), rtol=1e-4, atol=1e-5)
                np.testing.assert_allclose((orr.grid_grad(x, grid, bb, oo, extrap) * gout[..., None]).sum(1), pb[1].numpy(), rtol=1e-4, atol=1e-5)
                np.testing.assert_allclose(orr.grid_pull(gvol, grid, bb, oo, extrap), sb[0].numpy(), rtol=1e-4, atol=1e-5)
                np.testing.assert_allclose((orr.grid_grad(gvol, grid, bb, oo, extrap) * xin[..., None]).sum(1), sb[1].numpy(), rtol=1e-4, atol=1e-5)
                np.testing.assert_allclose(orr.grid_grad(gcnt, grid, bb, oo, extrap)[:, 0], cb.numpy(), rtol=1e-4, atol=1e-5)
                if order in (1, 3) and (extrap or bound == 7):
                    for name, val in (("x", x), ("grid", grid), ("gout", gout), ("xin", xin), ("gvol", gvol), ("gcnt", gcnt), ("pull_dx", pb[0].numpy()),
                                      ("pull_dg", pb[1].numpy()), ("push_dx", sb[0].numpy()), ("push_dg", sb[1].numpy()), ("count_dg", cb.numpy())):
                        out[f"b{k}.{name}"] = val
                    out[f"b{k}.cfg"] = np.array([bound, order, int(extrap)], dtype=np.int64)
                    k += 1
    out["n_bwd"] = np.array(k)
    save("grid_push.npz", **out)


def lazy_inverse():
    """Lazy resampling (Compose(lazy=True): Spacingd o RandAffined composed into one resample) and the inversion of Spacingd through
    Invertd, both from the real reference."""
    from monai.data import MetaTensor
    from monai.transforms import Compose, Invertd, RandAffined, Spacingd

    out = {}
    g = torch.Generator().manual_seed(61)
    img = torch.rand((1, 20, 24, 18), generator=g)
    aff = np.diag([1.25, 1.25, 1.25, 1.0])

    def pipe(lazy):
        c = Compose([Spacingd(keys=["image"], pixdim=(1.0, 1.0, 1.0), mode="bilinear"),
                     RandAffined(keys=["image"], prob=1.0, rotate_range=(0.2,) * 3, scale_range=(0.1,) * 3, translate_range=(5,) * 3, mode="bilinear", padding_mode="border")],
                    lazy=lazy)
        c.transforms[1].set_random_state(seed=0)
        return c

    for tag, lazy in (("eager", False), ("lazy", True)):
        y = pipe(lazy)({"image": MetaTensor(img.clone(), affine=torch.as_tensor(aff))})["image"]
        out[f"{tag}.y"], out[f"{tag}.affine"] = y.numpy(), np.asarray(y.affine)
        out[f"{tag}.n_applied"] = np.array(len(y.applied_operations))
    out["x"], out["x_affine"] = img.numpy(), aff
    # inversion: pre-process, "predict" on the 1 mm grid, bring the prediction back to the 1.25 mm grid
    pre = Spacingd(keys=["image"], pixdim=(1.0, 1.0, 1.0), mode="bilinear")
    d = pre({"image": MetaTensor(img.clone(), affine=torch.as_tensor(aff))})
    pred = MetaTensor(torch.cat([d["image"].as_tensor() * 2.0, 1.0 - d["image"].as_tensor()], 0))   # network outputs are MetaTensors
    for tag, nearest in (("nearest", True), ("bilinear", False)):
        inv = Invertd(keys=["pred"], transform=pre, orig_keys=["image"], nearest_interp=nearest)({"image": d["image"], "pred": pred.clone()})["pred"]
        out[f"inv.{tag}"], out[f"inv.{tag}.affine"] = inv.numpy(), np.asarray(inv.affine)
    out["pre.y"], out["pred"] = d["image"].numpy(), pred.numpy()
    save("lazy_inverse.npz", **out)


def transforms():
    from monai.data import MetaTensor
    from monai.transforms import GaussianSmooth, RandAffined, Spacing, Spacingd

    out = {}
    g = torch.Generator().manual_seed(21)
    img = torch.rand((1, 20, 24, 18), generator=g)
    for tag, aff, pixdim, kw in [
        ("s0", np.diag([1.25, 1.25, 1.25, 1.0]), (1.0, 1.0, 1.0), {}),
        ("s1", np.diag([0.83, 1.5, 1.1, 1.0]), (0.97, 1.23, 0.71), {"mode": "nearest"}),  # tie-free: exact .5 coordinates are round-off dependent
        ("s2", np.array([[0.0, -1.3, 0.0, 10.0], [1.1, 0.0, 0.0, -5.0], [0.0, 0.0, 2.0, 3.0], [0, 0, 0, 1.0]]), (1.0, 1.0, 1.5), {"padding_mode": "zeros"}),
        ("s3", np.diag([1.25, 1.25, 1.25, 1.0]), (1.0, 1.0, 1.0), {"align_corners": True}),
        ("s4", np.diag([1.5, 1.5, 1.5, 1.0]), (1.0, 1.0, 1.0), {"diagonal": True, "padding_mode": "reflection"}),
    ]:
        m = MetaTensor(img.clone(), affine=torch.as_tensor(aff))
        r = Spacing(pixdim=pixdim, **kw)(m)
        out[f"{tag}.affine"], out[f"{tag}.pixdim"], out[f"{tag}.y"], out[f"{tag}.new_affine"] = aff, np.array(pixdim), r.numpy(), r.affine.numpy()
        out[f"{tag}.kw"] = np.array(repr(kw))
    out["img"] = img.numpy()
    # RandAffined, seeded as in SURVEY.md section 8(d) config C4
    img2 = torch.rand((2, 24, 20, 16), generator=g)
    for tag, kw in [
        ("r0", dict(prob=1.0, rotate_range=(0.2,) * 3, scale_range=(0.1,) * 3, translate_range=(5,) * 3, mode="bilinear", padding_mode="border")),
        ("r1", dict(prob=1.0, rotate_range=(0.3, 0.0, 0.1), shear_range=(0.05,) * 6, mode="nearest", padding_mode="zeros")),
        ("r2", dict(prob=1.0, rotate_range=((0.1, 0.4),), scale_range=(0.2,), spatial_size=(16, 28, 12), mode="bilinear", padding_mode="reflection")),
    ]:
        t = RandAffined(keys=["image"], **kw)
        t.set_random_state(seed=0)
        r = t({"image": MetaTensor(img2.clone(), affine=torch.eye(4))})["image"]
        out[f"{tag}.y"], out[f"{tag}.kw"], out[f"{tag}.new_affine"] = r.numpy(), np.array(repr(kw)), r.affine.numpy()
    out["img2"] = img2.numpy()
    for tag, sigma in [("g0", 1.0), ("g1", (1.5, 0.5, 1.0)), ("g2", 0.3)]:
        out[f"{tag}.y"] = GaussianSmooth(sigma=sigma)(img2).numpy()
        out[f"{tag}.sigma"] = np.atleast_1d(np.array(sigma, dtype=np.float64))
    save("transforms.npz", **out)


def post():
    """Activations / AsDiscrete of the real reference on small logits (incl. ties and the goldens of its own unit tests)."""
    from monai.transforms import Activations, AsDiscrete

    out = {}
    g = torch.Generator().manual_seed(33)
    logits = torch.randn((3, 6, 7, 5), generator=g) * 2.0
    logits[:, 0, 0, 0] = 0.5            # three-way tie: argmax must pick channel 0
    logits[1:, 1, 1, 1] = 4.0           # two-way tie between channels 1 and 2
    out["logits"] = logits.numpy()
    out["softmax"] = Activations(softmax=True)(logits).numpy()
    out["sigmoid"] = Activations(sigmoid=True)(logits).numpy()
    out["argmax"] = AsDiscrete(argmax=True)(logits).numpy()
    out["argmax_onehot"] = AsDiscrete(argmax=True, to_onehot=3)(logits).numpy()
    out["threshold"] = AsDiscrete(threshold=0.25)(logits).numpy()
    out["round"] = AsDiscrete(rounding="torchrounding")(torch.tensor([[0.5, 1.5, 2.5, -0.5, -1.5, 0.49, 2.51]])).numpy()
    labels = torch.tensor([[[0.0, 2.0, 1.0], [1.0, 0.0, 2.0]]])
    out["labels"] = labels.numpy()
    out["onehot"] = AsDiscrete(to_onehot=3)(labels).numpy()
    out["sigmoid_threshold"] = AsDiscrete(threshold=0.5)(Activations(sigmoid=True)(logits)).numpy()
    save("post.npz", **out)


from make_golden_cases import PATCH_CASES  # noqa: E402


def _patch_net(p):          # tuple output: same size and a half-resolution head
    return p * 2.0 + 1.0, torch.nn.functional.avg_pool3d(p, 2) - 0.5


def patch():
    """SlidingWindowSplitter grids / patches and PatchInferer(AvgMerger) outputs of the real reference."""
    from monai.inferers import AvgMerger, PatchInferer, SlidingWindowSplitter

    out = {}
    g = torch.Generator().manual_seed(44)
    for name, (shape, kw) in PATCH_CASES.items():
        x = torch.rand(shape, generator=g)
        s = SlidingWindowSplitter(**kw)
        pl = list(s(x))
        out[f"{name}.x"] = x.numpy()
        out[f"{name}.loc"] = np.array([l for _, l in pl], dtype=np.int64)
        out[f"{name}.patches"] = torch.stack([p for p, _ in pl]).numpy()
        out[f"{name}.padded_shape"] = np.array(s.get_padded_shape(x), dtype=np.int64)
    # filter_fn
    x = torch.from_numpy(out["p2d.x"])
    s = SlidingWindowSplitter(filter_fn=lambda patch, loc: loc[0] >= 1 and float(patch.mean()) > 0.4, **PATCH_CASES["p2d"][1])
    out["p2d.filtered_loc"] = np.array([l for _, l in s(x)], dtype=np.int64)
    # PatchInferer: tuple output with a resized head, batches of 3, cropped back to the input extent
    x3 = torch.rand((1, 1, 10, 12, 10), generator=g)
    out["pi.x"] = x3.numpy()
    inf = PatchInferer(splitter=SlidingWindowSplitter(patch_size=4, overlap=0.5, pad_mode="constant"), merger_cls=AvgMerger, batch_size=3)
    a, b = inf(x3, _patch_net)
    out["pi.same"], out["pi.half"] = a.numpy(), b.numpy()
    # dict output with selected keys, no cropping of the padded merge, pre / post processing
    inf = PatchInferer(splitter=SlidingWindowSplitter(patch_size=(4, 5, 4), overlap=(2, 0, 1), pad_mode="constant", pad_value=0.25),
                       batch_size=2, preprocessing=lambda p: p + 1.0, postprocessing=lambda o: {"a": o[0], "b": o[1], "c": o[0] * 0},
                       output_keys=["b", "a"], match_spatial_shape=False)
    d = inf(x3, _patch_net)
    out["pi.dict_b"], out["pi.dict_a"] = d["b"].numpy(), d["a"].numpy()
    save("patch.npz", **out)


def unit_goldens():
    """Golden vectors of the reference's OWN unit tests (SURVEY.md section 8(c)), read mechanically from the TESTS lists of the
    test modules under /root/reference/tests (a stub stands in for the `parameterized` decorator package, which this image
    lacks): Spacing, GaussianSmooth, Activations, AsDiscrete and the 3-D RandAffined cases (seed 123).  Inputs, arguments and
    expected outputs are stored side by side; nothing is recomputed here."""
    import json
    import types

    stub = types.ModuleType("parameterized")

    class _P:
        @staticmethod
        def expand(*a, **k):
            return lambda fn: fn

    stub.parameterized = _P()
    sys.modules["parameterized"] = stub
    import tests.transforms.test_activations as t_act
    import tests.transforms.test_as_discrete as t_dis
    import tests.transforms.test_gaussian_smooth as t_gau
    import tests.transforms.test_rand_affined as t_rad
    import tests.transforms.test_spacing as t_spa

    def arr(v):
        return v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)

    def plain(d):
        out = {}
        for k, v in d.items():
            if k in ("device", "dtype"):
                continue
            if isinstance(v, torch.Tensor):
                v = v.tolist()
            elif isinstance(v, np.ndarray):
                v = v.tolist()
            elif callable(v):
                v = f"<callable {getattr(v, '__name__', 'fn')}>"
            out[k] = list(v) if isinstance(v, tuple) else v
        return out

    out, index = {}, []

    def add(kind, i, init, call, data, expected, extra=None):
        tag = f"{kind}{i}"
        out[f"{tag}.x"], out[f"{tag}.y"] = arr(data).astype(np.float64), arr(expected).astype(np.float64)
        rec = {"tag": tag, "kind": kind, "init": plain(init), "call": plain(call)}
        if extra:
            for k, v in extra.items():
                if isinstance(v, (torch.Tensor, np.ndarray)):
                    out[f"{tag}.{k}"] = arr(v).astype(np.float64)
                else:
                    rec[k] = v
        index.append(rec)

    for i, c in enumerate(t_spa.TESTS):
        if arr(c[1]).size <= 100000:      # the 368x336x368 shape-only case carries no golden values worth 45 M elements
            add("spacing", i, c[0], c[3], c[1], c[4], {"affine": c[2]})
    for i, c in enumerate(t_gau.TESTS):
        add("gauss", i, c[0], {}, c[1], c[2])
    for i, c in enumerate(t_act.TEST_CASES):
        add("act", i, c[0], {}, c[1], c[2])
    for i, c in enumerate(t_dis.TEST_CASES):
        add("disc", i, c[0], {}, c[1], c[2])
    for i, c in enumerate(t_rad.TESTS):
        if isinstance(c[1], dict) and "img" in c[1]:
            add("randaffd", i, c[0], {}, c[1]["img"], c[2] if not isinstance(c[2], dict) else c[2]["img"], {"seed": 123})
    import tests.transforms.test_rand_affine as t_ra

    for i, c in enumerate(t_ra.TESTS):
        if isinstance(c[1], dict) and "img" in c[1]:
            call = {k: v for k, v in c[1].items() if k != "img"}
            add("randaff", i, c[0], call, c[1]["img"], c[2], {"seed": 123})
    out["index"] = np.array(json.dumps(index))
    save("ref_unit_goldens.npz", **out)


if __name__ == "__main__":
    print("reference monai", monai.__version__, "torch", torch.__version__)
    which = sys.argv[1:] or ["planner", "sliding", "nets", "nets_r2", "dynunet", "segresnet", "unetr", "buffered", "resampler", "grid_pull_ref", "grid_pull_ref_dst2", "grid_push_ref", "lazy_inverse", "transforms", "post", "patch", "unit_goldens"]
    for w in which:
        globals()[w]()
