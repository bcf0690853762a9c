"""Host-side window tables of the SwinUNETR tensor-core path, checked without a GPU.

`window_plan` turns pad + roll(-shift) + window_partition (swin_unetr.py:596-625) and compute_mask (779-816) into index tables, and
`window_attention_tc_plan` groups the windows by shift-mask pattern for the tcgen05 attention.  Every launch of the Swin stages reads
these tables, so they are compared here with the torch restatement in oracle/networks.py for every (grid, window, shift) that the
network meets at the listed input sizes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from monai_b200 import _kernels as K
from monai_b200.networks.nets.swin_unetr import _get_window_size, window_plan
from oracle import networks as onet

INPUTS = [(64, 64, 64), (96, 96, 96), (128, 128, 128), (96, 64, 64), (160, 96, 64)]
WINDOW, SHIFT = (7, 7, 7), (3, 3, 3)


def _cases():
    """(dims, window, shift) of every Swin block: four stages on the input / 2, / 4, / 8, / 16 grids, unshifted and shifted blocks."""
    seen = []
    for inp in INPUTS:
        for stage in range(1, 5):
            dims = tuple(s // 2**stage for s in inp)
            for shift in ((0, 0, 0), SHIFT):
                case = (dims, *_get_window_size(dims, WINDOW, shift))
                if case not in seen:
                    seen.append(case)
    return seen


CASES = _cases()


def _mask(labels: torch.Tensor) -> torch.Tensor:
    """[nW, n] region labels -> the [nW, n, n] attention mask: -100 where the labels of a pair differ."""
    return torch.where(labels[:, None, :] != labels[:, :, None], -100.0, 0.0)


@pytest.mark.parametrize("dims,ws,ss", CASES, ids=[f"{'x'.join(map(str, d))}-w{'x'.join(map(str, w))}-s{''.join(map(str, s))}" for d, w, s in CASES])
def test_window_plan_matches_the_reference_partition_and_mask(dims, ws, ss):
    src, region, nW, n = window_plan(dims, WINDOW, SHIFT if any(ss) else (0, 0, 0))   # the block's module shift, clamped inside
    S = dims[0] * dims[1] * dims[2]
    pdims = [-(-d // w) * w for d, w in zip(dims, ws)]
    assert n == ws[0] * ws[1] * ws[2] and nW * n == pdims[0] * pdims[1] * pdims[2]
    assert src.dtype == np.int32 and src.shape == (nW * n,)

    # pad -> roll(-shift) -> window_partition of the token ids, -1 on the padding
    ids = torch.arange(S, dtype=torch.float64).reshape(1, *dims, 1)
    ids = F.pad(ids, (0, 0, 0, pdims[2] - dims[2], 0, pdims[1] - dims[1], 0, pdims[0] - dims[0]), value=-1.0)
    if any(ss):
        ids = torch.roll(ids, shifts=tuple(-s for s in ss), dims=(1, 2, 3))
    want = onet._window_partition(ids, ws).reshape(-1).to(torch.int64).numpy()
    np.testing.assert_array_equal(src, want)
    live = np.sort(src[src >= 0])
    np.testing.assert_array_equal(live, np.arange(S))   # every token exactly once

    if not any(ss):
        assert region is None
        sched, reps, ntypes = K.window_attention_tc_plan(region, nW, n)
        assert ntypes == 1 and reps is None
        assert sched[0] == nW and sched[8] == 0 and not sched[1:8].any()
        np.testing.assert_array_equal(sched[16:], np.arange(nW))
        return

    assert region.shape == (nW, n) and region.dtype == np.int32
    got_mask = _mask(torch.from_numpy(region))
    want_mask = onet._compute_mask(pdims, ws, ss).float()
    assert torch.equal(got_mask, want_mask)

    sched, reps, ntypes = K.window_attention_tc_plan(region, nW, n)
    assert 1 <= ntypes <= 8
    assert sched.shape == (16 + nW,) and sched.dtype == np.int32
    counts, starts = sched[:8], sched[8:16]
    assert not counts[ntypes:].any()
    assert counts.sum() == nW
    order = sched[16:]
    np.testing.assert_array_equal(np.sort(order), np.arange(nW))   # each window listed exactly once
    assert reps.shape == (ntypes, n)
    rep_masks = _mask(torch.from_numpy(reps))
    for t in range(ntypes):
        assert counts[t] > 0
        wins = order[starts[t]: starts[t] + counts[t]]
        assert len(wins) == counts[t]
        for w in wins:
            assert torch.equal(rep_masks[t], got_mask[w]), (t, int(w))


def test_the_enumeration_reaches_clamped_partly_shifted_and_small_windows():
    """The cases above include what the network actually launches: windows clamped on some axes only (shift dropped there),
    the unshifted n = 216 window of the 6^3 grid and the n = 64 window of the 4^3 grid."""
    assert any(any(ss) and not all(ss) for _, _, ss in CASES)
    ns = {w[0] * w[1] * w[2] for _, w, _ in CASES}
    assert {343, 216, 64} <= ns
