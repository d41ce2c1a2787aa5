"""Pin the plain-C restatements of torchvision nms / scipy linear_sum_assignment (oracle/oracle_kernels.c)
against (a) the committed known-answer vectors and (b) torchvision / scipy black-box,
through their answers on seeded random trials stored in tests/golden/nms_torchvision.npz and lap_scipy.npz
(`PYTHONPATH=. python tests/test_oracle_thirdparty.py` in the repository root regenerates both with the installed binaries)."""
import os

import numpy as np
import pytest
import torch

import oracle
from conftest import GOLDEN


@pytest.fixture(scope="module")
def kat():
    return np.load(os.path.join(GOLDEN, "thirdparty.npz"))


def test_nms_known_answers(kat):
    for t in range(5):
        boxes = torch.from_numpy(kat[f"nms{t}.boxes"])
        scores = torch.from_numpy(kat[f"nms{t}.scores"])
        cls = torch.from_numpy(kat[f"nms{t}.cls"])
        for thr in (0.5, 0.75):
            keep = oracle.batched_nms(boxes, scores, cls, thr)
            assert keep.tolist() == kat[f"nms{t}.{thr}.keep"].tolist()


def test_lap_known_answers(kat):
    for t in range(8):
        r, c = oracle.lap(kat[f"lap{t}.cost"])
        assert r.tolist() == kat[f"lap{t}.row"].tolist()
        assert c.tolist() == kat[f"lap{t}.col"].tolist()


NMS_TV = os.path.join(GOLDEN, "nms_torchvision.npz")


def _nms_trials():
    """(boxes, scores, cls, thr) of the black-box trials: clustered boxes, many exact score ties."""
    g = torch.Generator().manual_seed(123)
    for trial in range(60):
        n = int(torch.randint(1, 400, (1,), generator=g))
        ctr = torch.rand(max(n // 8, 1), 2, generator=g) * 300 - 30
        c = ctr[torch.randint(0, ctr.shape[0], (n,), generator=g)] + torch.randn(n, 2, generator=g) * 3
        wh = torch.rand(n, 2, generator=g) * 30 + 10
        boxes = torch.cat([c - wh / 2, c + wh / 2], 1)
        scores = torch.rand(n, generator=g)
        scores[torch.randint(0, n, (n // 4 + 1,), generator=g)] = 0.5     # many exact ties
        cls = torch.randint(0, 5, (n,), generator=g).float()
        yield boxes, scores, cls, (0.3, 0.5, 0.75)[trial % 3]


def test_nms_blackbox_vs_torchvision():
    tv = np.load(NMS_TV)
    for trial, (boxes, scores, cls, thr) in enumerate(_nms_trials()):
        assert float(boxes.double().sum()) == float(tv[f"{trial}.box_sum"]), f"trial {trial}: inputs differ from the stored ones"
        got = oracle.batched_nms(boxes, scores, cls, thr)
        assert got.tolist() == tv[f"{trial}.batched_keep"].tolist(), f"trial {trial}"
        assert oracle.nms(boxes, scores, thr).tolist() == tv[f"{trial}.keep"].tolist()


def test_nms_empty_and_single():
    assert oracle.batched_nms(torch.zeros(0, 4), torch.zeros(0), torch.zeros(0), 0.5).numel() == 0
    assert oracle.nms(torch.tensor([[0., 0., 1., 1.]]), torch.tensor([0.3]), 0.5).tolist() == [0]


LAP_SP = os.path.join(GOLDEN, "lap_scipy.npz")


def _lap_trials():
    """Cost matrices of the black-box trials: random shapes, heavy ties, float32-rounded values."""
    rng = np.random.default_rng(7)
    for trial in range(80):
        r, c = int(rng.integers(1, 60)), int(rng.integers(1, 60))
        cost = rng.random((r, c))
        if trial % 4 == 0:
            cost = np.round(cost * 4) / 4            # heavy ties
        if trial % 7 == 0:
            cost = cost.astype(np.float32).astype(np.float64)
        yield cost


def test_lap_blackbox_vs_scipy():
    sp = np.load(LAP_SP)
    for trial, cost in enumerate(_lap_trials()):
        assert float(cost.sum()) == float(sp[f"{trial}.cost_sum"]), f"trial {trial}: inputs differ from the stored ones"
        ga, gb = oracle.lap(cost)
        assert ga.tolist() == sp[f"{trial}.row"].tolist() and gb.tolist() == sp[f"{trial}.col"].tolist(), f"trial {trial} shape {cost.shape}"


if __name__ == "__main__":
    import torchvision
    from torchvision.ops import boxes as tvb
    out = {}
    for trial, (boxes, scores, cls, thr) in enumerate(_nms_trials()):
        out[f"{trial}.box_sum"] = np.float64(boxes.double().sum())
        out[f"{trial}.batched_keep"] = tvb._batched_nms_coordinate_trick(boxes, scores, cls, thr).numpy().astype(np.int16)
        out[f"{trial}.keep"] = torchvision.ops.nms(boxes, scores, thr).numpy().astype(np.int16)
    np.savez_compressed(NMS_TV, **out)
    from scipy.optimize import linear_sum_assignment
    out = {}
    for trial, cost in enumerate(_lap_trials()):
        a, b = linear_sum_assignment(cost)
        out[f"{trial}.cost_sum"], out[f"{trial}.row"], out[f"{trial}.col"] = np.float64(cost.sum()), a.astype(np.int8), b.astype(np.int8)
    np.savez_compressed(LAP_SP, **out)
