"""CPU tests of the two capacity tiers: the default tier (max_proposals <= 512) keeps its limits and messages, the wide tier
(513 .. 2048) has its own, and CAFMState widening keeps a video's CAFM memory row for row."""
import pytest
import torch

from tscd_b200 import ops, selection, stage


def _cfg(C, **sel):
    return stage.StageConfig(num_classes=C, selection=selection.SelectionConfig(mode="B", use_pre_nms=False, **sel))


def test_constants_mirror_the_header():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "tscd_b200.h")) as f:
        assert f"#define TSCD_MAX_PROPOSALS {selection.MAX_PROPOSALS}" in f.read()
    assert selection.DEFAULT_TIER_MAX == 512 and selection.MAX_PROPOSALS == 2048
    assert ops.NMS_MAX_CAP == 16384 and ops.NMS_WIDE_CAP == 65536


def test_default_tier_limits_and_messages_unchanged():
    stage.validate_config(_cfg(30, max_proposals=512))                 # VID-L default: 512 x 30 = 15360 rows
    with pytest.raises(RuntimeError, match=r"exceed the NMS capacity of 16384; lower max_proposals / maximal_limit to <= 204"):
        stage.validate_config(_cfg(80, maximal_limit=500))
    with pytest.raises(RuntimeError, match=r"minimal_limit / maximal_limit = 0 / 600 exceed max_proposals = 512"):
        stage.validate_config(_cfg(5, maximal_limit=600))
    with pytest.raises(RuntimeError, match=r"exceed the NMS capacity of 16384"):
        stage.validate_config(_cfg(40, max_proposals=512))              # 512 x 40 > 16384 stays a default-tier error


def test_wide_tier_limits():
    stage.validate_config(_cfg(30, max_proposals=2048))                # 61440 final-NMS rows
    stage.validate_config(_cfg(32, max_proposals=2048))                # exactly 65536
    stage.validate_config(_cfg(80, max_proposals=800))                 # 64000
    with pytest.raises(RuntimeError, match=r"wide tier.*NMS capacity of 65536; lower max_proposals / maximal_limit to <= 1638"):
        stage.validate_config(_cfg(40, max_proposals=2048))
    with pytest.raises(RuntimeError, match=r"max_proposals = 2049: the CAFM chain holds at most 2048"):
        stage.validate_config(_cfg(30, max_proposals=2049))
    with pytest.raises(RuntimeError, match=r"max_proposals = 0"):
        stage.validate_config(_cfg(30, max_proposals=0))
    assert not selection.is_wide(512) and selection.is_wide(513)
    assert selection.SelectionConfig(mode="B", max_proposals=2048).max_keep(6804) == 2048


def test_cafm_state_widening_on_cpu():
    s = stage.CAFMState(2, 4, dim=8, device="cpu")
    g = torch.Generator().manual_seed(1)
    s.flat.copy_(torch.randn(s.flat.shape, generator=g))
    s.n.copy_(torch.tensor([3, 4], dtype=torch.int32))
    w = s.widened(10)
    assert w.kmax == 10 and w.slots == 2 and w.dim == 8
    assert w.n.tolist() == [3, 4] and torch.equal(w.time, s.time)
    for f in ("out", "edge", "reg", "cls", "nreg", "ncls"):
        a, b = getattr(s, f), getattr(w, f)
        assert torch.equal(b[:, :4], a), f
        assert not b[:, 4:].any(), f
    assert w.flat.data_ptr() != s.flat.data_ptr()
    with pytest.raises(RuntimeError, match="kmax"):
        s.widened(3)
