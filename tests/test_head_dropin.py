"""CPU test (runs where the reference package is available: installed under baseline/_ref, or a checkout): the drop-in head
keeps the reference's constructor, state_dict keys/shapes (strict load) and rejects unsupported configurations loudly."""
import os
import sys

import pytest

TOOLS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
if TOOLS not in sys.path:
    sys.path.insert(0, TOOLS)
import ref_shim  # noqa: E402

REF = ref_shim.reference_root()
pytestmark = pytest.mark.skipif(REF is None, reason="reference package not installed (baseline/_ref)")


def _install():
    ref_shim.install()


def test_dropin_head_state_dict_and_config():
    _install()
    import make_goldens as mg
    from yolox.models.tscd_head import TSCDHead
    from tscd_b200.head import make_head_class, stage_config_from_head
    cls = make_head_class()
    ref = TSCDHead(25, 1.0, in_channels=[256, 512, 1024], heads=4, **mg.MORE_ARGS)
    mine = cls(25, 1.0, in_channels=[256, 512, 1024], heads=4, **mg.MORE_ARGS)
    assert [(k, tuple(v.shape)) for k, v in ref.state_dict().items()] == [(k, tuple(v.shape)) for k, v in mine.state_dict().items()]
    mine.load_state_dict(ref.state_dict(), strict=True)
    cfg = stage_config_from_head(mine)
    assert cfg.selection.mode == "B" and cfg.selection.minimal_limit == 50 and cfg.selection.maximal_limit == 500
    assert cfg.selection.use_pre_nms is False and cfg.conf_sim_thresh == 0.99 and cfg.num_classes == 25
    with pytest.raises(RuntimeError):        # unsupported configurations are rejected when the head is BUILT
        cls(25, 1.0, in_channels=[256, 512, 1024], heads=4, **dict(mg.MORE_ARGS, agg_type="localagg"))
    with pytest.raises(RuntimeError, match="max_proposals"):
        cls(25, 1.0, in_channels=[256, 512, 1024], heads=4, **dict(mg.MORE_ARGS, maximal_limit=2000))
    # VID TSCD-L: no maximal_limit -> explicit per-frame capacity instead of the anchor count (exps/TSCD_VID/vid_tscd_large.py:39-42)
    vid_args = {k: v for k, v in mg.MORE_ARGS.items() if k not in ("maximal_limit", "conf_sim_thresh")}
    vid = cls(30, 1.0, in_channels=[256, 512, 1024], heads=4, **vid_args)
    vcfg = stage_config_from_head(vid)
    assert vcfg.selection.maximal_limit == 0 and vcfg.selection.max_proposals == 512 and vcfg.selection.max_keep(6804) == 512
    # the weight snapshot is invalidated by a PARENT module's load_state_dict and by .half() / .to()
    import torch
    mine._b200_stage = object()
    torch.nn.Sequential(mine).load_state_dict({"0." + k: v for k, v in ref.state_dict().items()})
    assert mine._b200_stage is None
    mine._b200_stage = object()
    mine.half()
    assert mine._b200_stage is None


def test_exp_file_swaps_head(monkeypatch):
    if not os.path.exists(os.path.join(REF, "exps", "TSCD_OVIS", "ovis_tscd_large.py")):
        pytest.skip("the reference's exp files are not part of the installed package")
    _install()
    monkeypatch.setenv("TSCD_REFERENCE_ROOT", REF)
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("exp_b200", os.path.join(root, "exps_b200", "ovis_tscd_large_b200.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    model = mod.Exp().get_model()
    assert type(model.head).__name__ == "TSCDHeadB200"
    assert type(model).__name__ == "TSCD"
