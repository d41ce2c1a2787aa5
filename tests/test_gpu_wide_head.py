"""The drop-in VID head on frames that keep more than 512 proposals (the reference's list is unbounded without a maximal_limit):
TSCDHeadB200.forward reruns such a call on the wide tier from the CAFM memory the call started with, stays there for the
video's resume=True calls and returns to the default tier at the next resume=False call.  Compared with TSCDHead.forward built
from the same state dict.  An explicit kwargs['max_proposals'] never escalates."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "baseline"))
import ref_runner  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not ref_runner.available(), reason="reference package not installed (baseline/_ref)")]


def _heads(extra=None):
    from tscd_b200.head import make_head_class
    ref_runner.install(cpu_redirect=False)
    from yolox.models.tscd_head import TSCDHead
    args = dict(ref_runner.VID_L_ARGS, **(extra or {}))
    mk = lambda cls_: cls_(30, 1.0, in_channels=[256, 512, 1024], heads=4, defualt_p=30, defulat_pre=750, pre_nms=0.75,  # noqa: E731
                           sim_thresh=0.75, ave=True, **args)
    torch.manual_seed(3)
    ref = mk(TSCDHead)
    ref.initialize_biases(1e-2)
    sd = ref.state_dict()
    for k in range(3):     # objectness pushed up: most of the 1344 anchors of a 256 x 256 frame pass the 0.001 filter
        sd[f"obj_preds.{k}.bias"] = sd[f"obj_preds.{k}.bias"] + 4.6
        sd[f"cls_preds.{k}.weight"] = sd[f"cls_preds.{k}.weight"] * 3.0
    mine = mk(make_head_class())
    mine.load_state_dict(sd, strict=True)
    ref.load_state_dict(sd, strict=True)
    return ref.cuda().eval(), mine.cuda().eval()


def _inputs(F, H, shift):
    g = torch.Generator().manual_seed(11)
    return [torch.randn(F, c, H // s, H // s, generator=g).cuda() + shift for c, s in ((256, 8), (512, 16), (1024, 32))]


def test_vid_head_escalates_to_the_wide_tier():
    from test_gpu_reference import _match
    from tscd_b200.weights import timing_signal_1d
    ref, mine = _heads()
    F, Lf, H = 6, 1, 256
    imgs = torch.zeros(F, 3, H, H).cuda()
    tot_m = tot = 0
    kmax_seen = []
    for call, resume in enumerate((False, True, False)):
        te = timing_signal_1d(torch.arange(call * Lf, (call + 1) * Lf), 256).cuda()
        xs = _inputs(F, H, 0.05 * call)
        with torch.no_grad():
            r_res, r_ori = ref(xs, None, imgs, te, nms_thresh=0.5, lframe=Lf, gframe=F - Lf, resume=resume)
            m_res, m_ori = mine(xs, None, imgs, te, nms_thresh=0.5, lframe=Lf, gframe=F - Lf, resume=resume)
        kmax_seen.append((mine._b200_on_wide, mine._b200_state.kmax))
        for f in range(Lf):
            for got, want in ((m_res[f], r_res[f]), (m_ori[f], r_ori[f])):
                assert (got is None) == (want is None)
                a, b = _match(got, want)
                tot_m += a
                tot += b
    print(f"wide drop-in head vs reference: detections {tot_m}/{tot}, tiers {kmax_seen}")
    assert kmax_seen[0][0] and kmax_seen[1][0] and kmax_seen[0][1] > 512      # escalated, and stayed wide on resume
    assert tot > 100 and tot_m / tot >= 0.97


def test_explicit_max_proposals_still_raises():
    from tscd_b200.weights import timing_signal_1d
    _, mine = _heads(dict(max_proposals=64))
    F, H = 6, 256
    with torch.no_grad(), pytest.raises(RuntimeError, match="capacity of 64"):
        mine(_inputs(F, H, 0.0), None, torch.zeros(F, 3, H, H).cuda(), timing_signal_1d(torch.arange(1), 256).cuda(),
             lframe=1, gframe=F - 1)
