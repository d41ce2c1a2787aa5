"""CPU tests of VideoStream's host side (tscd_b200/video.py): the argument checks a submit runs before any launch, the frame
map that picks every video frame's detections out of the clip calls (padded tail frames left out), and the ctypes mirror of
the tscd_video_pack argument structs."""
import ctypes
import os
import random
import subprocess
import tempfile

import pytest
import torch

from conftest import ROOT


def _item(n, L=8, G=24, first=0, seed=0):
    from tscd_b200 import clips
    cl, pa = clips.demo_clips(n, L, G, rng=random.Random(seed))
    return dict(first_frame=first, num_frames=n, clips=cl, paths=pa, ratios=[1.0] * n)


@pytest.mark.parametrize("L,G", [(8, 24), (1, 31)])
def test_frame_map_against_demo_clips(L, G):
    """Every frame of every video length L .. 3 (L + G) (demo_clips needs at least L frames) maps to its first local
    occurrence; the copies of the last frame that pad the tail clip are never picked, and the map is what tools/tscd_demo.py
    keeps after trimming: clip-major local frames, the first n of them.  Short videos (n <= L + G) have clips of n frames."""
    from tscd_b200 import clips
    from tscd_b200.video import local_frames
    for n in range(L, 3 * (L + G) + 1):
        cl, pa = clips.demo_clips(n, L, G, rng=random.Random(n))
        where = local_frames(cl, pa, n)
        assert len(where) == n
        trimmed = [(c, l) for c in range(len(cl)) for l in range(L)][:n]    # demo: outputs of the clips in order, first n frames
        assert where == trimmed, n
        for f, (c, l) in enumerate(where):
            assert cl[c][l] == f and pa[c][l] == f
        if n <= L + G:                                  # short video: gframe shrinks to n - L
            assert all(len(c) == n for c in cl)


def test_frame_map_rejects_uncovered_frames():
    from tscd_b200.video import local_frames
    with pytest.raises(RuntimeError, match=r"frames \[2\] of the video are not a local frame"):
        local_frames([[0, 1, 2], [1, 0, 2]], [[0], [1]], 3)


def test_group_rejections():
    from tscd_b200.video import check_group
    ok = [_item(20), _item(13, first=20)]
    shapes, where = check_group(ok, slots=2, max_frames=40)
    assert shapes == [(20, 8), (13, 8)] and [len(w) for w in where] == [20, 13]
    with pytest.raises(RuntimeError, match="3 videos for 2 pool slots"):
        check_group(ok + [_item(8, first=33)], slots=2, max_frames=48)
    with pytest.raises(RuntimeError, match=r"video 1: frames \[20, 33\) exceed the 30 frames of a buffer set"):
        check_group(ok, slots=2, max_frames=30)
    bad = _item(13, first=20)
    bad["clips"][1][3] = 13
    with pytest.raises(RuntimeError, match="video 1, clip 1: frame 13 outside the video's 13 frames"):
        check_group([ok[0], bad], slots=2, max_frames=40)
    short = _item(13, first=20)
    short["ratios"] = [1.0] * 12
    with pytest.raises(RuntimeError, match="video 1: 12 ratios for 13 frames"):
        check_group([ok[0], short], slots=2, max_frames=40)
    with pytest.raises(RuntimeError, match="videos 0 and 1 overlap"):
        check_group([ok[0], _item(13, first=19)], slots=2, max_frames=40)
    with pytest.raises(RuntimeError, match="REPP needs 'img_sizes'"):
        check_group(ok, slots=2, max_frames=40, post=object())
    with pytest.raises(RuntimeError, match="no videos"):
        check_group([], slots=2, max_frames=40)


def _host(n, A, hw, row_w=32, pin=False):
    t = (lambda x: x.pin_memory()) if pin else (lambda x: x)
    h = dict(rows=[t(torch.zeros(n, A, row_w, dtype=torch.float16))], objp=[t(torch.zeros(n, A, dtype=torch.float16))])
    for k in ("f_cls", "f_reg", "f_edge"):
        h[k] = [t(torch.zeros(n, 256, a, b, dtype=torch.float16)) for a, b in hw]
    return h


def test_staging_rejections():
    from tscd_b200.video import check_staging
    hw = [(4, 4), (2, 2), (1, 1)]
    A = 21
    with pytest.raises(RuntimeError, match="pinned CPU tensors"):
        check_staging(_host(3, A, hw), 3, A, 32, hw)
    per_level = {"reg": [], "obj": [], "cls": []}
    with pytest.raises(RuntimeError, match="fused-row layout"):
        check_staging(per_level, 3, A, 32, hw)
    if not torch.cuda.is_available():
        return                                           # pinned allocations need the CUDA driver
    h = _host(3, A, hw, pin=True)
    check_staging(h, 3, A, 32, hw)
    with pytest.raises(RuntimeError, match="holds 3 frames, max_frames is 4"):
        check_staging(h, 4, A, 32, hw)


def test_video_pack_struct_layout_matches_header():
    from tscd_b200 import _lib
    pairs = [("tscd_video_pack_call", _lib.VideoPackCall), ("tscd_video_pack_args", _lib.VideoPackArgs)]
    fields = [("tscd_video_pack_args", f) for f, _ in _lib.VideoPackArgs._fields_] + \
             [("tscd_video_pack_call", f) for f, _ in _lib.VideoPackCall._fields_]
    body = "".join(f'printf("%zu\\n", sizeof({c}));' for c, _ in pairs)
    body += "".join(f'printf("%zu\\n", offsetof({c}, {f}));' for c, f in fields)
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "tscd_b200.h"\nint main(){' + body + 'return 0;}'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    want = [ctypes.sizeof(t) for _, t in pairs]
    want += [getattr(_lib.VideoPackArgs, f).offset for _, f in fields[:len(_lib.VideoPackArgs._fields_)]]
    want += [getattr(_lib.VideoPackCall, f).offset for _, f in fields[len(_lib.VideoPackArgs._fields_):]]
    assert got == want
