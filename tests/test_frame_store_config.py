"""CPU test: the frame store (tscd_b200.frames) -- the slot rules of frames.check_clip_args shared by
AggregationStage.ingest_frames and forward_clips, the store's single-buffer layout and byte count, -1 for never-written slots,
and the C layout of the new argument structs (compiled with gcc against include/tscd_b200.h)."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT

C, D, KMAX = 25, 256, 30


def _store(frames=10, kmax=KMAX, num_classes=C, dtype=torch.float16):
    from tscd_b200 import frames as fr
    return fr.FrameStore(frames, kmax, num_classes, D, dtype, device="cpu")


def _check(store, slots, L=None, kmax=KMAX, num_classes=C, dim=D, dtype=torch.float16, num_frames=None):
    from tscd_b200.frames import check_clip_args
    check_clip_args(store, slots, kmax, num_classes, dim, dtype, L=L, num_frames=num_frames)


def test_valid_arguments_pass():
    s = _store()
    _check(s, [3, 1, 0, 9], num_frames=4)                                    # ingest
    _check(s, np.array([5]), num_frames=1)
    _check(s, torch.tensor([2, 4], dtype=torch.int32), num_frames=2)
    _check(s, [[0, 1, 2, 3], [4, 5, 6, 7]], L=2)                             # clips
    _check(s, [[0, 0, 0, 9]], L=1)                                           # a slot may repeat inside a clip (padding)
    _check(s, torch.tensor([[1, 2, 3]]), L=3)


def test_store_layout_and_bytes():
    from tscd_b200 import frames as fr
    n, W = 7, 7 + C
    s = _store(frames=n)
    assert fr.FrameStore.bytes_per_slot(KMAX, C) == 8 + KMAX * (6 * D + 8 + 4 * W) == 50168
    pad = s.flat.numel() - n * fr.FrameStore.bytes_per_slot(KMAX, C)
    assert s.flat.dtype == torch.uint8 and 0 <= pad < 16 * 8                 # eight fields, each rounded up to 16 bytes
    fields = dict(count=(n,), status=(n,), bank_cls=(n, KMAX, D), bank_reg=(n, KMAX, D), bank_edge=(n, KMAX, D),
                  bank_score=(n, KMAX), sel_idx=(n, KMAX), sel_rows=(n, KMAX, W))
    base = s.flat.data_ptr()
    ends = []
    for name, shape in fields.items():
        t = getattr(s, name)
        assert tuple(t.shape) == shape and t.is_contiguous(), name
        assert t.untyped_storage().data_ptr() == s.flat.untyped_storage().data_ptr(), name     # one allocation
        assert (t.data_ptr() - base) % 16 == 0, name
        ends.append((t.data_ptr() - base, t.data_ptr() - base + t.numel() * t.element_size()))
    ends.sort()
    assert all(a[1] <= b[0] for a, b in zip(ends, ends[1:]))                 # fields do not overlap
    assert s.bank_cls.dtype == torch.float16 and s.sel_rows.dtype == torch.float32 and s.sel_idx.dtype == torch.int32
    assert _store(dtype=torch.bfloat16).bank_edge.dtype == torch.bfloat16
    with pytest.raises(RuntimeError, match="16-bit"):
        _store(dtype=torch.float32)


def test_never_written_slots_read_minus_one():
    s = _store(frames=5)
    assert s.count.tolist() == [-1] * 5
    assert s.status.tolist() == [0] * 5


@pytest.mark.parametrize("name,kw,expect", [("kmax", dict(kmax=40), "kmax = 40"), ("classes", dict(num_classes=30), "num_classes = 30"),
                                            ("dim", dict(dim=128), "dim = 128"), ("dtype", dict(dtype=torch.bfloat16), "bfloat16")])
def test_store_of_another_shape(name, kw, expect):
    s = _store()
    for L in (None, 2):
        with pytest.raises(RuntimeError, match=expect):
            _check(s, [0, 1] if L is None else [[0, 1]], L=L, **kw)
    with pytest.raises(RuntimeError, match="allocate FrameStore"):
        _check(s, [[0, 1]], L=1, **kw)


def test_wrong_shapes():
    s = _store()
    with pytest.raises(RuntimeError, match="1-D"):
        _check(s, [[0, 1]], num_frames=2)
    with pytest.raises(RuntimeError, match="one slot per frame"):
        _check(s, [0, 1, 2], num_frames=2)
    with pytest.raises(RuntimeError, match=r"\[B, F\]"):
        _check(s, [0, 1, 2], L=1)
    with pytest.raises(RuntimeError, match=r"\[B, F\]"):
        _check(s, np.zeros((0, 4), np.int64), L=1)
    with pytest.raises(RuntimeError, match="1 <= L <= F"):
        _check(s, [[0, 1]], L=3)
    with pytest.raises(RuntimeError, match="1 <= L <= F"):
        _check(s, [[0, 1]], L=0)


def test_out_of_range_host_slots():
    s = _store(frames=6)
    with pytest.raises(RuntimeError, match=r"slot\(s\) \[6\] outside \[0, 6\)"):
        _check(s, [0, 6], num_frames=2)
    with pytest.raises(RuntimeError, match=r"\[-1\]"):
        _check(s, [[0, 1], [2, -1]], L=1)
    with pytest.raises(RuntimeError, match="outside"):
        _check(s, torch.tensor([[7, 0]]), L=1)


def test_duplicate_slots_in_one_ingest():
    s = _store()
    with pytest.raises(RuntimeError, match=r"duplicate frame slot\(s\) \[2\]"):
        _check(s, [2, 0, 2], num_frames=3)
    _check(s, [[2, 0, 2]], L=1)                       # clips may repeat a slot


def test_keys_per_clip_limit_same_message_as_forward():
    s = _store(kmax=512)
    _check(s, [[0] * 128], L=1, kmax=512)             # 65536 keys: the limit itself
    with pytest.raises(RuntimeError, match="129 frames x 512 proposals per frame = 66048 keys per clip exceed the attention "
                                           "kernels' capacity of 65536; lower SelectionConfig.max_proposals"):
        _check(s, [[0] * 129], L=1, kmax=512)


def test_device_slot_tensor_rules_without_reading_values():
    """A device tensor is checked for dtype / shape only (its values stay on the device: capture-safe).  Without a GPU this
    exercises the same branch through a stand-in that reports is_cuda."""
    class FakeCuda(torch.Tensor):
        @property
        def is_cuda(self):
            return True
    s = _store()
    good = torch.tensor([[99, -5]], dtype=torch.int32).as_subclass(FakeCuda)         # out of range, but never read
    _check(s, good, L=1)
    with pytest.raises(RuntimeError, match="int32"):
        _check(s, torch.tensor([[0, 1]], dtype=torch.int64).as_subclass(FakeCuda), L=1)
    with pytest.raises(RuntimeError, match="contiguous"):
        _check(s, torch.zeros(4, 2, dtype=torch.int32).t().as_subclass(FakeCuda), L=1)


def test_struct_sizes_match_header():
    from tscd_b200 import _lib
    pairs = [("tscd_frame_store", _lib.FrameStoreC), ("tscd_frame_scatter_args", _lib.FrameScatterArgs),
             ("tscd_clip_assemble_args", _lib.ClipAssembleArgs)]
    offs = [("tscd_clip_assemble_args", "row_cap", _lib.ClipAssembleArgs), ("tscd_clip_assemble_args", "status", _lib.ClipAssembleArgs),
            ("tscd_frame_scatter_args", "status", _lib.FrameScatterArgs)]
    body = "".join(f'printf("%zu\\n", sizeof({c}));' for c, _ in pairs)
    body += "".join(f'printf("%zu\\n", offsetof({c}, {f}));' for c, f, _ in offs)
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "tscd_b200.h"\nint main(){' + body + 'return 0;}'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    want = [ctypes.sizeof(t) for _, t in pairs] + [getattr(t, f).offset for _, f, t in offs]
    assert got == want


def test_frame_slot_error_code_is_bound():
    from tscd_b200 import _lib
    assert _lib.TSCD_ERR_FRAME_SLOT == -5 and "never written" in _lib._ERR[-5]
    header = open(os.path.join(ROOT, "include", "tscd_b200.h")).read()
    assert "#define TSCD_ERR_FRAME_SLOT (-5)" in header
