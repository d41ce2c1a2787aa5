"""REPP tubelet post-processing (SURVEY.md section 8f-3): the step after the aggregation stage in `tscd_demo.py --post`
(tools/tscd_demo.py:286-290) and the VID evaluation recipe.

`REPPB200` keeps the constructor arguments and the `__call__(video_predictions) -> predictions_coco` contract of the
reference's `REPP` class (tools/REPP.py:24-277), and its output bit for bit.  Everything after the parsing of the dicts runs on
the device (csrc/repp.cu): the linking of all frame pairs (tscd_repp_link, one CTA per frame pair), the tubelet chains and the
unmatched singletons (tscd_repp_tubelets), the rescoring, the Gaussian re-coordination of the box tracks and the predictions
table (tscd_repp_emit).  The host reads the valid rows of that table once and builds the output dicts from it.

`REPPB200.from_detections` starts one step earlier, from the stage's packed detections (evalglue.pack_detections packed with the
resize ratios as scales): tscd_repp_prep does what Predictor.to_repp_heavy and the score filter of REPP.__call__ do, so no
per-detection dict is built on the way in.

Exactness: the device sums in the reference's order in fp64 without FMA contraction (see csrc/repp.cu).  The one input it cannot
compute bit-exactly itself, the Gaussian window (scipy.signal.windows.gaussian uses NumPy's exp), is computed here once per call
for the longest possible tubelet; every shorter window is its centred slice.  The box dtype NumPy would give a tubelet's
`np.array([p["bbox"] ...])` (float32 only if every coordinate is a float32, int64 if every one is an int, float64 otherwise) is
passed per detection as kind bits (`box_kind`), since the convolution writes its results in that dtype.

The logistic linking model is read from the reference's pickle (tools/matching_model_logreg.pckl, an sklearn
LogisticRegression over [center_distances_corrected, height_rel, iou, width_rel]) when `weight_path` is given, or passed as
plain numbers (`logreg=dict(features=..., coef=..., intercept=...)`) -- the kernel needs the four coefficients only.
Appearance matching (`descriptor_dist`, needs per-detection embeddings the TSCD tools never produce: `appearance_matching`
is false in tools/yolo_repp_cfg.json) is rejected loudly."""
import ctypes as C
import pickle
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L
from . import ops

_FEATURES = ["center_distances_corrected", "height_rel", "iou", "width_rel"]
_CLF_MODES = {"dot": 0, "max": 1, "dot_plus": 2, "raw": 3}
_KIND_F32, _KIND_INT, _KIND_OTHER = 1, 2, 4


def box_kind(bbox) -> int:
    """Kind bits of one box (include/tscd_b200.h): 1 per float32 coordinate, 2 per integer, 4 per anything else."""
    k = 0
    for v in bbox:
        t = type(v)
        k |= _KIND_F32 if t is np.float32 else _KIND_INT if (t is int or isinstance(v, np.integer)) else _KIND_OTHER
    return k


def gaussian_window(num_frames: int, std: float) -> np.ndarray:
    """The unnormalised window of the longest tubelet a `num_frames` video can have; a length-M tubelet uses its centred slice
    [num_frames - M, num_frames + M - 1), which equals scipy.signal.windows.gaussian(2 * M - 1, std)."""
    from scipy.signal import windows
    return windows.gaussian(2 * num_frames - 1, std=std)


class ReppTable:
    """Predictions of one video on the device: `table` [rows, 8] fp64 = (detection, x, y, w, h, score, category, track id),
    valid rows = `count[0]`; `status[0]` != 0 reports an error of the device steps.  `detection` indexes the REPP detections
    (for the packed input `src` gives their packed rows).  `predictions()` copies the valid rows to the host once and builds the
    reference's output dicts."""

    def __init__(self, table, count, status, image_ids, frame_off=None, src=None):
        self.table, self.count, self.status, self.src = table, count, status, src
        self._image_ids, self._frame_off = image_ids, frame_off

    def predictions(self) -> List[dict]:
        if self.table is None:
            return []
        n, st = (int(x) for x in torch.cat([self.count, self.status]).cpu().tolist())
        _raise_status(st)
        rows = self.table[:n].cpu().numpy()
        if self._frame_off is not None:              # packed input: image ids per frame
            which = np.searchsorted(np.asarray(self._frame_off), rows[:, 0], side="right") - 1
        else:                                        # dict input: image ids per detection
            which = rows[:, 0].astype(np.int64)
        ids = self._image_ids
        return [{"image_id": ids[i], "bbox": r[1:5], "score": r[5], "category_id": int(r[6]), "track_id": int(r[7])}
                for i, r in zip(which.tolist(), rows.tolist())]


def _raise_status(st):
    if st == L.TSCD_ERR_CAPACITY:
        raise RuntimeError("REPPB200: more than 4096 detections in a frame, or an output capacity exceeded")
    if st != 0:
        raise IndexError("REPPB200: a class id or a detection index is out of range")


class REPPB200:
    def __init__(self, min_tubelet_score, add_unmatched, min_pred_score, distance_func, clf_thr, clf_mode,
                 appearance_matching=False, recoordinate=True, recoordinate_std=0.4, weight_path=None, logreg: Optional[dict] = None,
                 num_classes: int = 30, device="cuda"):
        L.lib()                                   # no CPU fallback
        if appearance_matching:
            raise RuntimeError("REPPB200: appearance_matching needs detection embeddings; not produced by the TSCD tools")
        if distance_func not in ("def", "logreg"):
            raise ValueError(f"distance_func not recognized: {distance_func}")
        self.min_tubelet_score, self.add_unmatched, self.min_pred_score = min_tubelet_score, add_unmatched, min_pred_score
        self.distance_func, self.clf_thr, self.clf_mode = distance_func, float(clf_thr), clf_mode
        self.recoordinate, self.recoordinate_std = recoordinate, recoordinate_std
        self.num_classes, self.device = num_classes, device
        self.coef, self.intercept = [0.0] * 4, 0.0
        self._win, self._win_frames = None, 0
        if distance_func == "logreg":
            if clf_mode not in _CLF_MODES:
                raise ValueError("error post_clf")
            if logreg is None:
                if weight_path is None:
                    raise ValueError("REPPB200: distance_func='logreg' needs weight_path or logreg")
                model, feats = pickle.load(open(weight_path, "rb"))
                logreg = dict(features=list(feats), coef=np.asarray(model.coef_).reshape(-1).tolist(),
                              intercept=float(np.asarray(model.intercept_).reshape(-1)[0]))
            if list(logreg["features"]) != _FEATURES:
                raise RuntimeError(f"REPPB200: the linking model must use the features {_FEATURES}, got {logreg['features']}")
            self.coef, self.intercept = [float(c) for c in logreg["coef"]], float(logreg["intercept"])

    # ------------------------------------------------------------------------------------------------------------
    def __call__(self, video_predictions: Dict):
        """REPP.__call__ (tools/REPP.py:245-273).  video_predictions: {frame key: [dict(image_id, bbox [x,y,w,h], bbox_center,
        scores (obj, cls_score, class id))]} as Predictor.to_repp_heavy builds it (tools/val_to_imdb.py:193-218)."""
        keys = list(video_predictions.keys())
        preds = {}
        for fr in keys:                                            # :247-256 low-score filter, one-hot score vectors
            tmp = []
            for p in video_predictions[fr]:
                idx, sc = int(p["scores"][2]), p["scores"][0] * p["scores"][1]
                if sc >= self.min_tubelet_score:
                    if not 0 <= idx < self.num_classes:
                        raise IndexError(f"REPPB200: class id {idx} outside [0, {self.num_classes})")
                    tmp.append((p, idx, float(sc)))
            preds[fr] = tmp
        frames = sorted(keys, key=int)                             # get_video_pairs :84-85 links in sorted order
        off, ids, box64, kind, ctrs, scs, cls = [0], [], [], [], [], [], []
        for fr in frames:
            for p, idx, sc in preds[fr]:
                ids.append(p["image_id"])
                box64.append([float(v) for v in p["bbox"]])
                kind.append(box_kind(p["bbox"]))
                ctrs.append([float(np.float32(v)) for v in p["bbox_center"]])
                scs.append(sc)
                cls.append(idx)
            off.append(len(ids))
        nf, n = len(frames), off[-1]
        if nf < 2 or n == 0:
            return []
        data_off = data_cnt = None
        if keys != frames:                                         # get_tubelets / singletons index preds in insertion order
            start = {fr: off[i] for i, fr in enumerate(frames)}
            data_off, data_cnt = [start[k] for k in keys], [len(preds[k]) for k in keys]
        dev = self.device
        t_box64 = torch.tensor(box64, dtype=torch.float64).to(dev)
        ints = torch.tensor(off + kind + cls + [0, 0], dtype=torch.int32).to(dev)
        frame_off, t_kind, t_cls, nout_status = ints[:nf + 1], ints[nf + 1:nf + 1 + n], ints[nf + 1 + n:nf + 1 + 2 * n], ints[-2:]
        if data_off is not None:
            data = torch.tensor(data_off + data_cnt, dtype=torch.int32).to(dev)
            data_off, data_cnt = data[:nf], data[nf:]
        table, count = self._device(off, frame_off, t_box64.float(), torch.tensor(ctrs, dtype=torch.float32).to(dev),
                                    torch.tensor(scs, dtype=torch.float64).to(dev), t_cls, t_box64, t_kind, data_off, data_cnt, nout_status)
        return ReppTable(table, count, nout_status[1:], ids).predictions()

    # ------------------------------------------------------------------------------------------------------------
    def from_detections(self, packed: torch.Tensor, offsets: torch.Tensor, det_cand: Sequence[int],
                        img_sizes: Sequence[Sequence[int]], image_ids: Sequence) -> ReppTable:
        """REPP of one video straight from evalglue.pack_detections(rows, count, resize ratios) over its frames in order.
        The returned table's `predictions()` equals
        `self({str(f): p for f, p in enumerate(evalglue.repp_predictions(table, offsets, det_cand, img_sizes, image_ids))})`.
        Reads back the per-frame detection counts once (to size the linking workspace) before the final copy."""
        nf, cap, dev = offsets.numel() - 1, packed.shape[0], packed.device
        thr_dt = np.result_type(np.float32(0), self.min_tubelet_score)   # NumPy 2: a Python number adopts float32
        # per frame: det_cand, image (height, width), then frame_off [nf + 1] and the status, read back together
        ints = torch.tensor([int(v) for v in det_cand] + [int(v) for hw in img_sizes for v in hw] + [0] * (nf + 2),
                            dtype=torch.int32).to(dev)
        t_cand, t_size, fo_status = ints[:nf], ints[nf:3 * nf], ints[3 * nf:]
        frame_off, status = fo_status[:nf + 1], fo_status[nf + 1:]
        count_ws, t_cls, t_kind, t_src = (torch.empty(k, dtype=torch.int32, device=dev) for k in (nf, cap, cap, cap))
        t_box, t_ctr = torch.empty(cap, 4, dtype=torch.float32, device=dev), torch.empty(cap, 2, dtype=torch.float32, device=dev)
        t_sc, t_box64 = torch.empty(cap, dtype=torch.float64, device=dev), torch.empty(cap, 4, dtype=torch.float64, device=dev)
        ops.call("tscd_repp_prep", L.ReppPrepArgs, num_frames=nf, num_classes=self.num_classes,
                 thr_f32=int(thr_dt == np.float32), min_tubelet_score=float(self.min_tubelet_score), packed=packed,
                 offsets=offsets, det_cand=t_cand, img_size=t_size, count=count_ws, frame_off=frame_off, bbox=t_box,
                 center=t_ctr, score=t_sc, cls=t_cls, box64=t_box64, kind=t_kind, src=t_src, status=status)
        host = fo_status.cpu().tolist()
        off, st = host[:nf + 1], host[nf + 1]
        _raise_status(st)
        if nf < 2 or off[-1] == 0:
            return ReppTable(None, None, None, image_ids, off, t_src)
        nout_status = torch.zeros(2, dtype=torch.int32, device=dev)
        table, count = self._device(off, frame_off, t_box, t_ctr, t_sc, t_cls, t_box64, t_kind, None, None, nout_status)
        return ReppTable(table, count, nout_status[1:], image_ids, off, t_src)

    # ------------------------------------------------------------------------------------------------------------
    def _window(self, nf):
        if self._win is None or self._win_frames < nf:
            self._win = torch.from_numpy(gaussian_window(nf, self.recoordinate_std * 100 / 40)).to(self.device)
            self._win_frames = nf
        return self._win[self._win_frames - nf:self._win_frames + nf - 1]

    def _device(self, off, frame_off, bbox, center, score, cls, box64, kind, data_off, data_cnt, nout_status):
        """link -> tubelets -> emit for one video; `off` is the host copy of frame_off.  nout_status [2] int32 (zeroed) receives
        the number of valid rows and the status of every step.  Returns (table, count)."""
        nf, n, ncls = len(off) - 1, off[-1], self.num_classes
        dev = bbox.device
        counts = [off[i + 1] - off[i] for i in range(nf)]
        max_det = max(counts)
        ws_pitch = max(1, max(counts[i] * counts[i + 1] for i in range(nf - 1)))
        status = nout_status[1:]
        pairs = torch.empty(nf - 1, max_det, 2, dtype=torch.int32, device=dev)
        pair_count, nodes, ws, tcounts, tub_off, members, single, single_tub, tub_k, row_off = (
            torch.empty(k, dtype=torch.int32, device=dev) for k in (nf - 1, 3 * n, 2 * n + nf + 1, 2, n + 1, n, n, n, n, 2 * n + 1))
        ws_dist = torch.empty(nf - 1, ws_pitch, dtype=torch.float64, device=dev)
        ws_idx = torch.empty(nf - 1, ws_pitch, dtype=torch.int32, device=dev)
        a = L.ReppLinkArgs()
        a.num_frames, a.max_det = nf, max_det
        a.distance_func = 0 if self.distance_func == "def" else 1
        a.clf_mode = _CLF_MODES.get(self.clf_mode, 0)
        a.clf_thr, a.intercept = self.clf_thr, self.intercept
        for i in range(4):
            a.coef[i] = self.coef[i]
        a.frame_off, a.bbox, a.center, a.score, a.cls = ops._p(frame_off), ops._p(bbox), ops._p(center), ops._p(score), ops._p(cls)
        a.pairs, a.pair_count, a.ws_dist, a.ws_idx, a.ws_pitch, a.status = ops._p(pairs), ops._p(pair_count), ops._p(ws_dist), ops._p(ws_idx), ws_pitch, ops._p(status)
        with L.timed("tscd_repp_link"):
            L.check(L.lib().tscd_repp_link(C.byref(a), ops._stream()), "tscd_repp_link")
        ops.call("tscd_repp_tubelets", L.ReppTubeletsArgs, num_frames=nf, max_det=max_det, add_unmatched=int(bool(self.add_unmatched)),
                 cap=n, frame_off=frame_off, data_off=data_off, data_cnt=data_cnt, pairs=pairs, pair_count=pair_count,
                 next=nodes[:n], has_prev=nodes[n:2 * n], tail_of=nodes[2 * n:], ws=ws, counts=tcounts, tub_off=tub_off,
                 members=members, single=single, single_tub=single_tub, status=status)
        tub_score, mem_box = torch.empty(n * ncls, dtype=torch.float64, device=dev), torch.empty(n, 4, dtype=torch.float64, device=dev)
        table = torch.empty(2 * n * ncls, 8, dtype=torch.float64, device=dev)
        ops.call("tscd_repp_emit", L.ReppEmitArgs, num_frames=nf, num_classes=ncls, cap=n, recoordinate=int(bool(self.recoordinate)),
                 min_pred_score=float(self.min_pred_score), window=self._window(nf) if self.recoordinate else None,
                 box64=box64, kind=kind, score=score, cls=cls, counts=tcounts, tub_off=tub_off, members=members, single=single,
                 single_tub=single_tub, tub_score=tub_score, tub_k=tub_k, mem_box=mem_box, row_off=row_off,
                 row_cap=2 * n * ncls, out=table, n_out=nout_status[:1], status=status)
        return table, nout_status[:1]
