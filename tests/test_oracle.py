"""Pins the oracle (oracle/) against (a) cv2, (b) the golden fixtures produced by
the unmodified reference (tests/golden/make_golden.py).  CPU only."""
import hashlib

import numpy as np
import pytest

import frames
from oracle import host_ref as H


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# The fixtures were recorded with the oracle's torch-CPU executor on one host.  Its float32 convolutions round differently with
# the CPU's vector width and thread count (a few float32 ulps; its float32 vs float64 gap on the detector is 1e-4 / 7e-7 relative),
# so executor outputs are compared within these bounds, while the host code, fed the recorded network outputs, must match exactly.
DET_ROW_RTOL = 1e-5                  # detector rows: |d| <= DET_ROW_RTOL * (1 + |v|)
KPS_NET_TOL_PX, KPS_NET_TOL_SCORE = 2e-4, 2e-5      # twice test_student_executor_fp64_tie_breaker's float32 vs float64 bound
RUN_TOL_PX, RUN_TOL_SCORE = 5e-4, 2e-5              # whole run(): landmarks and boxes in frame pixels


class _Replay:
    """Stands in for an oracle executor Session: returns recorded network outputs in call order."""

    def __init__(self, outputs):
        self.outputs = list(outputs)

    def run(self, x):
        return self.outputs.pop(0)


def _recorded_det_raw(g, t):
    """The detector output of frame t as far as the fixture keeps it: every row scoring over 0.25 (NMS reads rows over 0.5)."""
    raw = np.zeros((15120, 16), np.float32)
    raw[g["f%d_det_cand_idx" % t]] = g["f%d_det_cand_rows" % t]
    return raw


@pytest.mark.parametrize("shape,dst", [
    ((273, 410), (640, 426)), ((1080, 1920), (640, 360)), ((2160, 3840), (640, 360)),
    ((214, 214), (256, 256)), ((97, 97), (256, 256)), ((300, 301), (256, 256)),
    ((720, 1280), (640, 360)), ((617, 617), (256, 256)), ((256, 256), (256, 256)),
    ((33, 57), (256, 256)), ((1000, 999), (256, 256)),
])
def test_resize_matches_cv2(shape, dst):
    import cv2
    rng = np.random.default_rng(shape[0] * 7 + dst[0])
    src = rng.integers(0, 256, size=shape + (3,), dtype=np.uint8)
    ref = cv2.resize(src, dst)
    got = H.resize_linear_u8(src, dst[0], dst[1])
    assert np.array_equal(ref, got)


def test_letterbox_matches_reference_golden(golden):
    for name, fr in [("test1", frames.load_test1()), ("canvas640", frames.canvas_640())]:
        g = golden(name)
        assert sha(fr) == str(g["f0_frame_sha"])
        x, rec = H.letterbox(fr)
        assert sha(x) == str(g["f0_letterbox_sha"])
        assert np.allclose(rec, g["f0_recover"], rtol=0, atol=0)


@pytest.fixture(scope="module")
def ref_nets():
    from oracle.faceana_ref import DetectorRef, LandmarkRef
    return DetectorRef(), LandmarkRef()


def test_detector_restated_matches_golden(golden, ref_nets):
    det, _ = ref_nets
    for name, fr in [("test1", frames.load_test1()), ("uhd4k_top16", frames.frame_4k())]:
        g = golden(name)
        raw, recover, _ = det.raw(fr)
        raw = np.asarray(raw).reshape(15120, 16)
        cand = g["f0_det_cand_idx"]
        assert np.array_equal(np.where(raw[:, 4] > 0.25)[0], cand)
        ref = g["f0_det_cand_rows"]
        assert (np.abs(raw[cand] - ref) <= DET_ROW_RTOL * (1 + np.abs(ref))).all(), np.abs(raw[cand] - ref).max()
        kept, idx = H.detect_post(raw, recover)
        assert np.array_equal(idx, g["f0_det_keep_idx"])
        kept, idx = H.detect_post(_recorded_det_raw(g, 0), recover)
        assert np.array_equal(idx, g["f0_det_keep_idx"])


def test_crop_and_landmarks_match_golden(golden, ref_nets):
    det, kps = ref_nets
    for name, fr, topk in [("test1", frames.load_test1(), 5), ("uhd4k_top5", frames.frame_4k(), 5)]:
        g = golden(name)
        boxes = det(fr)
        boxes = H.sort_and_filter(boxes, 1600, topk)
        for i, b in enumerate(boxes):
            crop, detail = H.crop_face(fr, b.copy())
            assert np.array_equal(crop, g["f0_crops"][i])
            assert list(detail) == list(g["f0_details"][i])
        xy, sc = kps.forward_crops(g["f0_crops"][:2])
        assert np.abs(xy.reshape(len(xy), -1) - g["f0_kps_raw"][:2]).max() * 256 <= KPS_NET_TOL_PX
        assert np.abs(sc - g["f0_kps_score"][:2]).max() <= KPS_NET_TOL_SCORE


def test_heatmap_decode_matches_graph(ref_nets, golden):
    _, kps = ref_nets
    g = golden("test1")
    crop = g["f0_crops"][0]
    x = crop.transpose(2, 0, 1).astype(np.float32)[None] / np.float32(255.)
    hm_name = [n.outputs[0] for n in kps.net.graph.nodes if n.name == "/student/hm/Conv"][0]
    (out, score), kept = kps.net.run(x, keep={hm_name})
    xy, sc = H.heatmap_decode(kept[hm_name][0].numpy())
    assert np.array_equal(xy.reshape(-1), np.asarray(out).reshape(-1))
    assert np.array_equal(sc, np.asarray(score).reshape(-1))


def test_faceana_restated_matches_reference_video(golden):
    """Whole run() incl. track-state, EMA and One-Euro smoothing over a 6-frame clip."""
    from oracle.faceana_ref import FaceAnaRef
    from golden.make_golden_frames import video_frames
    g = golden("video1080")
    live, replay = FaceAnaRef(), FaceAnaRef()
    for t, fr in enumerate(video_frames()):
        n = int(g["f%d_res_n" % t])
        res = live.run(fr.copy())
        assert len(res) == n
        if res:
            assert np.abs(np.stack([r["kps"] for r in res]) - g["f%d_res_kps" % t]).max() <= RUN_TOL_PX
            assert np.abs(np.stack([r["scores"] for r in res]) - g["f%d_res_scores" % t]).max() <= RUN_TOL_SCORE
            assert np.abs(np.stack([r["box"] for r in res]) - g["f%d_res_box" % t]).max() <= RUN_TOL_PX
        # the same frame through the host code with the networks replaced by the outputs recorded from the reference
        replay.det.net = _Replay([[_recorded_det_raw(g, t)]] if "f%d_det_cand_idx" % t in g else [])
        replay.kps.net = _Replay(zip(g["f%d_kps_raw" % t], g["f%d_kps_score" % t]) if "f%d_kps_raw" % t in g else [])
        res = replay.run(fr.copy())
        assert len(res) == n and not replay.det.net.outputs and not replay.kps.net.outputs
        if res:
            assert np.array_equal(np.stack([r["kps"] for r in res]).astype(np.float32), g["f%d_res_kps" % t])
            assert np.array_equal(np.stack([r["scores"] for r in res]), g["f%d_res_scores" % t])
            assert np.allclose(np.stack([r["box"] for r in res]), g["f%d_res_box" % t], rtol=0, atol=0)


def test_detector_graph_cross_check_cv2_dnn(ref_nets):
    """Independent executor for the detector graph: OpenCV's dnn module."""
    import cv2
    det, _ = ref_nets
    from oracle.faceana_ref import DET_ONNX
    net = cv2.dnn.readNetFromONNX(DET_ONNX)
    x, _ = H.letterbox(frames.load_test1())
    net.setInput(x)
    y = net.forward().reshape(15120, 16)
    mine = np.asarray(det.net.run(x)[0]).reshape(15120, 16)
    assert np.abs(y - mine).max() < 2e-3
    assert np.array_equal(np.where(y[:, 4] > 0.5)[0], np.where(mine[:, 4] > 0.5)[0])


def test_student_executor_fp64_tie_breaker():
    """SURVEY 8c item 4: kps_student.onnx has a single independent executor here (cv2.dnn cannot import it), so the same
    executor run in float64 is the tie-breaker reference: the float32 oracle every parity test compares against must sit
    within a small fraction of the 1e-3 px budget of the float64 result, arg-max decisions included."""
    import torch
    import frames
    from oracle.onnx_exec import Session
    from oracle.faceana_ref import LandmarkRef
    import os
    path = os.path.join(os.path.dirname(__file__), "..", "peppa_pig_face_landmark_b200", "pretrained", "kps_student.onnx")
    crops = frames.crop_variants(3)
    s64 = Session(path, dtype=torch.float64)
    xy32, sc32 = LandmarkRef().forward_crops(crops)
    for i, c in enumerate(crops):
        o, k = s64.run(c.transpose(2, 0, 1)[None].astype(np.float64) / 255.0)
        dpx = np.abs(np.asarray(o).reshape(98, 2) - np.asarray(xy32[i], np.float64)).max() * 256
        dsc = np.abs(np.asarray(k).reshape(-1) - np.asarray(sc32[i], np.float64)).max()
        assert dpx < 1e-4 and dsc < 1e-5, (i, dpx, dsc)
