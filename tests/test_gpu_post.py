"""GPU parity of the fused resize + NMS + PAF + greedy + assembly kernels (caffe_rtpose_b200/csrc/post.cu)
through the C ABI, against the oracle (which tests/test_oracle.py pins to the reference's own CUDA kernels).
Everything here is bit-exact."""
import os

import numpy as np
import pytest

from caffe_rtpose_b200 import engine, synth
from oracle import orc

pytestmark = pytest.mark.gpu


def oracle_parse(model, maps8, net_w, net_h, disp_w, disp_h, start, gap, thr=None, params=None):
    full = orc.imresize(maps8, net_h, net_w, start, gap)
    t, p = orc.default_params(model)
    peaks = orc.nms(full, orc.num_parts(model), orc.max_peaks(model), t if thr is None else thr)
    cnt, joints = orc.connect(model, full, peaks, disp_w, disp_h, params or p)
    return full, peaks, cnt, joints


@pytest.mark.parametrize("model,net_w,net_h,S,n_people", [
    (engine.COCO_18, 320, 176, 1, 8), (engine.MPI_15, 240, 176, 1, 5), (engine.COCO_18, 320, 176, 3, 6),
    (engine.COCO_18, 656, 368, 1, 24), (engine.MPI_15, 496, 368, 2, 12)])
def test_parse_stage_bit_exact(model, net_w, net_h, S, n_people):
    eng = engine.PoseEngine(model, net_w, net_h, 2 * net_w, 2 * net_h, num_scales=S, start_scale=1.0, scale_gap=0.15,
                            precision=engine.PREC_FP32_SIMT, max_batch=2)
    scenes = []
    for seed in (1, 2):
        people = synth.make_people(model, n_people, net_w, net_h, seed=seed, drop_prob=0.15)
        scenes.append(synth.make_maps(model, people, net_w, net_h, num_scales=S, start_scale=1.0, scale_gap=0.15, seed=seed))
    eng.forward_maps(np.concatenate(scenes))
    for i, maps8 in enumerate(scenes):
        _, opk, ocnt, oj = oracle_parse(model, maps8, net_w, net_h, 2 * net_w, 2 * net_h, 1.0, 0.15)
        cnt, joints, peaks = eng.fetch(i)
        assert opk[:, 0, 0].max() <= eng.max_peaks
        assert np.array_equal(peaks, opk)
        assert cnt == ocnt and cnt >= n_people // 2
        assert np.array_equal(joints, oj)
        assert eng.json(joints, 1.0) == orc.json_text(oj, eng.num_parts, 1.0)
    eng.close()


@pytest.mark.parametrize("name", ["coco", "coco_s3", "mpi"])
def test_golden_fixtures(name, golden_dir):
    g = np.load(os.path.join(golden_dir, "parse_%s.npz" % name))
    model, net_w, net_h, disp_w, disp_h, S, _ = [int(v) for v in g["meta"]]
    eng = engine.PoseEngine(model, net_w, net_h, disp_w, disp_h, num_scales=S, start_scale=float(g["start_scale"]),
                            scale_gap=float(g["scale_gap"]), precision=engine.PREC_FP32_SIMT)
    eng.nms_layer.SetThreshold(float(g["nms_threshold"]))
    eng.forward_maps(g["maps"])
    cnt, joints, peaks = eng.fetch(0)
    assert np.array_equal(peaks, g["peaks"]) and cnt == len(g["joints"]) and np.array_equal(joints, g["joints"])
    assert eng.json(joints) == str(g["json"])
    eng.close()


def test_layer_setters_change_behaviour():
    model, net_w, net_h = engine.COCO_18, 320, 176
    eng = engine.PoseEngine(model, net_w, net_h, 640, 352, num_scales=2, start_scale=1.0, scale_gap=0.3,
                            precision=engine.PREC_FP32_SIMT)
    assert (eng.nms_layer.GetMaxPeaks(), eng.nms_layer.GetNumParts(), eng.nms_layer.type()) == (64, 18, "Nms")
    assert abs(eng.nms_layer.GetThreshold() - 0.05) < 1e-7 and eng.resize_layer.type() == "ImResize"
    people = synth.make_people(model, 6, net_w, net_h, seed=9)
    maps8 = synth.make_maps(model, people, net_w, net_h, num_scales=2, start_scale=1.0, scale_gap=0.25, seed=9)
    eng.resize_layer.SetScaleGap(0.25)
    eng.nms_layer.SetThreshold(0.3)
    eng.set_connect_params(4, 0.5, 0.06, 9)
    assert abs(eng.resize_layer.GetScaleGap() - 0.25) < 1e-7 and eng.resize_layer.GetStartScale() == 1.0
    _, p = orc.default_params(model)
    prm = orc.ConnectParams(4, 0.5, 0.06, 9, 1)
    _, opk, ocnt, oj = oracle_parse(model, maps8, net_w, net_h, 640, 352, 1.0, 0.25, thr=0.3, params=prm)
    eng.forward_maps(maps8)
    cnt, joints, peaks = eng.fetch(0)
    assert np.array_equal(peaks, opk) and cnt == ocnt and np.array_equal(joints, oj)
    eng.close()


def test_nms_quirks_on_gpu():
    """border exclusion, strict >, score>0 filter, width-for-height aliasing, >max_peaks: count unclamped, first
    max_peaks kept in raster order, consumers clamp (documented extension)."""
    model, net_w, net_h = engine.COCO_18, 320, 176
    rng = np.random.default_rng(5)
    maps8 = rng.normal(0, 0.3, (1, 57, net_h // 8, net_w // 8)).astype(np.float32)  # noise: hundreds of peaks per part
    eng = engine.PoseEngine(model, net_w, net_h, 640, 352, precision=engine.PREC_FP32_SIMT)
    eng.forward_maps(maps8)
    cnt, joints, peaks = eng.fetch(0)
    full, opk, ocnt, oj = oracle_parse(model, maps8, net_w, net_h, 640, 352, 1.0, 0.3)
    assert opk[:, 0, 0].max() > 64          # the case the reference leaves undefined
    assert np.array_equal(peaks, opk)       # count unclamped + first 64 in raster order, bit-exact
    assert cnt == ocnt and np.array_equal(joints, oj)
    eng.close()


def test_empty_scene():
    eng = engine.PoseEngine(engine.MPI_15, 240, 176, 480, 352, precision=engine.PREC_FP32_SIMT)
    eng.forward_maps(np.zeros((1, 44, 22, 30), np.float32))
    cnt, joints, peaks = eng.fetch(0)
    assert cnt == 0 and not peaks.any() and eng.json(joints) == '{\n"version":0.1,\n"bodies":[\n]\n}\n'
    eng.close()
