"""CPU tests that PIN THE ORACLE (SURVEY.md section 8c) before anything trusts it:

  * graph table            == tests/golden/netspec_*.json parsed from the reference prototxts
  * model descriptors      == the reference's own modelDescriptorFactory.cpp
  * im2col                 == the reference's own im2col_cpu                                  bit-exact
  * connectLimbs / COCO    == the reference's own functions on seeded scenes                  bit-exact
  * MAX pooling            == upstream Caffe known-answer vector (test_pooling_layer.cpp:49-120)
  * convolution            vs a naive direct loop at 1e-4 (the bar of test_convolution_layer.cpp:231-265)
  * INTER_AREA             == committed cv2 fixtures (tests/golden/area_cv2.npz)               bit-exact
  * stage-level goldens    == tests/golden/parse_*.npz (peaks, joints, subset, JSON)          bit-exact
ImResize/NMS are pinned against what the reference's own CUDA kernels computed (test_reference_cuda_kernels_equal_oracle).
What the reference's own code computes on each test's inputs is stored in tests/golden/ref_host.npz and, for the CUDA kernels,
ref_cuda.npz (tools/gen_ref_golden.py runs it, compiled from the reference sources into oracle/_ref, on the cases of
oracle/refcases.py that these tests take their inputs from).
"""
import json
import os

import numpy as np
import pytest

from caffe_rtpose_b200 import synth
from oracle import orc
from oracle import refcases as rc

MODELS = [(orc.COCO_18, "coco"), (orc.MPI_15, "mpi")]
REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_host.npz"))


@pytest.mark.parametrize("model,name", MODELS)
def test_graph_matches_prototxt_fixture(model, name, golden_dir):
    spec = json.load(open(os.path.join(golden_dir, "netspec_%s.json" % name)))
    mine = orc.Net(model).layers()
    assert len(mine) == len(spec["layers"]) == 183
    for a, b in zip(mine, spec["layers"]):
        assert a["name"] == b["name"] and a["type"] == b["type"]
        assert a["bottom"] == b["bottom"] and [a["top"]] == b["top"]
        if a["type"] == "Convolution":
            assert (a["num_output"], a["kernel_size"], a["pad"], a["stride"]) == (
                b["num_output"], b["kernel_size"], b["pad"], b["stride"])
            assert b["weight_filler"] == {"type": "gaussian", "std": "0.01"}
        if a["type"] == "Pooling":
            assert (a["kernel_size"], a["stride"], a["pad"], b["pool"]) == (b["kernel_size"], b["stride"], b["pad"], "MAX")
    nms = spec["layers"][-1]
    assert nms["num_parts"] == orc.num_parts(model) and nms["max_peaks"] == orc.max_peaks(model)
    assert spec["layers"][-2]["factor"] == 8.0
    # conv table used by the weight generator == oracle's
    assert orc.Net(model).convs() == synth.conv_table(model)


def test_flops_match_baseline():
    assert orc.flops(orc.COCO_18, 368, 656) == 484634285056.0
    assert orc.flops(orc.COCO_18, 736, 992) == 1465723203584.0
    assert orc.flops(orc.MPI_15, 368, 496) == 361694564352.0


@pytest.mark.parametrize("model,name", MODELS)
def test_model_descriptor_vs_reference_code(model, name):
    assert int(REF["md%d_parts" % model]) == orc.num_parts(model)
    assert list(REF["md%d_limb_seq" % model]) == orc.limb_seq(model) == synth._LIMBS[model]
    assert list(REF["md%d_map_idx" % model]) == orc.map_idx(model) == synth._MAPIDX[model]
    ref_names = str(REF["md%d_names" % model]).split("\n")[:-1]
    assert ref_names == [orc.lib().orc_model_map_name(model, i).decode() for i in range(orc.num_maps(model))]


def test_im2col_vs_reference_code():
    rng = np.random.default_rng(0)
    for i, (c, h, w, k, pad) in enumerate(rc.IM2COL_CASES):
        im = rng.standard_normal((c, h, w)).astype(np.float32)
        assert np.array_equal(orc.im2col(im, k, pad), REF["im2col%d" % i])


def test_maxpool_known_answer_upstream():
    # test_pooling_layer.cpp:49-120 (kernel 2, stride 1)
    x = np.tile(np.array([[1, 2, 5, 2, 3], [9, 4, 1, 4, 8], [1, 2, 5, 2, 3]], np.float32), (2, 2, 1, 1))
    y = orc.maxpool(x, 2, 1, 0)
    assert y.shape == (2, 2, 2, 4)
    assert np.array_equal(y, np.tile(np.array([[9, 5, 5, 8], [9, 5, 5, 8]], np.float32), (2, 2, 1, 1)))


def test_maxpool_ceil_dims():
    # pooling_layer.cpp:90-93: ceil -> odd sizes keep the last partial window
    x = np.arange(2 * 5 * 7, dtype=np.float32).reshape(1, 2, 5, 7)
    y = orc.maxpool(x, 2, 2, 0)
    assert y.shape == (1, 2, 3, 4)
    assert y[0, 0, 2, 3] == x[0, 0, 4, 6] and y[0, 0, 0, 0] == x[0, 0, 1, 1]


def _naive_conv(x, w, b, pad):
    n, cin, h, ww = x.shape
    cout, _, k, _ = w.shape
    xp = np.zeros((n, cin, h + 2 * pad, ww + 2 * pad), np.float64)
    xp[:, :, pad:pad + h, pad:pad + ww] = x
    out = np.zeros((n, cout, h + 2 * pad - k + 1, ww + 2 * pad - k + 1), np.float64)
    for o in range(cout):
        for y in range(out.shape[2]):
            for xx in range(out.shape[3]):
                out[:, o, y, xx] = (xp[:, :, y:y + k, xx:xx + k] * w[o]).sum((1, 2, 3)) + b[o]
    return out


@pytest.mark.parametrize("k,pad", [(3, 1), (1, 0), (7, 3)])
def test_conv_vs_naive_loop(k, pad):
    # upstream bar: 1e-4 vs caffe_conv (test_convolution_layer.cpp:231-265, 443-468), Gaussian-filled 2x3x6x4
    rng = np.random.default_rng(k)
    x = rng.standard_normal((2, 3, 6, 4)).astype(np.float32)
    w = rng.standard_normal((4, 3, k, k)).astype(np.float32)
    b = rng.standard_normal(4).astype(np.float32)
    assert np.abs(orc.conv2d(x, w, b, pad) - _naive_conv(x, w, b, pad)).max() < 1e-4


def test_conv_vs_reference_code_same_blas():
    """ConvolutionLayer::Forward_cpu -> forward_cpu_gemm / forward_cpu_bias -> caffe_cpu_gemm (conv_layer.cpp:27-39,
    base_conv_layer.cpp:259-271, 277-279, math_functions.cpp:12-21) compiled from the reference, its cblas_sgemm bound to the SAME
    OpenBLAS the oracle loads: identical calls into an identical library, so the outputs must be bit-identical - including the
    is_1x1_ shortcut, the bias-as-gemm form and batches.  (The BLAS binary itself is third-party and unpinned in the reference.)
    The reference's outputs are stored as a hash of every value plus a fixed sample, computed with OpenBLAS's sgemm kernel
    rc.BLAS_CORE, which tests/conftest.py makes the oracle's OpenBLAS run: there the oracle must reproduce them bit for bit.  Only
    on a CPU that cannot run that kernel (another kernel sums in another order) does the sample have to agree at fp32 rounding
    level instead."""
    blas = orc.find_blas()
    if blas is None or not orc.lib().orc_have_blas():
        pytest.skip("needs an OpenBLAS")
    assert str(REF["conv_blas_core"]) == rc.BLAS_CORE
    exact = rc.cpu_runs_blas_core()
    if exact:
        assert rc.blas_core(blas) == rc.BLAS_CORE, "%s runs its %s kernel (OPENBLAS_CORETYPE=%s); the reference's outputs were recorded with %s" % (
            blas, rc.blas_core(blas), os.environ.get("OPENBLAS_CORETYPE"), rc.BLAS_CORE)
    rng = np.random.default_rng(9)
    for i, (n, cin, h, w, cout, k, pad) in enumerate(rc.CONV_CASES):
        x = rng.standard_normal((n, cin, h, w)).astype(np.float32)
        wt = (rng.standard_normal((cout, cin, k, k)) * np.sqrt(2.0 / (cin * k * k))).astype(np.float32)
        b = rng.standard_normal(cout).astype(np.float32)
        got = orc.conv2d(x, wt, b, pad)
        want = REF["conv%d_val" % i]
        sample = got.reshape(-1)[np.linspace(0, got.size - 1, want.size).astype(np.int64)]
        if exact:
            assert rc.sha(got) == str(REF["conv%d_sha" % i]), (i, float(np.abs(sample - want).max()))
        else:
            assert np.abs(sample - want).max() <= 1e-5 * np.abs(want).max(), (i, float(np.abs(sample - want).max()))


def test_relu():
    x = np.array([-1.5, 0.0, 2.0, -0.0], np.float32)
    orc.lib().orc_relu(x, x.size)
    assert np.array_equal(x, np.array([0, 0, 2, 0], np.float32))


def test_pool_and_relu_vs_reference_code():
    """PoolingLayer::Reshape + Forward_cpu MAX (pooling_layer.cpp:90-105, 151-186) and ReLULayer::Forward_cpu (relu_layer.cpp:15-18)
    compiled from the reference: sizes (ceil mode, clipped last window), first-maximum semantics, -0.0 / NaN-free inputs."""
    rng = np.random.default_rng(3)
    for i, (n, c, h, w, k, s, pad) in enumerate(rc.POOL_CASES):
        x = rng.standard_normal((n, c, h, w)).astype(np.float32)
        x[0, 0, :2, :2] = 0.5          # ties inside one window
        got = orc.maxpool(x, k, s, pad)
        ref = REF["pool%d" % i]
        assert got.shape == ref.shape
        assert np.array_equal(got, ref)
    x = rng.standard_normal(4099).astype(np.float32)
    x[:3] = (0.0, -0.0, -1e-38)
    y = x.copy()
    orc.lib().orc_relu(y, y.size)
    assert np.array_equal(y, REF["relu"])


def test_preprocess_vs_reference_code():
    """process_and_pad_image (rtpose.cpp:239-269), the display scale (:474-479) and the per-scale target size (:509-511) compiled from
    the reference; the INTER_AREA resize between them is OpenCV's (pinned to cv2 by the fixtures above)."""
    targets = [orc.scale_target(nw, nh, start, gap, i) for (nw, nh, start, gap, S) in rc.SCALE_CASES for i in range(S)]
    assert targets == [tuple(t) for t in REF["scale_targets"].tolist()]
    for j, (cols, rows, dw, dh) in enumerate(rc.DISPLAY_CASES):
        assert orc.lib().orc_display_scale(cols, rows, dw, dh) == REF["display_scales"][j]
    seed, fh, fw, net_h, net_w, S, start, gap = rc.PAD_CASE
    img = synth.make_frame(seed, fh, fw)
    out = orc.preprocess(img, net_h, net_w, S, start, gap)
    for i in range(S):
        assert np.array_equal(out[i], REF["pad%d" % i])
    # normalize = 0: the float canvas of the renderers (rtpose.cpp:499)
    assert rc.sha(orc.canvas_from_u8(img)) == str(REF["canvas_u8_sha"])


def test_json_writer_vs_reference_code():
    """The JSON block of displayFrame (rtpose.cpp:1395-1414, `fs << double` formatting) compiled from the reference, byte for byte -
    for the oracle AND for the product's pe_write_json."""
    from caffe_rtpose_b200 import engine
    rng = np.random.default_rng(5)
    for k, (people, parts, scale) in enumerate(rc.JSON_CASES):
        j = rc.json_joints(rng, people, parts)
        want = str(REF["json"][k])
        assert orc.json_text(j, parts, scale) == want
        assert engine.write_json(j, parts, scale) == want


def test_model_default_thresholds_vs_reference_code():
    """warmup()'s model selection (rtpose.cpp:212-229) compiled from the reference: the NMS / connect thresholds each model starts with."""
    for model in (orc.MPI_15, orc.COCO_18):
        thr, score, inter = [float(v) for v in REF["defaults%d_f" % model]]
        cnt, above = [int(v) for v in REF["defaults%d_i" % model]]
        othr, p = orc.default_params(model)
        assert (othr, p.min_subset_cnt, p.min_subset_score, p.inter_threshold, p.inter_min_above) == (thr, cnt, score, inter, above)


def test_render_dispatch_vs_reference_code():
    """render() (rtpose.cpp:271-300) compiled from the reference with recording launchers: for every --part_to_show value of both
    models (and past the last view) the oracle picks the same launcher with the same `part`, googly / num_parts_accum arguments."""
    for m, model in enumerate((orc.MPI_15, orc.COCO_18)):
        for p2s in range(0, 48):
            for googly in (0, 1):
                got = np.zeros(3, np.int32)
                orc.lib().orc_render_dispatch(model, p2s, googly, got)
                assert list(got) == list(REF["render_dispatch"][m, p2s, googly]), (model, p2s, googly)


def test_inter_area_vs_cv2_fixture(golden_dir):
    d = np.load(os.path.join(golden_dir, "area_cv2.npz"))
    n = len([k for k in d.files if k.startswith("src")])
    assert n >= 6
    for i in range(n):
        dst = d["dst%d" % i]
        assert np.array_equal(orc.resize_area(d["src%d" % i], dst.shape[0], dst.shape[1]), dst)


def test_inter_area_live_cv2():
    cv2 = pytest.importorskip("cv2")
    img = synth.make_frame(3, 180, 320)
    # (184, 248): one axis enlarges -> OpenCV's fixed-point bilinear "area mode"; (200, 400): both enlarge
    for dh, dw in [(92, 164), (80, 140), (90, 160), (60, 160), (184, 248), (200, 400)]:
        assert np.array_equal(orc.resize_area(img, dh, dw), cv2.resize(img, (dw, dh), interpolation=cv2.INTER_AREA))


def test_scale_targets():
    # SURVEY section 8d C3: 656x368 @ {1, .85, .70} -> 656x368, 560x320, 464x272
    assert [orc.scale_target(656, 368, 1.0, 0.15, i) for i in range(3)] == [(656, 368), (560, 320), (464, 272)]
    assert [synth.scale_geometry(656, 368, 1.0, 0.15, i)[:2] for i in range(3)] == [(656, 368), (560, 320), (464, 272)]


def test_preprocess_pad_and_normalise():
    img = synth.make_frame(1, 90, 160)
    out = orc.preprocess(img, 48, 96, 2, 1.0, 0.3)
    assert out.shape == (2, 3, 48, 96)
    r0 = orc.resize_area(img, 48, 96)
    assert np.array_equal(out[0], (r0.transpose(2, 0, 1).astype(np.float32) / np.float32(256) - np.float32(0.5)))
    tw, th = orc.scale_target(96, 48, 1.0, 0.3, 1)
    assert (tw, th) == (80, 48) or (tw, th) == (80, 34 + 14)  # 16*ceil(67.2/16)=80, 16*ceil(33.6/16)=48
    padw = (96 - tw) // 2
    assert np.all(out[1][:, :, :padw] == 0) and np.all(out[1][:, :, padw + tw:] == 0)


@pytest.mark.parametrize("name", ["coco", "coco_s3", "mpi"])
def test_stage_goldens(name, golden_dir):
    g = np.load(os.path.join(golden_dir, "parse_%s.npz" % name))
    model, net_w, net_h, disp_w, disp_h, S, _ = [int(v) for v in g["meta"]]
    full = orc.imresize(g["maps"], net_h, net_w, float(g["start_scale"]), float(g["scale_gap"]))
    peaks = orc.nms(full, orc.num_parts(model), orc.max_peaks(model), float(g["nms_threshold"]))
    assert np.array_equal(peaks, g["peaks"])
    cnt, joints, subset = orc.connect(model, full, peaks, disp_w, disp_h, want_subset=True)
    assert cnt == len(g["joints"]) and cnt >= 3
    assert np.array_equal(joints, g["joints"]) and np.array_equal(subset, g["subset"])
    assert orc.json_text(joints, orc.num_parts(model)) == str(g["json"])


@pytest.mark.parametrize("model,net_w,net_h,n", rc.CONNECT_CASES)
def test_connect_vs_reference_code(model, net_w, net_h, n):
    for seed in rc.CONNECT_SEEDS:
        people = synth.make_people(model, n, net_w, net_h, seed=seed, drop_prob=0.2)
        maps = synth.make_maps(model, people, net_w, net_h, seed=seed)
        full = orc.imresize(maps, net_h, net_w, 1.0, 0.3)
        thr, p = orc.default_params(model)
        peaks = orc.nms(full, orc.num_parts(model), orc.max_peaks(model), thr)
        assert peaks[:, 0, 0].max() <= orc.max_peaks(model)
        cnt, joints, subset = orc.connect(model, full, peaks, 2 * net_w, 2 * net_h, want_subset=True)
        key = "connect_m%d_%dx%d_n%d_s%d" % (model, net_w, net_h, n, seed)
        assert cnt == int(REF[key + "_cnt"]) and cnt >= n // 2
        assert np.array_equal(joints, REF[key + "_joints"]) and np.array_equal(subset, REF[key + "_subset"])


def test_connect_special_cases_vs_reference_code():
    """nA==0 / nB==0 singleton rows, duplicate check (COCO only), nothing at all."""
    for model, net_w, net_h in rc.SPECIAL_NETS:
        P, mp = orc.num_parts(model), orc.max_peaks(model)
        thr, p = orc.default_params(model)
        people = synth.make_people(model, 5, net_w, net_h, seed=5, drop_prob=0.0)
        for i, drop in enumerate(rc.special_drops(P)):
            ppl = [{k: v for k, v in q.items() if k not in drop} for q in people]
            maps = synth.make_maps(model, ppl, net_w, net_h, seed=1)
            full = orc.imresize(maps, net_h, net_w, 1.0, 0.3)
            peaks = orc.nms(full, P, mp, thr)
            a = orc.connect(model, full, peaks, net_w, net_h, want_subset=True)
            key = "special_m%d_d%d" % (model, i)
            assert a[0] == int(REF[key + "_cnt"]) and np.array_equal(a[1], REF[key + "_joints"]) and np.array_equal(a[2], REF[key + "_subset"])


@pytest.mark.parametrize("S", rc.CPM_SCALES)
def test_reference_cuda_kernels_equal_oracle(S):
    """Pins the oracle's ImResize/NMS restatement to the reference's OWN kernels (imresize_layer.cu, nms_layer.cu) compiled for
    sm_100a.  What they computed on a B200 for these inputs is stored in tests/golden/ref_cuda.npz: the peaks blob, and the
    SHA-256 of the full-resolution maps."""
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_cuda.npz"))
    model, net_w, net_h = rc.CPM_NET
    rng = np.random.default_rng(S)
    for kind in ("scene", "noise"):
        if kind == "scene":
            people = synth.make_people(model, 7, net_w, net_h, seed=S)
            maps8 = synth.make_maps(model, people, net_w, net_h, num_scales=S, start_scale=1.0, scale_gap=0.15, seed=S)
        else:
            maps8 = rng.normal(0, 0.5, (S, 57, net_h // 8, net_w // 8)).astype(np.float32)
        full = orc.imresize(maps8, net_h, net_w, 1.0, 0.15)
        key = "cpm_S%d_%s" % (S, kind)
        assert full.shape == (57, net_h, net_w) and rc.sha(full) == str(ref[key + "_full_sha"])
        for thr in rc.CPM_THRESHOLDS:
            assert np.array_equal(orc.nms(full, 18, 64, thr), ref["%s_thr%g_peaks" % (key, thr)])


def test_nms_quirks():
    """strict >, border exclusion, score>0 filter, width-for-height window bound (nms_layer.cu:79)."""
    H, W = 20, 40
    m = np.zeros((2, H, W), np.float32)
    m[0, 5, 5] = 1.0
    m[0, 5, 6] = 1.0            # tie with neighbour -> neither is a peak (strict >)
    m[0, 10, 10] = 0.9
    m[0, 9, 10] = -5.0          # negative neighbour ignored in the centroid (score > 0)
    m[0, 10, 11] = 0.3
    m[0, 0, 20] = 2.0           # border row: never a peak
    m[0, H - 2, 30] = 0.8       # bottom interior row: window rows H..H+1 alias channel 1 rows 0..1
    m[1, 0, 30] = 0.4
    pk = orc.nms(m, 1, 8, 0.05)
    assert pk[0, 0, 0] == 2
    x, y, s = pk[0, 1]
    assert s == np.float32(0.9) and y == 10 and abs(x - (10 * 0.9 + 11 * 0.3) / 1.2) < 1e-6
    x, y, s = pk[0, 2]
    assert s == np.float32(0.8) and abs(y - ((H - 2) * 0.8 + H * 0.4) / 1.2) < 1e-5  # aliased row pulled y down


def test_nms_count_unclamped_and_first_max_peaks_kept():
    H, W = 16, 64
    m = np.zeros((2, H, W), np.float32)
    for i in range(10):
        m[0, 3 + (i % 2) * 6, 4 + 5 * i] = 0.5 + 0.01 * i
    pk = orc.nms(m, 1, 4, 0.05)
    assert pk[0, 0, 0] == 10                     # total, not clamped (nms_layer.cu:110)
    assert [int(round(v)) for v in pk[0, 1:, 1]] == [3, 3, 3, 3]  # raster order: the y=3 row first


def test_json_format():
    j = np.zeros((1, 18, 3), np.float32)
    j[0, 0] = (618.56, 289.597, 0.950805)
    t = orc.json_text(j, 18, 0.5)
    assert t.startswith('{\n"version":0.1,\n"bodies":[\n{\n"joints":[1237.12,579.194,0.950805,0,0,0,')
    assert t.endswith("]\n}]\n}\n")
    assert orc.json_text(np.zeros((0, 18, 3), np.float32), 18) == '{\n"version":0.1,\n"bodies":[\n]\n}\n'


def test_warp_affine_vs_cv2_fixture(golden_dir):
    d = np.load(os.path.join(golden_dir, "warp_cv2.npz"))
    n = len([k for k in d.files if k.startswith("src")])
    assert n >= 5
    for i in range(n):
        dst = d["dst%d" % i]
        out, s = orc.display_image(d["src%d" % i], dst.shape[1], dst.shape[0])
        assert s == float(d["scale%d" % i]) and np.array_equal(out, dst)


def test_warp_affine_live_cv2():
    cv2 = pytest.importorskip("cv2")
    for (sh, sw, dw, dh) in [(108, 192, 128, 72), (48, 64, 128, 72), (72, 128, 128, 72), (100, 100, 128, 72)]:
        img = synth.make_frame(5, sh, sw)
        out, s = orc.display_image(img, dw, dh)
        M = np.eye(2, 3)
        M[0, 0] = M[1, 1] = s
        ref = cv2.warpAffine(img, M, (dw, dh), flags=cv2.INTER_CUBIC, borderMode=cv2.BORDER_CONSTANT, borderValue=(0, 0, 0))
        assert np.array_equal(out, ref)
    same, s = orc.display_image(synth.make_frame(1, 72, 128), 128, 72)   # scale 1: identity
    assert s == 1.0 and np.array_equal(same, synth.make_frame(1, 72, 128))


# ---- renderers (render() rtpose.cpp:271-300, renderFunctions.cu): GPU-only in the reference, so the CPU suite holds
# regression vectors of the restatement + its invariants; the bit-level pin against the reference's own kernels
# (oracle/_ref/libref_render.so) is tests/test_gpu_render.py.
@pytest.mark.parametrize("name", ["coco", "mpi"])
def test_render_goldens(name, golden_dir):
    g = np.load(os.path.join(golden_dir, "parse_%s.npz" % name))
    r = np.load(os.path.join(golden_dir, "render_%s.npz" % name))
    model, net_w, net_h, disp_w, disp_h, S, _ = [int(v) for v in g["meta"]]
    full = orc.imresize(g["maps"], net_h, net_w, float(g["start_scale"]), float(g["scale_gap"]))
    canvas = np.full((3, disp_h, disp_w), 96.0, np.float32)
    for key in r.files:
        part, googly = int(key.split("_")[0][1:]), int(key.split("_")[1][1:])
        img = orc.canvas_to_u8(orc.render(model, canvas, net_w, net_h, full, g["joints"], len(g["joints"]), part, bool(googly)))
        assert (img != r[key]).any(2).mean() < 1e-4, key   # libm sinf/cosf may move a border pixel between glibc builds


def test_render_invariants():
    model, w, h = orc.COCO_18, 96, 64
    canvas = orc.canvas_from_u8(synth.make_frame(3, h, w))
    joints = np.zeros((1, 18, 3), np.float32)
    # no people / no confident joint: the skeleton view leaves the canvas untouched (renderFunctions.cu:1006, :437)
    assert np.array_equal(orc.render(model, canvas, 48, 32, None, joints, 0, 0), canvas)
    assert np.array_equal(orc.render(model, canvas, 48, 32, None, joints, 1, 0), canvas)
    # one limb (neck-right shoulder): an ellipse around the segment in the limb's colour, alpha 0.5, plus two joint discs
    joints[0, 1] = (30, 30, 1.0)
    joints[0, 2] = (60, 30, 1.0)
    out = orc.render(model, canvas, 48, 32, None, joints, 1, 0)
    changed = np.argwhere((out != canvas).any(0))
    assert len(changed) > 0 and changed[:, 1].min() >= 29 and changed[:, 1].max() <= 61 and abs(changed[:, 0].mean() - 30) < 1
    mid = out[:, 30, 45]
    assert np.allclose(mid, 0.5 * canvas[:, 30, 45] + 0.5 * np.array([0, 0, 255], np.float32))   # colour 0 = (r 255, g 0, b 0)
    # float canvas -> uint8: int(v + 0.5) with clamping (rtpose.cpp:1291-1293)
    c = np.zeros((3, 1, 4), np.float32)
    c[0, 0] = (-3.0, 0.49, 0.5, 300.0)
    assert orc.canvas_to_u8(c)[0, :, 0].tolist() == [0, 0, 1, 255]
    with pytest.raises(ValueError):
        orc.render(model, canvas, 48, 32, np.zeros((57, 32, 48), np.float32), joints, 1, 40)


def test_bench_golden_is_the_oracle(golden_dir):
    """tests/golden/bench_c2.npz (what the -m gpu parity tests compare the benched configuration with) is the oracle's
    own output: frame 3 re-derived live.  Another host CPU may pick another BLAS kernel (different summation order),
    so the live maps are compared at the level two fp32 implementations differ by, and the decisions (noise maps,
    ~800 peaks) may move by a few near-ties."""
    g = np.load(os.path.join(golden_dir, "bench_c2.npz"))
    i = 3
    seed, h, w = [int(v) for v in g["frames"][i]]
    net = orc.Net(orc.COCO_18)
    net.set_weights(synth.make_weights(orc.COCO_18, "he"))
    cnt, joints, peaks, maps = net.process_frame(synth.make_frame(seed, h, w), 368, 656)
    sub = [int(c) for c in g["map_subset"]]
    assert np.abs(maps[:, sub] - g["maps_sub%d" % i]).max() / float(g["maps_absmax%d" % i]) < 1e-5
    assert np.abs(peaks[:, 0, 0] - g["peaks%d" % i][:, 0, 0]).max() <= 2
    assert abs(cnt - int(g["cnt%d" % i])) <= 2
