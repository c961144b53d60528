#!/usr/bin/env python3
"""Record what the reference's own code (oracle/_ref, built by oracle/build_ref.py from the reference sources) computes on the
inputs of the tests that pin the oracle and the engine to it, so that those tests run from the repository alone.

  python tools/gen_ref_golden.py host [DIR]   reference host code (CPU)          -> DIR/ref_host.npz  (default tests/golden)
  python tools/gen_ref_golden.py cuda [DIR]   reference CUDA kernels (needs a GPU) -> DIR/ref_cuda.npz

Each section below builds the inputs of one test from the cases in oracle/refcases.py, which the tests use too, and stores the
reference's answer; large outputs (full-resolution maps, rendered canvases, the float canvas of an image) are stored as the
SHA-256 of their float32 bytes, so the tests still compare bit for bit.  The convolution goes through the reference's cblas_sgemm
call into the OpenBLAS the oracle loads, run with the kernel refcases.BLAS_CORE: its outputs are stored as a hash plus a fixed
sample.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import refcases as rc  # noqa: E402

rc.pin_blas_core()   # before anything loads an OpenBLAS
from caffe_rtpose_b200 import synth  # noqa: E402
from oracle import orc  # noqa: E402


def sha(a):
    return np.array(rc.sha(a))


# ---- host code of the reference (tests/test_oracle.py, tests/test_host_pipeline.py) -------------------------------------------
def gen_host(out_dir):
    R = orc.ref_host()
    assert R is not None and hasattr(R, "ref_handle_keys"), "oracle/_ref/libref_host.so missing: build it from the reference first"
    d = {}
    for model in (orc.MPI_15, orc.COCO_18):
        npart, nlimb = C.c_int(), C.c_int()
        ls, mi = np.zeros(64, np.int32), np.zeros(64, np.int32)
        names = C.create_string_buffer(8192)
        assert R.ref_model_descriptor(model, C.byref(npart), C.byref(nlimb), ls, mi, names, 8192) == 0
        d["md%d_parts" % model] = np.int32(npart.value)
        d["md%d_limb_seq" % model] = ls[:2 * nlimb.value].copy()
        d["md%d_map_idx" % model] = mi[:2 * nlimb.value].copy()
        d["md%d_names" % model] = np.array(names.value.decode())

    rng = np.random.default_rng(0)
    for i, (c, h, w, k, pad) in enumerate(rc.IM2COL_CASES):
        im = rng.standard_normal((c, h, w)).astype(np.float32)
        ref = np.empty((c * k * k, (h + 2 * pad - k + 1) * (w + 2 * pad - k + 1)), np.float32)
        R.ref_im2col(im, c, h, w, k, k, pad, pad, 1, 1, ref)
        d["im2col%d" % i] = ref

    blas = orc.find_blas()
    assert blas and R.ref_load_blas(blas.encode()) == 0
    orc.lib()
    assert rc.blas_core(blas) == rc.BLAS_CORE, (blas, rc.blas_core(blas))
    d["conv_blas_core"] = np.array(rc.BLAS_CORE)
    rng = np.random.default_rng(9)
    for i, (n, cin, h, w, cout, k, pad) in enumerate(rc.CONV_CASES):
        x = rng.standard_normal((n, cin, h, w)).astype(np.float32)
        wt = (rng.standard_normal((cout, cin, k, k)) * np.sqrt(2.0 / (cin * k * k))).astype(np.float32)
        b = rng.standard_normal(cout).astype(np.float32)
        ref = np.full((n, cout, h + 2 * pad - k + 1, w + 2 * pad - k + 1), 3.0, np.float32)
        assert R.ref_conv_forward(x, n, cin, h, w, wt, b.ctypes.data, cout, k, pad, ref) == 0
        d["conv%d_sha" % i], d["conv%d_val" % i] = sha(ref), ref.reshape(-1)[np.linspace(0, ref.size - 1, min(ref.size, rc.CONV_SAMPLE)).astype(np.int64)]

    rng = np.random.default_rng(3)
    for i, (n, c, h, w, k, s, pad) in enumerate(rc.POOL_CASES):
        x = rng.standard_normal((n, c, h, w)).astype(np.float32)
        x[0, 0, :2, :2] = 0.5
        hw = np.zeros(2, np.int32)
        R.ref_maxpool(x, n, c, h, w, k, s, pad, None, hw)
        ref = np.empty((n, c, hw[0], hw[1]), np.float32)
        R.ref_maxpool(x, n, c, h, w, k, s, pad, ref.ctypes.data, hw)
        d["pool%d" % i] = ref
    x = rng.standard_normal(4099).astype(np.float32)
    x[:3] = (0.0, -0.0, -1e-38)
    ref = np.empty_like(x)
    R.ref_relu(x, ref, x.size, 0.0)
    d["relu"] = ref

    targets = []
    for (nw, nh, start, gap, S) in rc.SCALE_CASES:
        for i in range(S):
            tw, th = C.c_int(), C.c_int()
            R.ref_scale_target(nw, nh, start, gap, i, C.byref(tw), C.byref(th))
            targets.append((tw.value, th.value))
    d["scale_targets"] = np.array(targets, np.int32)
    d["display_scales"] = np.array([R.ref_display_scale(*c) for c in rc.DISPLAY_CASES], np.float64)
    seed, fh, fw, net_h, net_w, S, start, gap = rc.PAD_CASE
    img = synth.make_frame(seed, fh, fw)
    for i in range(S):
        tw, th = orc.scale_target(net_w, net_h, start, gap, i)
        ref = np.full((3, net_h, net_w), 7.0, np.float32)
        R.ref_process_and_pad_image(ref, orc.resize_area(img, th, tw), tw, th, net_w, net_h, 1)
        d["pad%d" % i] = ref
    ref = np.empty((3, fh, fw), np.float32)
    R.ref_process_and_pad_image(ref, img, fw, fh, fw, fh, 0)
    d["canvas_u8_sha"] = sha(ref)

    import tempfile
    rng = np.random.default_rng(5)
    texts = []
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ref.json")
        for people, parts, scale in rc.JSON_CASES:
            j = rc.json_joints(rng, people, parts)
            R.ref_write_json(path.encode(), j if j.size else np.zeros(1, np.float32), people, parts, scale)
            texts.append(open(path).read())
    d["json"] = np.array(texts)

    R.ref_model_defaults.argtypes = [C.c_int] + [C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int)]
    for model, parts in ((orc.MPI_15, 15), (orc.COCO_18, 18)):
        thr, cnt, score, inter, above = C.c_float(), C.c_int(), C.c_float(), C.c_float(), C.c_int()
        R.ref_model_defaults(parts, C.byref(thr), C.byref(cnt), C.byref(score), C.byref(inter), C.byref(above))
        d["defaults%d_f" % model] = np.array([thr.value, score.value, inter.value], np.float32)
        d["defaults%d_i" % model] = np.array([cnt.value, above.value], np.int32)

    disp = np.zeros((2, 48, 2, 3), np.int32)
    for m, parts in enumerate((15, 18)):
        for p2s in range(48):
            for googly in (0, 1):
                assert R.ref_render_dispatch(parts, p2s, googly, disp[m, p2s, googly]) == 1
    d["render_dispatch"] = disp   # [0] MPI_15, [1] COCO_18

    for model, net_w, net_h, n in rc.CONNECT_CASES:
        for seed in rc.CONNECT_SEEDS:
            people = synth.make_people(model, n, net_w, net_h, seed=seed, drop_prob=0.2)
            full = orc.imresize(synth.make_maps(model, people, net_w, net_h, seed=seed), net_h, net_w, 1.0, 0.3)
            thr, p = orc.default_params(model)
            peaks = orc.nms(full, orc.num_parts(model), orc.max_peaks(model), thr)
            p0 = orc.ConnectParams(p.min_subset_cnt, p.min_subset_score, p.inter_threshold, p.inter_min_above, 0)
            key = "connect_m%d_%dx%d_n%d_s%d" % (model, net_w, net_h, n, seed)
            c2, j2, s2 = orc.ref_connect(model, full, peaks, 2 * net_w, 2 * net_h, p0)
            d[key + "_cnt"], d[key + "_joints"], d[key + "_subset"] = np.int32(c2), j2, s2

    for model, net_w, net_h in rc.SPECIAL_NETS:
        P, mp = orc.num_parts(model), orc.max_peaks(model)
        thr, p = orc.default_params(model)
        p0 = orc.ConnectParams(p.min_subset_cnt, p.min_subset_score, p.inter_threshold, p.inter_min_above, 0)
        people = synth.make_people(model, 5, net_w, net_h, seed=5, drop_prob=0.0)
        for k, drop in enumerate(rc.special_drops(P)):
            ppl = [{a: v for a, v in q.items() if a not in drop} for q in people]
            full = orc.imresize(synth.make_maps(model, ppl, net_w, net_h, seed=1), net_h, net_w, 1.0, 0.3)
            peaks = orc.nms(full, P, mp, thr)
            key = "special_m%d_d%d" % (model, k)
            c2, j2, s2 = orc.ref_connect(model, full, peaks, net_w, net_h, p0)
            d[key + "_cnt"], d[key + "_joints"], d[key + "_subset"] = np.int32(c2), j2, s2

    # handleKey on random key sequences that keep --part_to_show inside the views this build renders (0..39)
    R.ref_handle_keys.argtypes = [C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    rng = np.random.default_rng(rc.KEY_SEED)
    alphabet = rc.KEY_ALPHABET
    keys_out, f_out, i_out = [], [], []
    for trial in range(rc.KEY_TRIALS):
        while True:
            keys = "".join(alphabet[i] for i in rng.integers(0, len(alphabet), rc.KEY_LENGTH))
            f = (C.c_float * 3)(0.05, 0.4, 0.05)
            i = (C.c_int * 7)(9, 3, 0, 0, 0, 0, 0)
            ok = True
            for ch in keys:
                R.ref_handle_keys((C.c_int * 1)(ord(ch)), 1, 0, f, i)
                ok = ok and 0 <= i[2] <= 39
            if ok:
                break
        keys_out.append(keys)
        f_out.append(list(f))
        i_out.append(list(i))
    d["keys"], d["keys_f"], d["keys_i"] = np.array(keys_out), np.array(f_out, np.float32), np.array(i_out, np.int32)

    path = os.path.join(out_dir, "ref_host.npz")
    np.savez_compressed(path, **d)
    print(path, len(d), "arrays,", os.path.getsize(path), "bytes; BLAS core", d["conv_blas_core"])


# ---- CUDA kernels of the reference (tests/test_oracle.py, tests/test_gpu_render.py) --------------------------------------------
def render_scene(model, net_w, net_h, disp_w, disp_h, n_people, seed):
    """The scene of tests/test_gpu_render.py::scene, parsed by the oracle (the engine's parse stage is bit-identical to it)."""
    people = synth.make_people(model, n_people, net_w, net_h, seed=seed)
    maps8 = synth.make_maps(model, people, net_w, net_h, num_scales=1, start_scale=1.0, scale_gap=0.15, seed=seed)
    full = orc.imresize(maps8, net_h, net_w, 1.0, 0.15)
    thr, _ = orc.default_params(model)
    peaks = orc.nms(full, orc.num_parts(model), orc.max_peaks(model), thr)
    cnt, joints = orc.connect(model, full, peaks, disp_w, disp_h)
    return cnt, joints, full, synth.make_frame(seed, disp_h, disp_w)


def gen_cuda(out_dir):
    R = orc.ref_cpm()
    assert R is not None and orc.ref_render_lib() is not None, "oracle/_ref CUDA libraries missing: build them from the reference first"
    d = {}
    model, net_w, net_h = rc.CPM_NET
    for S in rc.CPM_SCALES:
        rng = np.random.default_rng(S)
        for kind in ("scene", "noise"):
            if kind == "scene":
                people = synth.make_people(model, 7, net_w, net_h, seed=S)
                maps8 = synth.make_maps(model, people, net_w, net_h, num_scales=S, start_scale=1.0, scale_gap=0.15, seed=S)
            else:
                maps8 = rng.normal(0, 0.5, (S, 57, net_h // 8, net_w // 8)).astype(np.float32)
            rfull = np.zeros((57, net_h, net_w), np.float32)
            assert R.ref_imresize_host(np.ascontiguousarray(maps8), rfull, S, 57, net_h // 8, net_w // 8, net_h, net_w, 1.0, 0.15) == 0
            d["cpm_S%d_%s_full_sha" % (S, kind)] = sha(rfull)
            for thr in rc.CPM_THRESHOLDS:
                rpk = np.zeros((18, 65, 3), np.float32)
                assert R.ref_nms_host(rfull, rpk, 57, net_h, net_w, 18, 64, thr) == 0
                d["cpm_S%d_%s_thr%g_peaks" % (S, kind, thr)] = rpk

    for prefix, cases, seed, n_people in (("render", rc.RENDER_CASES, rc.RENDER_SEED, rc.RENDER_PEOPLE),
                                          ("devrender", rc.DEVICE_RENDER_CASES, rc.DEVICE_RENDER_SEED, rc.DEVICE_RENDER_PEOPLE)):
        for model, net_w, net_h, disp_w, disp_h, parts in cases:
            cnt, joints, full, frame = render_scene(model, net_w, net_h, disp_w, disp_h, n_people, seed)
            key = "%s_m%d_%dx%d" % (prefix, model, disp_w, disp_h)
            d[key + "_joints"] = joints
            canvas0 = orc.canvas_from_u8(frame)
            for part, googly in parts:
                d["%s_p%d_g%d_sha" % (key, part, googly)] = sha(orc.ref_render(model, canvas0, net_w, net_h, full, joints, cnt, part, bool(googly)))

    path = os.path.join(out_dir, "ref_cuda.npz")
    np.savez_compressed(path, **d)
    print(path, len(d), "arrays,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "host"
    out = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    {"host": gen_host, "cuda": gen_cuda}[what](out)
