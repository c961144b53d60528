"""Renderers on the GPU (pe_render, csrc/render.cu) against
  (1) the reference's OWN render kernels (src/rtpose/renderFunctions.cu) compiled for sm_100a and launched with the
      reference's geometry on a B200 - the bit-level pin: the SHA-256 of each canvas they drew is stored in
      tests/golden/ref_cuda.npz with the persons they were given (tools/gen_ref_golden.py, on the cases of oracle/refcases.py), and
  (2) the CPU restatement in oracle/ (libm trigonometry, unfused sums) - equal up to shape-border pixels.
Inputs are injected stride-8 maps, so joints and the full-resolution maps are bit-identical on both sides."""
import os

import numpy as np
import pytest

from caffe_rtpose_b200 import engine, synth
from oracle import orc
from oracle import refcases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = np.load(os.path.join(ROOT, "tests", "golden", "ref_cuda.npz"))


def scene(model, net_w, net_h, disp_w, disp_h, n_people, seed, S=1):
    people = synth.make_people(model, n_people, net_w, net_h, seed=seed)
    maps8 = synth.make_maps(model, people, net_w, net_h, num_scales=S, start_scale=1.0, scale_gap=0.15, seed=seed)
    eng = engine.PoseEngine(model, net_w, net_h, disp_w, disp_h, num_scales=S, start_scale=1.0, scale_gap=0.15,
                            precision=engine.PREC_FP32_SIMT)
    eng.forward_maps(maps8)
    cnt, joints, _ = eng.fetch(0)
    full = orc.imresize(maps8, net_h, net_w, 1.0, 0.15)
    frame = synth.make_frame(seed, disp_h, disp_w)
    return eng, cnt, joints, full, frame


def canvas_sha(canvas):
    return refcases.sha(np.asarray(canvas, np.float32))


def compare_cpu(tag, got_canvas, got_img, want_canvas):
    """CPU restatement: measured max 2.3e-4 on the float canvas, <= 1.2e-5 of the uint8 pixels differ."""
    diff = np.abs(got_canvas - want_canvas)
    img_bad = float((got_img != orc.canvas_to_u8(want_canvas)).any(2).mean())
    assert diff.max() <= 2e-3 and img_bad <= 1e-4, (tag, float(diff.max()), float((diff.max(0) > 1e-3).mean()), img_bad)


@pytest.mark.parametrize("model,net_w,net_h,disp_w,disp_h,parts", refcases.RENDER_CASES)
def test_render_vs_reference_kernels_and_oracle(model, net_w, net_h, disp_w, disp_h, parts):
    eng, cnt, joints, full, frame = scene(model, net_w, net_h, disp_w, disp_h, refcases.RENDER_PEOPLE, seed=refcases.RENDER_SEED)
    assert cnt >= 3
    key = "render_m%d_%dx%d" % (model, disp_w, disp_h)
    assert np.array_equal(joints, REF[key + "_joints"])        # the persons the reference's kernels drew
    canvas0 = orc.canvas_from_u8(frame)
    for part, googly in parts:
        img, canvas = eng.render(0, part, bool(googly), display_bgr=frame, want_canvas=True)
        tag = "m%d_%dx%d_p%d_g%d" % (model, disp_w, disp_h, part, googly)
        assert canvas.shape == (3, disp_h, disp_w)
        assert canvas_sha(canvas) == str(REF["%s_p%d_g%d_sha" % (key, part, googly)]), tag   # bit-identical to the reference's kernels
        cpu = orc.render(model, canvas0, net_w, net_h, full, joints, cnt, part, bool(googly))
        compare_cpu(tag + "_cpu", canvas, img, cpu)
        assert np.array_equal(img, orc.canvas_to_u8(canvas))   # the uint8 conversion itself is exact
    eng.close()


def test_render_from_resident_frame_and_errors():
    model, net_w, net_h, disp_w, disp_h = engine.COCO_18, 160, 96, 320, 192
    W = synth.make_weights(model, "he")
    eng = engine.PoseEngine(model, net_w, net_h, disp_w, disp_h, precision=engine.PREC_F16X2, max_batch=2)
    eng.set_weights(W)
    frames = [synth.make_frame(i, disp_h, disp_w) for i in range(2)]
    eng.forward_frames(frames)
    for idx in range(2):
        a = eng.render(idx, 0)                              # display frame still on the device
        b = eng.render(idx, 0, display_bgr=frames[idx])     # same frame passed explicitly
        assert np.array_equal(a, b)
        h = eng.render(idx, 3)
        assert h.shape == (disp_h, disp_w, 3) and (h != frames[idx]).any()
    cnt, joints, _ = eng.fetch(0)
    if cnt == 0:   # noise maps rarely give persons: the skeleton view must then return the frame itself
        assert np.array_equal(eng.render(0, 0), frames[0])
    with pytest.raises(engine.PoseEngineError):
        eng.render(0, 40)
    with pytest.raises(engine.PoseEngineError):
        eng.render(2, 0)
    people = synth.make_people(model, 3, net_w, net_h, seed=5)
    eng.forward_maps(synth.make_maps(model, people, net_w, net_h, seed=5))
    with pytest.raises(engine.PoseEngineError):             # no display frame on the map-injection path
        eng.render(0, 0)
    assert eng.render(0, 0, display_bgr=frames[0]).shape == (disp_h, disp_w, 3)
    eng.close()


def test_device_pointer_render_api_equals_reference_kernels():
    """render_mpi_parts / render_coco_parts / render_coco_aff with the reference's device-pointer arguments
    (include/rtpose/renderFunctions.h shim -> pe_render_device): canvas, full-resolution heat maps and joints in caller-owned
    device memory, no engine handle.  Bit-identical to the reference's own kernels for every view."""
    import ctypes as C
    import torch
    L = engine.lib()
    for model, net_w, net_h, disp_w, disp_h, parts in refcases.DEVICE_RENDER_CASES:
        eng, cnt, joints, full, frame = scene(model, net_w, net_h, disp_w, disp_h, refcases.DEVICE_RENDER_PEOPLE, seed=refcases.DEVICE_RENDER_SEED)
        eng.close()
        key = "devrender_m%d_%dx%d" % (model, disp_w, disp_h)
        assert np.array_equal(joints, REF[key + "_joints"])    # the persons the reference's kernels drew
        P = 15 if model == engine.MPI_15 else 18
        canvas0 = orc.canvas_from_u8(frame)
        d_full = torch.from_numpy(np.ascontiguousarray(full)).cuda()
        d_poses = torch.from_numpy(np.ascontiguousarray(joints[:cnt].reshape(-1))).cuda()
        n = (C.c_int * 1)(cnt)
        for part, googly in parts:
            d_canvas = torch.from_numpy(canvas0.copy()).cuda()
            if model == engine.MPI_15:
                kind, p, extra = 0, part, 0
            elif part - 1 <= P:                      # render() of rtpose.cpp:271-300
                kind, p, extra = 1, part, googly
            else:
                aff, accum = ((part - 1) - P - 1) * 2, 1
                if aff == 0:
                    accum = 19
                else:
                    aff -= 2
                kind, p, extra = 2, aff + 1 + P, accum
            rc = L.pe_render_device(kind, d_canvas.data_ptr(), disp_w, disp_h, net_w, net_h, d_full.data_ptr(), d_poses.data_ptr(), n, 1, p, extra)
            assert rc == 0
            assert canvas_sha(d_canvas.cpu().numpy()) == str(REF["%s_p%d_g%d_sha" % (key, part, googly)]), (model, part, googly)
