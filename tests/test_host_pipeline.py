"""Host pipeline of rtpose.bin (producers -> worker threads -> re-orderer / writer; examples/rtpose/rtpose.cpp:1459-1549) on a
machine WITHOUT a GPU: host/rtpose.cpp is built with ThreadSanitizer against tests/stub/stub_engine.cpp, a test double of the
GPU-touching entry points of poseengine.h that encodes every frame's identity into its "joints" (all host code of the library -
codecs, AVI reader, JSON writer, prototxt reader - stays the real libposeengine.so).  What is asserted: every frame's result lands
in its own file, in order, exactly once, whatever the number of producers / workers / frames per forward; the 0.1 s frame-drop
policy (rtpose.cpp:1107-1124); handleKey's thresholds reach the engines (:1617-1651); a failing device ends the run instead of
hanging it; no data race anywhere in the host code (TSAN), no handle used from two threads at once (checked by the stub)."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "caffe_rtpose_b200")


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    if not os.path.exists(os.path.join(PKG, "libposeengine.so")):
        subprocess.check_call(["make", "-C", PKG, "-j8"])
    out = str(tmp_path_factory.mktemp("hostpipe") / "rtpose_tsan")
    r = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=thread", "-Wall", "-I", os.path.join(ROOT, "include"),
                        os.path.join(PKG, "host", "rtpose.cpp"), os.path.join(ROOT, "tests", "stub", "stub_engine.cpp"), "-o", out,
                        "-L", PKG, "-lposeengine", "-Wl,-rpath," + PKG, "-pthread"], capture_output=True, text=True, timeout=300)
    if r.returncode != 0 and "tsan" in r.stderr.lower():
        pytest.skip("this g++ has no ThreadSanitizer runtime")
    assert r.returncode == 0, r.stderr[-3000:]
    return out


def run(exe, args, env=None, stdin=None, timeout=120, model="COCO"):
    e = dict(os.environ)
    e["TSAN_OPTIONS"] = "halt_on_error=0 exitcode=66"
    e.update(env or {})
    base = ["--model", model, "--caffeproto", "/nonexistent.prototxt", "--random_init", "he"]
    r = subprocess.run([exe] + base + args, capture_output=True, text=True, env=e, input=stdin, timeout=timeout)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[-6000:]
    assert "STUB: concurrent calls" not in r.stderr, r.stderr[-3000:]
    return r


def write_bmp(path, w, h, ident):
    """24-bit bottom-up .bmp whose top-left pixel (the first bytes of the decoded BGR image) carries `ident`."""
    img = np.random.RandomState(ident).randint(0, 256, size=(h, w, 3), dtype=np.uint8)
    img[0, 0, 0], img[0, 0, 1] = ident % 256, ident // 256
    stride = (w * 3 + 3) & ~3
    rows = b"".join(img[y].tobytes() + b"\0" * (stride - w * 3) for y in range(h - 1, -1, -1))
    hdr = b"BM" + struct.pack("<IHHI", 54 + len(rows), 0, 0, 54) + struct.pack("<IiiHHIIiiII", 40, w, h, 1, 24, 0, len(rows), 2835, 2835, 0, 0)
    with open(path, "wb") as f:
        f.write(hdr + rows)
    return img


def read_result(path, parts=18):
    d = json.load(open(path))
    bodies = [np.array(b["joints"], dtype=np.float64).reshape(parts, 3) for b in d["bodies"]]
    return bodies


def check_identity(bodies, ident, scale=1.0):
    """what stub_engine.cpp's forward writes: people = 1 + B % 3, x = the identity bytes, y = 100 * person + part"""
    assert len(bodies) == 1 + (ident % 256) % 3
    for q, b in enumerate(bodies):
        assert np.allclose(b[:, 0] * scale, ident, atol=0.51 * max(1.0, scale)), (b[0], ident)
        assert np.allclose(b[:, 1] * scale, 100 * q + np.arange(b.shape[0]), atol=0.51 * max(1.0, scale))


@pytest.mark.parametrize("topology", [
    dict(num_gpu=1, engines=1, producers=1, batch=1),      # the reference's topology: one producer, one Net per GPU, one frame per forward
    dict(num_gpu=2, engines=2, producers=4, batch=3),      # two GPUs x two handles, four decoder threads, three frames per forward
    dict(num_gpu=4, engines=1, producers=3, batch=0),      # automatic batch
])
def test_every_frame_lands_in_its_own_file_in_order(exe, tmp_path, topology):
    d = tmp_path / "images"
    d.mkdir()
    n = 75
    for i in range(n):
        w, h = (40, 24) if i % 11 != 5 else (32, 32)       # a frame of another size closes the batch it arrives in (one forward = one size)
        write_bmp(str(d / ("im%04d.bmp" % i)), w, h, 1000 + i)
    (d / "im0007.bmp").write_bytes(b"BM" + b"\0" * 20)     # undecodable: skipped like an empty cv::imread result, never blocks the order
    out, log = tmp_path / "json", tmp_path / "stub.log"
    r = run(exe, ["--image_dir", str(d), "--resolution", "40x24", "--net_resolution", "48x32", "--write_json", str(out), "--no_frame_drops",
                  "--num_gpu", str(topology["num_gpu"]), "--engines_per_gpu", str(topology["engines"]),
                  "--num_producers", str(topology["producers"]), "--batch", str(topology["batch"])],
            env={"STUB_LOG": str(log), "STUB_FORWARD_MS": "2"})
    assert r.returncode == 0, r.stderr[-3000:]
    assert "cannot decode" in r.stderr and "im0007.bmp" in r.stderr
    files = sorted(os.listdir(out))
    assert files == ["im%04d.json" % i for i in range(n) if i != 7]
    for i in range(n):
        if i == 7:
            continue
        w, h = (40, 24) if i % 11 != 5 else (32, 32)
        scale = min(40 / w, 24 / h)                         # frame.scale of rtpose.cpp:474-480; the writer multiplies by 1/scale (:1399-1400)
        check_identity(read_result(str(out / ("im%04d.json" % i))), 1000 + i, scale)
    lines = log.read_text().splitlines()
    creates = [l for l in lines if l.startswith("create")]
    assert len(creates) == topology["num_gpu"] * topology["engines"]
    assert [int(l.split("device=")[1].split()[0]) for l in creates] == [g for g in range(topology["num_gpu"]) for _ in range(topology["engines"])]
    assert sum(l.startswith("broadcast") for l in lines) == (1 if topology["num_gpu"] > 1 else 0)     # the path's only collective, once
    assert sum(l.startswith("share") for l in lines) == topology["num_gpu"] * (topology["engines"] - 1)
    fw = [l for l in lines if l.startswith("forward") and "calibrate" not in l]
    sizes = [int(l.split(" n=")[1].split()[0]) for l in fw]
    assert sum(sizes) == n - 1                              # every decodable frame went through exactly one forward
    if topology["batch"] > 0:
        assert max(sizes) <= topology["batch"]
    assert any("camera size=32x32" in l for l in fw)        # frames of another size take the warpAffine entry point
    assert "# frames: %d " % (n - 1) in r.stderr


def test_frame_drop_policy(exe, tmp_path):
    """processFrame drops frames that waited more than 0.1 s for a GPU (rtpose.cpp:1107-1124); --no_frame_drops keeps all."""
    out = tmp_path / "json"
    common = ["--synthetic", "60", "--resolution", "32x24", "--net_resolution", "32x24", "--batch", "1", "--engines_per_gpu", "1", "--write_json", str(out)]
    r = run(exe, common, env={"STUB_FORWARD_MS": "30"})
    assert r.returncode == 0, r.stderr[-3000:]
    kept = len(os.listdir(out))
    dropped = int(r.stderr.split(" dropped)")[0].split()[-1])
    assert dropped > 0 and kept + dropped == 60 and "# frames: %d " % kept in r.stderr
    out2 = tmp_path / "json2"
    common[-1] = str(out2)
    r = run(exe, common + ["--no_frame_drops"], env={"STUB_FORWARD_MS": "30"})
    assert r.returncode == 0 and len(os.listdir(out2)) == 60 and "0 dropped)" in r.stderr


def test_runtime_keys_reach_every_engine(exe, tmp_path):
    """handleKey (rtpose.cpp:1551-1671): '=' raises the NMS threshold by 0.005, ']' connect_inter_threshold, '}' the min-above count,
    \"'\" min_subset_cnt, '+' min_subset_score; the workers apply them before their next forward (:1145)."""
    log = tmp_path / "stub.log"
    r = run(exe, ["--synthetic", "600", "--resolution", "32x24", "--net_resolution", "32x24", "--batch", "1", "--num_gpu", "2", "--engines_per_gpu", "1",
                  "--no_frame_drops", "--keys_from_stdin"], env={"STUB_LOG": str(log), "STUB_FORWARD_MS": "5"}, stdin="==]}'+\n")
    assert r.returncode == 0, r.stderr[-3000:]
    assert "nms_threshold: 0.06" in r.stderr
    last = {}
    for l in log.read_text().splitlines():
        if l.startswith("forward"):
            last[l.split("engine=")[1].split()[0]] = l
    assert len(last) == 2
    for l in last.values():
        assert "nms=0.0600" in l and "connect=4,0.4050,0.0550,10" in l, l


def test_model_defaults_reach_the_engines(exe, tmp_path):
    """warmup()'s per-model thresholds (rtpose.cpp:212-226; pinned to the reference's text in tests/test_oracle.py) are what the
    workers hand to their engines before the first forward."""
    for model, want in (("COCO", "nms=0.0500 connect=3,0.4000,0.0500,9"), ("MPI", "nms=0.2000 connect=3,0.4000,0.0100,8")):
        log = tmp_path / ("%s.log" % model)
        r = run(exe, ["--synthetic", "6", "--resolution", "32x24", "--net_resolution", "32x24", "--no_frame_drops"], env={"STUB_LOG": str(log)}, model=model)
        assert r.returncode == 0, r.stderr[-2000:]
        fw = [l for l in log.read_text().splitlines() if l.startswith("forward") and "calibrate" not in l]
        assert fw and all(want in l for l in fw), fw[:2]


def test_device_failure_ends_the_run(exe, tmp_path):
    """A failing forward on one GPU stops every thread (no hang, exit code 1) and the frames finished before it are still written."""
    out = tmp_path / "json"
    r = run(exe, ["--synthetic", "200", "--resolution", "32x24", "--net_resolution", "32x24", "--batch", "2", "--num_gpu", "2", "--write_json", str(out),
                  "--no_frame_drops"], env={"STUB_FAIL_AT": "12", "STUB_FORWARD_MS": "3"}, timeout=60)
    assert r.returncode == 1
    assert "stub: injected device failure" in r.stderr
    assert 0 < len(os.listdir(out)) < 200


def test_setup_errors(exe, tmp_path):
    r = run(exe, ["--synthetic", "4", "--resolution", "32x24", "--net_resolution", "32x24", "--num_gpu", "3"], env={"STUB_NUM_DEVICES": "2"})
    assert r.returncode == 1 and "invalid device ordinal" in r.stderr
    # without NCCL every GPU loads the model itself (the reference's behaviour) and the run still completes
    out = tmp_path / "json"
    r = run(exe, ["--synthetic", "12", "--resolution", "32x24", "--net_resolution", "32x24", "--num_gpu", "2", "--write_json", str(out), "--no_frame_drops"],
            env={"STUB_NO_NCCL": "1"})
    assert r.returncode == 0 and "every GPU loads the model itself" in r.stderr and len(os.listdir(out)) == 12
    # no page-locked memory: frames go through the staged path, results unchanged
    out2 = tmp_path / "json2"
    r = run(exe, ["--synthetic", "12", "--resolution", "32x24", "--net_resolution", "32x24", "--write_json", str(out2), "--no_frame_drops"],
            env={"STUB_NO_PINNED": "1"})
    assert r.returncode == 0
    for f in os.listdir(out):
        assert (out / f).read_text() == (out2 / f).read_text()


def test_write_frames_with_overlays(exe, tmp_path):
    """--write_frames: pe_render per frame, displayFrame's text overlays unless --no_text (rtpose.cpp:1317-1353), one file per frame."""
    outs = {}
    for name, extra in (("text", []), ("notext", ["--no_text"])):
        out = tmp_path / name
        r = run(exe, ["--synthetic", "35", "--resolution", "320x96", "--net_resolution", "32x24", "--write_frames", str(out), "--frame_format", "bmp",
                      "--no_frame_drops", "--part_to_show", "3"] + extra, env={"STUB_LOG": str(tmp_path / (name + ".log"))})
        assert r.returncode == 0, r.stderr[-3000:]
        assert sorted(os.listdir(out)) == ["frame%06d.bmp" % i for i in range(35)]
        outs[name] = out
        assert all("part=3" in l for l in (tmp_path / (name + ".log")).read_text().splitlines() if l.startswith("render"))
    # [extension] --num_writers: the images are encoded off the display thread; the files do not depend on how many threads write them
    jpg = {}
    for nw in (1, 4):
        out = tmp_path / ("jpg%d" % nw)
        r = run(exe, ["--synthetic", "40", "--resolution", "320x96", "--net_resolution", "32x24", "--write_frames", str(out), "--no_frame_drops", "--no_text",
                      "--num_writers", str(nw)], env={"STUB_KEEP_FRAMES": "1"})
        assert r.returncode == 0, r.stderr[-3000:]
        assert sorted(os.listdir(out)) == ["frame%06d.jpg" % i for i in range(40)]
        jpg[nw] = [(out / f).read_bytes() for f in sorted(os.listdir(out))]
        assert all(b[:2] == b"\xff\xd8" and b[-2:] == b"\xff\xd9" for b in jpg[nw])   # complete files: the run ends after the writers
    assert jpg[1] == jpg[4] and len(set(jpg[1])) > 30                                    # and every frame's own picture
    a = np.frombuffer((outs["text"] / "frame000034.bmp").read_bytes()[54:], dtype=np.uint8)
    b = np.frombuffer((outs["notext"] / "frame000034.bmp").read_bytes()[54:], dtype=np.uint8)
    assert (b == 40).mean() > 0.99            # the stub's flat canvas
    assert 50 < (a != b).sum() < a.size // 4  # people count, part name (and the s/gpu line once 30 frames have passed)


def test_video_loops_until_quit_and_quit_is_not_an_error(exe, tmp_path):
    """--video without a writer loops at its end (rtpose.cpp:525-545) at the file's frame rate until ESC ('Q' on stdin), which ends
    the run with exit code 0 like the reference (:1564); with --write_json the clip is processed once, frame numbers in the names."""
    import time
    import cv2
    path = str(tmp_path / "clip.avi")
    wr = cv2.VideoWriter(path, cv2.CAP_OPENCV_MJPEG, cv2.VideoWriter_fourcc(*"MJPG"), 100.0, (64, 48))
    assert wr.isOpened()
    for i in range(8):
        wr.write(np.full((48, 64, 3), 20 * i, dtype=np.uint8))
    wr.release()
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66", STUB_LOG=str(tmp_path / "stub.log"))
    base = ["--model", "COCO", "--caffeproto", "/nonexistent.prototxt", "--random_init", "he", "--video", path, "--resolution", "64x48",
            "--net_resolution", "32x24"]
    p = subprocess.Popen([exe] + base + ["--keys_from_stdin"], stdin=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
    time.sleep(1.5)                       # 8 frames at 100 fps: several loops
    _, err = p.communicate("Q", timeout=60)
    assert p.returncode == 0, err[-3000:]
    assert "ThreadSanitizer" not in err, err[-6000:]
    assert err.count("Looping video after 8 frames") >= 2
    n_forward = sum(l.startswith("forward") and "calibrate" not in l for l in (tmp_path / "stub.log").read_text().splitlines())
    assert n_forward > 16                 # the clip went round more than twice
    out = tmp_path / "json"
    r = run(exe, base[6:] + ["--write_json", str(out), "--no_frame_drops"])
    assert r.returncode == 0 and sorted(os.listdir(out)) == ["frame%06d.json" % i for i in range(8)]
    assert "Looping" not in r.stderr


def test_handle_key_vs_reference_code(exe, tmp_path):
    """handleKey (rtpose.cpp:1551-1671) compiled from the reference (minus its cv:: window calls) against rtpose.bin's handle_key on
    random key sequences: the thresholds the engines end up with are bit-identical (float members stepped by the double 0.005), the
    integer parameters, the shown part and the googly-eyes switch equal.  The key sequences (random, kept inside the views this build
    renders: 0..39, where the reference lets the counter run to 55) and the state the reference's handleKey leaves after them, starting
    from the COCO defaults (pinned in tests/test_oracle.py), are stored in tests/golden/ref_host.npz (tools/gen_ref_golden.py draws
    them with the seed and alphabet of oracle/refcases.py)."""
    ref = np.load(os.path.join(ROOT, "tests", "golden", "ref_host.npz"))
    for trial, keys in enumerate(ref["keys"]):
        keys, f, i = str(keys), ref["keys_f"][trial], [int(v) for v in ref["keys_i"][trial]]
        log = tmp_path / ("keys%d.log" % trial)
        r = run(exe, ["--synthetic", "600", "--resolution", "32x24", "--net_resolution", "32x24", "--batch", "1", "--engines_per_gpu", "1", "--no_frame_drops",
                      "--keys_from_stdin"], env={"STUB_LOG": str(log), "STUB_FORWARD_MS": "3"}, stdin=keys + "\n")
        assert r.returncode == 0, r.stderr[-2000:]
        last = [l for l in log.read_text().splitlines() if l.startswith("forward")][-1]
        exact = [np.float32(v) for v in last.split("exact=")[1].split(",")]
        assert [e.tobytes() for e in exact] == [np.float32(f[j]).tobytes() for j in range(3)], (keys, last, list(f))
        cnt, above = int(last.split("connect=")[1].split(",")[0]), int(last.split("connect=")[1].split(",")[3].split()[0])
        assert (above, cnt) == (i[0], i[1])
        p2s = [int(l.split("p2s: ")[1]) for l in r.stderr.splitlines() if "p2s: " in l]
        assert (p2s[-1] if p2s else 0) == i[2]
        googly = [int(l.split("googly eyes: ")[1]) for l in r.stderr.splitlines() if "googly eyes: " in l]
        assert (googly[-1] if googly else 0) == i[3]
