"""f3 (SURVEY.md section 8f rank 3): the execution plan is built from the deploy prototxt, as `new caffe::Net(proto, TEST)`
does (rtpose.cpp:183, net.cpp:30-280), for every stage count the reference ships (model/mpi/pose_deploy_linevec_{1,2,4}).

CPU part (no GPU): the engine's prototxt reader + plan builder (pe_plan_describe) against tests/golden/netspec_*.json - the
layer tables tools/gen_netspec_fixture.py parsed from the reference's files - and against the files themselves (stored gzipped
under tests/golden/prototxt/); error reporting for graphs outside the pose path.  GPU part: a 2-stage MPI net created from its
prototxt, conv stack and whole path against the oracle."""
import gzip
import json
import os

import numpy as np
import pytest

from caffe_rtpose_b200 import engine, synth
from oracle import orc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REF = os.path.join(GOLD, "prototxt")   # deploy files of the reference's model/ directory
SPECS = [("coco", engine.COCO_18, 6), ("mpi", engine.MPI_15, 6), ("mpi_1", engine.MPI_15, 1), ("mpi_2", engine.MPI_15, 2), ("mpi_4", engine.MPI_15, 4)]


def spec_prototxt(name, tmp_path):
    spec = json.load(open(os.path.join(GOLD, "netspec_%s.json" % name)))
    p = tmp_path / ("%s.prototxt" % name)
    p.write_text(synth.netspec_to_prototxt(spec))
    return spec, str(p)


def parse_plan(text):
    ops = [l.split() for l in text.splitlines()]
    return {"model": int(ops[0][1]), "convs": [o for o in ops if o[0] == "conv"], "pools": [o for o in ops if o[0] == "pool"],
            "copies": [o for o in ops if o[0] == "copy"], "nms": [o for o in ops if o[0] == "nms"][0], "resize": [o for o in ops if o[0] == "resize"][0]}


@pytest.mark.parametrize("name,model,stages", SPECS)
def test_plan_from_prototxt_matches_the_layer_table(name, model, stages, tmp_path):
    spec, path = spec_prototxt(name, tmp_path)
    plan = parse_plan(engine.plan_describe(prototxt=path))
    assert plan["model"] == model                                       # inferred from nms num_parts (rtpose.cpp:212-229)
    convs = [l for l in spec["layers"] if l["type"] == "Convolution"]
    relu_on = {l["bottom"][0] for l in spec["layers"] if l["type"] == "ReLU"}
    assert len(plan["convs"]) == len(convs) == len(synth.conv_table(model, stages))
    table = {n: (co, ci, k) for n, co, ci, k in synth.conv_table(model, stages)}
    for got, want in zip(plan["convs"], convs):                         # prototxt order, shapes, fused ReLU
        assert got[1] == want["name"]
        assert (int(got[2]), int(got[4])) == (want["num_output"], want["kernel_size"])
        assert int(got[3]) == table[want["name"]][1]                    # input channels inferred through Concat / Pooling
        assert int(got[5]) == (want["name"] in relu_on)
    assert len(plan["pools"]) == 3
    nms, rsz = spec["layers"][-1], spec["layers"][-2]
    assert (float(plan["nms"][1]), int(plan["nms"][2]), int(plan["nms"][3])) == (pytest.approx(nms["threshold"]), nms["max_peaks"], nms["num_parts"])
    assert (float(plan["resize"][1]), float(plan["resize"][2])) == (pytest.approx(rsz["start_scale"]), pytest.approx(rsz["scale_gap"]))
    # the last stage writes the planar concat_stage7 = [L2 | L1] (prototxt :2966-2975): L1 at channel offset c_l2
    last = {c[1]: c for c in plan["convs"][-2:]}
    c_l2 = table[[n for n in table if n.endswith("_L2")][-1]][0]
    assert all(int(c[9]) == -1 for c in last.values())
    assert sorted(int(c[11]) for c in last.values()) == [0, c_l2]
    # one F copy when two concat buffers ping-pong (>= 3 stages), none otherwise
    assert len(plan["copies"]) == (1 if stages >= 3 else 0)
    if stages == 6:                                                     # the built-in graph is the same plan
        assert engine.plan_describe(model=model).split("\nnms")[0] == engine.plan_describe(prototxt=path).split("\nnms")[0]


def test_reference_prototxt_files_parse_directly(tmp_path):
    def ref_file(rel):
        path = tmp_path / os.path.basename(rel)
        with gzip.open(os.path.join(REF, rel + ".gz"), "rb") as f:
            path.write_bytes(f.read())
        return str(path)
    for rel, name in (("coco/pose_deploy_linevec.prototxt", "coco"), ("mpi/pose_deploy_linevec.prototxt", "mpi"),
                      ("mpi/pose_deploy_linevec_1.prototxt", "mpi_1"), ("mpi/pose_deploy_linevec_2.prototxt", "mpi_2"),
                      ("mpi/pose_deploy_linevec_4.prototxt", "mpi_4")):
        spec = json.load(open(os.path.join(GOLD, "netspec_%s.json" % name)))
        plan = parse_plan(engine.plan_describe(prototxt=ref_file(rel)))
        assert [c[1] for c in plan["convs"]] == [l["name"] for l in spec["layers"] if l["type"] == "Convolution"]
    # graphs that are not the PAF pose path are refused with the layer named (the reference would need generic Caffe layers)
    with pytest.raises(engine.PoseEngineError, match="Switch"):
        engine.plan_describe(prototxt=ref_file("mpi/pose_deploy_linevec_switch.prototxt"))
    with pytest.raises(engine.PoseEngineError, match="3 channels"):
        engine.plan_describe(prototxt=ref_file("mpi/pose_deploy_resize.prototxt"))


def test_prototxt_syntax_and_errors(tmp_path):
    spec, path = spec_prototxt("mpi_1", tmp_path)
    text = open(path).read()
    base = engine.plan_describe(prototxt=path)

    def plan_of(t):
        p = tmp_path / "t.prototxt"
        p.write_text(t)
        return engine.plan_describe(prototxt=str(p))
    # text-format variants protobuf accepts: comments, `key: { }`, single quotes, input_shape, hex / float integers are refused
    alt = text.replace("convolution_param {", "convolution_param: {  # comment").replace('"conv1_1"', "'conv1_1'")
    alt = alt.replace("input_dim: 1\ninput_dim: 3", "input_shape { dim: 1 dim: 3").replace("input_dim: %d\ninput_dim: %d" % tuple(spec["input_dim"][2:]),
                                                                                             "dim: %d dim: %d }" % tuple(spec["input_dim"][2:]))
    assert plan_of(alt) == base
    # legacy V1 `layers` blocks with enum types (upgrade_proto.cpp:957 UpgradeV1Net)
    v1 = text.replace("layer {", "layers {")
    for a, b in (("Convolution", "CONVOLUTION"), ("ReLU", "RELU"), ("Pooling", "POOLING"), ("Concat", "CONCAT")):
        v1 = v1.replace('type: "%s"' % a, "type: %s" % b)
    with pytest.raises(engine.PoseEngineError, match="legacy layer type"):   # ImResize / Nms have no V1 enum: such a file cannot exist
        plan_of(v1)
    for bad, msg in ((text.replace("kernel_size: 3", "kernel_size: 5", 1).replace("pad: 1", "pad: 1", 1), "same"),
                     (text.replace("pool: MAX", "pool: AVE", 1), "MAX pooling"),
                     (text.replace("factor: 8", "factor: 4"), "factor"),
                     (text.replace('type: "ReLU"', 'type: "Sigmoid"', 1), "Sigmoid"),
                     (text.replace("num_output: 64", "num_output: x64", 1), "integer"),
                     (text[:text.index("layer {", len(text) // 2) + 9], "unbalanced|end of file"),
                     (text.replace("num_output: 64", "num_output: 2147483647", 1), "num_output 2147483647 is larger"),   # found by the fuzzer below
                     (text.replace('bottom: "conv1_1"', 'bottom: "nope"', 1), "unknown bottom")):
        with pytest.raises(engine.PoseEngineError, match=msg):
            plan_of(bad)
    with pytest.raises(engine.PoseEngineError, match="cannot open"):
        engine.plan_describe(prototxt=str(tmp_path / "missing.prototxt"))


def test_prototxt_reader_survives_corrupt_files(tmp_path):
    """--caffeproto is a user file: the reader and the plan builder under ASAN + UBSan on mutated deploy files (bytes, cut-offs, dropped
    and repeated blocks, extreme numbers, renamed blobs) - every outcome is a plan or an error message, never a crash."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = os.path.join(root, "caffe_rtpose_b200", "csrc")
    files = [spec_prototxt(n, tmp_path)[1] for n in ("coco", "mpi_2")]
    exe = str(tmp_path / "fuzz_prototxt")
    r = subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-I", os.path.join(root, "include"),
                        "-I", src, "-I", "/usr/local/cuda/include", os.path.join(root, "tests", "fuzz", "fuzz_prototxt.cpp"), os.path.join(src, "prototxt.cpp"),
                        os.path.join(src, "plan.cpp"), "-o", exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([exe, "1200"] + files, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-3000:])
    parsed, planned, rejected = [int(v) for v in r.stdout.split()[1::2]]
    assert parsed > 200 and planned > 100 and rejected > 200   # the mutations are neither all harmless nor all fatal


@pytest.mark.gpu
def test_two_stage_net_from_prototxt_vs_oracle(tmp_path):
    """model/mpi/pose_deploy_linevec_2.prototxt (36 convolutions, one concat buffer, max_peaks from the proto default):
    stride-8 maps within the conv tolerance of the oracle's 2-stage net, peaks / joints as the oracle's post-processing
    gives them on the engine's own maps (bit-exact parse stage)."""
    _, path = spec_prototxt("mpi_2", tmp_path)
    net_w, net_h = 240, 176
    W = synth.make_weights(engine.MPI_15, "he", stages=2)
    onet = orc.Net(orc.MPI_15, stages=2)
    onet.set_weights(W)
    frame = synth.make_frame(77, 2 * net_h, 2 * net_w)
    x = orc.preprocess(frame, net_h, net_w, 1, 1.0, 0.3)
    omaps = onet.forward(x)
    for prec, tol in ((engine.PREC_FP32_SIMT, 5e-5), (engine.PREC_BF16X2, 3e-5)):
        eng = engine.PoseEngine(None, net_w, net_h, 2 * net_w, 2 * net_h, precision=prec, prototxt=path)
        assert eng.model == engine.MPI_15 and eng.nms_layer.GetNumParts() == 15 and eng.nms_layer.GetMaxPeaks() == 20
        assert len(eng.conv_layers()) == 36
        eng.set_weights(W)
        eng.forward_frames([frame])
        cnt, joints, peaks = eng.fetch(0)
        maps = eng.fetch_maps(1)
        eng.close()
        assert float(np.abs(maps - omaps).max() / np.abs(omaps).max()) < tol
        full = orc.imresize(maps, net_h, net_w, 1.0, 0.3)
        thr, _ = orc.default_params(orc.MPI_15)
        opk = orc.nms(full, 15, 20, thr)
        ocnt, oj = orc.connect(orc.MPI_15, full, opk, 2 * net_w, 2 * net_h)
        assert np.array_equal(peaks, opk) and cnt == ocnt and np.array_equal(joints, oj)
