#!/usr/bin/env python3
"""bench.py - frames/sec of the rtpose hot path at 656x368 COCO-18 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            one rank per GPU (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's CPU path (oracle) on the host cores

Workload (config.workload = "C2", the default): COCO model, net 656x368, 1 scale, synthetic 1280x720 uint8 BGR
stream (72 distinct frames, 199 MB > L2), random-init "W-he" weights (SURVEY.md section 8d), B frames per forward.
`--workload C1|C3|C5` times the other BASELINE.json configs the same way (extra lines for BASELINE.md section 5).
A step = one forward of B frames per GPU through the whole path: INTER_AREA/pad/normalise, the 92-conv
stack, fused resize+NMS, PAF integral + greedy assignment + assembly, results to pinned host memory.

  value     frames/s, all GPUs, frames already resident in HBM (pe_forward_frames_device, two handles per GPU)
  e2e       frames/s through the public C-ABI call with HOST (pinned) frames: H2D of every frame and D2H of
            joints/peaks inside the timed region, two handles per GPU so copies overlap compute
  roofline  conv stack (tcgen05 kernel, all its launches of one step): algorithmic FLOPs / device time
            from CUDA events on the engine stream, vs the measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline  the oracle (Caffe CPU arithmetic, im2col + OpenBLAS sgemm, best host thread count) on one full frame
`--impl reference` times the same oracle on FULL frames of the same workload (one frame per step).
Frames are sharded one-per-GPU; the only collective is the init broadcast of the packed weights (NCCL).
`--dump-outputs DIR` writes what the last timed step computed on rank 0 (seeded inputs: two builds compare output for output).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs that fit one GPU.  C2 is the configuration the metric is quoted on (the default and the only
# one the driver runs); the others are extra lines for BASELINE.md section 5 (`--workload C3` ...).
#            model   net_w net_h disp_w disp_h S  start gap  frames/step  distinct frames   description
WORKLOADS = {
    "C1": ("MPI_15", 496, 368, 640, 480, 1, 1.0, 0.3, 11, 99, "C1: MPI 496x368, 1 scale, synthetic 640x480 stream, W-he random-init weights"),
    "C2": ("COCO_18", 656, 368, 1280, 720, 1, 1.0, 0.3, 9, 72, "C2: COCO 656x368, 1 scale, synthetic 720p stream, W-he random-init weights"),
    "C3": ("COCO_18", 656, 368, 1280, 720, 3, 1.0, 0.15, 3, 72, "C3: COCO 656x368, 3 scales (1.0/0.85/0.70), synthetic 720p stream, W-he random-init weights"),
    "C5": ("COCO_18", 992, 736, 1920, 1080, 4, 1.0, 0.15, 1, 24, "C5 per GPU: COCO 992x736, 4 scales (gap 0.15), synthetic 1080p stream, W-he random-init weights"),
}
DUMP_BUDGET = 64 << 20   # bytes written by --dump-outputs at most


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS), help="BASELINE.json config (default C2 = the metric's config)")
    ap.add_argument("--batch", type=int, default=0, help="frames per forward per GPU (default: per workload; C2: 9 x 4165 rows = 1.98 waves of 128-row tiles on 148 SMs)")
    ap.add_argument("--precision", type=int, default=2, help="0 fp32 SIMT, 1 bf16, 2 f16x2 split (parity mode), 3 bf16x3")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--handles", type=int, default=int(os.environ.get("PE_BENCH_HANDLES", "2")),
                    help="engine handles (worker streams) per GPU that alternate over the steps, as rtpose.bin --engines_per_gpu")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed device-resident steps, write what rank 0's last step computed as DIR/<name>.npy (float32): "
                         "num_people, joints, peaks and the stride-8 maps (leading frames only beyond %d MB)" % (DUMP_BUDGET >> 20))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def dump_outputs(path, results, maps, max_people):
    """What a caller of the timed path receives for the B frames of its last step - results[k] = (num_people, joints, peaks) of
    frame k (pe_fetch), maps = the stride-8 maps of all B frames (pe_fetch_maps) - as float32 .npy files.  joints are zero-padded
    to max_people persons; maps are kept whole for as many leading frames as the 64 MB budget allows (all of them for every
    BASELINE workload)."""
    B = len(results)
    out = {"num_people": np.array([n for n, _, _ in results], np.float32),
           "joints": np.zeros((B, max_people) + results[0][1].shape[1:], np.float32),
           "peaks": np.stack([p for _, _, p in results]).astype(np.float32)}
    for k, (n, j, _) in enumerate(results):
        out["joints"][k, :n] = j
    per_frame = maps.nbytes // B
    keep = max(0, min(B, (DUMP_BUDGET - sum(a.nbytes for a in out.values())) // per_frame))
    out["maps"] = maps[:keep * (maps.shape[0] // B)]
    os.makedirs(path, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(path, name + ".npy"), arr)


def peaks_info():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured"
    return 1400.0, 6650.0, "fallback"  # B200_PROFILING.md fallback (sustained), "of fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")] + [time.time()])

    def stop(self, windows=()):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        rows = [r for r in self.rows if len(r) >= 10 and num(r[1]) is not None]
        inside = [r for r in rows if any(a <= r[-1] <= b + 0.25 for a, b in windows)]
        loaded = inside or [r for r in rows if (num(r[3]) or 0) > 300.0] or rows   # samples taken during the timed regions
        sm = [num(r[1]) for r in loaded]
        mx = [num(r[2]) for r in rows if num(r[2]) is not None]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in (inside or rows):
            if len(r) >= 10:
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows), "samples_under_load": len(sm)}


class Workload:
    def __init__(self, name):
        (m, self.net_w, self.net_h, self.disp_w, self.disp_h, self.S, self.start, self.gap, self.batch, self.n_frames,
         self.desc) = WORKLOADS[name]
        self.name = name
        self.model_name = m

    def model(self, mod):
        return getattr(mod, self.model_name)

    def metric(self):
        return "frames/sec at %dx%d %s" % (self.net_w, self.net_h, "COCO-18" if self.model_name == "COCO_18" else "MPI-15")


def tune_threads(net, wl, synth, orc):
    """OpenBLAS on these GEMM shapes is SLOWER with all 128 threads than with 16-32 (fork/join cost): try a few thread
    counts up to every core on a band of a frame and keep the fastest."""
    cores = os.cpu_count() or 1
    band_h = 96 if wl.net_h >= 96 else wl.net_h
    disp_band = max(16, int(round(wl.disp_h * band_h / float(wl.net_h))))
    band = np.ascontiguousarray(synth.make_frame(1000, wl.disp_h, wl.disp_w)[:disp_band])
    net.process_frame(band, band_h, wl.net_w, wl.S, wl.start, wl.gap)   # warm-up (BLAS threads, page faults)
    best_t, best_n = None, cores
    for nthr in sorted({cores, max(cores // 2, 1), max(cores // 4, 1), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        orc.lib().orc_set_threads(nthr)
        t = time.time()
        net.process_frame(band, band_h, wl.net_w, wl.S, wl.start, wl.gap)
        t = time.time() - t
        if best_t is None or t < best_t:
            best_t, best_n = t, nthr
    orc.lib().orc_set_threads(best_n)
    return best_n, cores


def cpu_baseline_full_frame(wl, weights, frame):
    """The oracle (reference CPU path restated) on ONE full frame of the workload; ~5-60 s of CPU work."""
    from caffe_rtpose_b200 import synth
    from oracle import orc
    net = orc.Net(wl.model(orc))
    net.set_weights(weights)
    best_n, cores = tune_threads(net, wl, synth, orc)
    t = time.time()
    cnt, joints, peaks, _ = net.process_frame(frame, wl.net_h, wl.net_w, wl.S, wl.start, wl.gap)
    dt = time.time() - t
    return {"value": 1.0 / dt, "unit": "frames/s", "cores": best_n, "kind": "port",
            "sample": "1 full %dx%d frame (net %dx%d, %d scale(s), whole path incl. resize/NMS/connect), %.1f s; im2col + "
                      "OpenBLAS sgemm with %d threads (fastest of the counts tried on a band; %d cores available)"
                      % (wl.disp_w, wl.disp_h, wl.net_w, wl.net_h, wl.S, dt, best_n, cores)}, (cnt, joints, peaks)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path = the oracle port (the reference
    cannot be built here: no glog/gflags/boost/OpenCV-C++/protoc; its Forward_cpu for Nms/ImResize are
    different algorithms - SURVEY.md section 0).  SAME workload as the engine arm: one step = one FULL frame through
    the whole CPU path (the engine arm's step is `frames_per_step_per_gpu` such frames; the metric is frames/s).
    Rank 0 only."""
    if rank != 0:
        return
    from caffe_rtpose_b200 import synth
    from oracle import orc
    wl = Workload(args.workload)
    model = wl.model(orc)
    net = orc.Net(model)
    net.set_weights(synth.make_weights(model, "he"))
    best_n, cores = tune_threads(net, wl, synth, orc)
    frames = [synth.make_frame(i, wl.disp_h, wl.disp_w) for i in range(4)]
    for i in range(args.warmup):
        net.process_frame(frames[i % 4], wl.net_h, wl.net_w, wl.S, wl.start, wl.gap)
    t0 = time.time()
    for i in range(args.steps):
        cnt, joints, peaks, maps = net.process_frame(frames[i % 4], wl.net_h, wl.net_w, wl.S, wl.start, wl.gap)
    dt = time.time() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(cnt, joints, peaks)], maps, orc.MAX_PEOPLE)
    fps = args.steps / dt
    line = {"metric": wl.metric(), "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": wl.desc, "step": "one full frame through the whole CPU path (bounded sample of the engine arm's step)"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": best_n, "kind": "port",
                             "sample": "%d steps x one full %dx%d frame (net %dx%d, %d scale(s)); %d BLAS/OpenMP threads "
                                       "(fastest of the counts tried, %d cores available)"
                                       % (args.steps, wl.disp_w, wl.disp_h, wl.net_w, wl.net_h, wl.S, best_n, cores)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def parity_note(wl, eng, frame, ref):
    """Engine vs oracle on one frame at the default thresholds (the asserting version is tests/test_gpu_bench_parity.py)."""
    ocnt, ojoints, opeaks = ref
    eng.forward_frames([frame])
    cnt, joints, peaks = eng.fetch(0)
    mp = peaks.shape[1] - 1
    note = "frame 0: people engine/oracle %d/%d, peak counts per part identical: %s" % (
        cnt, ocnt, bool(np.array_equal(peaks[:, 0, 0], opeaks[:, 0, 0])))
    if np.array_equal(peaks[:, 0, 0], opeaks[:, 0, 0]):
        n = np.minimum(peaks[:, 0, 0], mp).astype(int)
        d = max([float(np.abs(peaks[p, 1:1 + n[p], :2] - opeaks[p, 1:1 + n[p], :2]).max()) for p in range(len(n)) if n[p]] or [0.0])
        note += ", max peak offset %.1e px" % d
    if cnt == ocnt and cnt > 0 and np.array_equal(joints[:, :, 2] > 0, ojoints[:, :, 2] > 0):
        d = float(np.abs(joints[:, :, :2] - ojoints[:, :, :2]).max()) * wl.net_w / wl.disp_w
        note += "; identical part->person assignment for all %d persons, max joint offset %.1e net px (bar: 1e-3)" % (cnt, d)
    else:
        note += "; person assignment differs"
    return note


_JSON_FD = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON line: everything else that libraries write to file descriptor 1 while the bench runs
    (NCCL prints "NCCL version ..." there at the first communicator, whatever NCCL_DEBUG says) is routed to stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
        return
    sys.stdout.flush()
    while data:
        data = data[os.write(_JSON_FD, data):]


def main():
    args = parse()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    # NCCL's own log (communicator ranks, transports) is NOT silenced; it goes to stderr so that stdout carries the
    # JSON line only
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    from caffe_rtpose_b200 import engine, synth

    wl = Workload(args.workload)
    torch.cuda.set_device(local_rank)
    # nvidia-smi takes ~1 s to deliver its first sample: start it now, keep only the samples whose arrival time
    # falls inside the two timed regions (device-resident loop, end-to-end loop)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    model = wl.model(engine)
    B = args.batch or wl.batch
    n_frames = max(wl.n_frames // B, 2) * B

    NH = max(1, min(4, args.handles))
    # ---- engines: NH (default two) handles per GPU (as the reference runs one Net per worker thread) so that the H2D of
    # one batch overlaps the compute of the other in the end-to-end loop
    engs = [engine.PoseEngine(model, wl.net_w, wl.net_h, wl.disp_w, wl.disp_h, num_scales=wl.S, start_scale=wl.start, scale_gap=wl.gap,
                              device=local_rank, max_batch=B, precision=args.precision) for _ in range(NH)]
    table = synth.conv_table(model)
    if rank == 0:
        W = synth.make_weights(model, "he")
    else:  # layout only; the values arrive by broadcast
        W = {name: (np.zeros((co, ci, k, k), np.float32), np.zeros(co, np.float32)) for name, co, ci, k in table}
    for e in engs:
        e.set_weights(W)
    if world > 1:
        # the ONE collective of the path: rank 0's packed weight replica -> every GPU over NVLink (NCCL)
        class _Dev:
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3}
        for e in engs:
            ptr, nbytes = e.packed_weights()
            t = torch.as_tensor(_Dev(ptr, nbytes), device="cuda")
            dist.broadcast(t, src=0)
        torch.cuda.synchronize()

    # ---- frames: distinct synthetic frames, sharded round-robin over ranks; pinned host + device copies
    frame_bytes = wl.disp_h * wl.disp_w * 3
    host = torch.empty((n_frames, wl.disp_h, wl.disp_w, 3), dtype=torch.uint8, pin_memory=True)
    hnp = host.numpy()
    for i in range(n_frames):
        hnp[i] = synth.make_frame(rank * n_frames + i, wl.disp_h, wl.disp_w)
    dev = host.cuda(non_blocking=False)
    nb = n_frames // B

    def batch_dev(i):
        return dev.data_ptr() + (i % nb) * B * frame_bytes

    def batch_host(i):
        j = (i % nb) * B
        return [hnp[j + k] for k in range(B)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sumreduce(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- single-process replica check (rtpose.bin --num_gpu topology): rank 0, child process with a timeout, before any
    # timed region; its JSON goes into the line as "replica_check"
    replica = None
    if world > 1 and rank == 0:
        try:
            r = subprocess.run([sys.executable, "-m", "caffe_rtpose_b200.replica_check", str(min(world, 2))], cwd=ROOT, capture_output=True,
                               text=True, timeout=180)
            replica = json.loads(r.stdout.strip().splitlines()[-1]) if r.stdout.strip() else {"result": "no output", "stderr": r.stderr[-300:]}
        except Exception as ex:   # never let the check take the bench down
            replica = {"result": "failed: %r" % (ex,)}
    barrier()

    e0 = engs[0]
    # ---- (1) device-resident throughput
    # two worker handles (two streams) alternate, like two of the reference's per-GPU worker threads would: the
    # small-grid parse kernels of one batch overlap the conv stack of the next.  Timed with torch CUDA events on
    # the null stream bracketing both engine streams (device-wide sync on both sides).
    for i in range(max(args.warmup, 2 * NH)):   # >= 2 forwards per handle: the 2nd captures its CUDA graph
        engs[i % NH].forward_frames_device(batch_dev(i), B)
    barrier()
    launches0 = sum(e.launch_count() for e in engs)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.time()
    ev0.record()
    for i in range(args.steps):
        engs[i % NH].forward_frames_device(batch_dev(args.warmup + i), B)
    for e in engs:
        e.sync()
    ev1.record()
    barrier()
    tw1 = time.time()
    ms_dev = maxreduce(ev0.elapsed_time(ev1))
    launches = sumreduce(sum(e.launch_count() for e in engs) - launches0)
    value = world * B * args.steps / (ms_dev * 1e-3)
    if args.dump_outputs and rank == 0:
        last = engs[(args.steps - 1) % NH]
        dump_outputs(args.dump_outputs, [last.fetch(k) for k in range(B)], last.fetch_maps(B), engine.MAX_PEOPLE)

    # ---- (2) end to end through the public call: host frames in, joints out, every step
    for i in range(NH):
        engs[i].forward_frames(batch_host(i))
    for e in engs:
        e.fetch(0)
    barrier()
    tw2 = time.time()
    t0 = time.perf_counter()
    got = 0
    for i in range(args.steps):
        e = engs[i % NH]
        if i >= NH:
            for k in range(B):
                n, joints, _ = e.fetch(k)   # results of step i-NH (sync on that handle's stream only)
            got += 1
        e.forward_frames(batch_host(i))
    for j in range(min(NH, args.steps) - 1, -1, -1):   # drain in submission order
        e = engs[(args.steps - 1 - j) % NH]
        for k in range(B):
            e.fetch(k)
        got += 1
    torch.cuda.synchronize()
    dt_e2e = maxreduce(time.perf_counter() - t0)
    clocks = sampler.stop([(tw0, tw1), (tw2, time.time())]) if rank == 0 else None
    assert got == args.steps
    e2e = world * B * args.steps / dt_e2e
    P, MP = e0.num_parts, e0.max_peaks
    d2h = B * (engine.MAX_PEOPLE * P * 3 * 4 + 4 + P * (MP + 1) * 3 * 4)

    if rank == 0:
        # ---- (3) roofline of the dominant kernel (conv stack), instrumented pass with events between launches
        e0.forward_frames_device(batch_dev(0), B)
        e0.sync()
        runs = [e0.profile_layers(B) for _ in range(5)]   # per-layer median of 5 passes: one pass right after the e2e loop can sit in a clock dip
        prof = [(runs[0][i][0], statistics.median(r[i][1] for r in runs), runs[0][i][2]) for i in range(len(runs[0]))]
        conv = [(n, ms, fl) for (n, ms, fl) in prof if fl > 0]
        conv_ms = sum(ms for _, ms, _ in conv)
        conv_flops = sum(fl for _, _, fl in conv)
        other_ms = sum(ms for _, ms, fl in prof if fl == 0)
        peak, _, how = peaks_info()
        achieved = conv_flops / (conv_ms * 1e-3) / 1e12
        step_ms = ms_dev / args.steps
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tp):   # dram__bytes_read+write per launch from the committed ncu capture of this same workload and build
            tj = json.load(open(tp))
            if tj.get("batch") == B and tj.get("precision") == args.precision and tj.get("workload", "C2") == wl.name:
                traffic, traffic_src = tj["traffic_bytes_per_launch"], tj["source"]
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_unit": "bytes per launch (dram read+write, avg over the conv launches of a step)",
                    "traffic_source": traffic_src, "peak_source": "%s (bf16 dense, sustained)" % how,
                    "kernel": "pe::conv_tc{w,p}_kernel (persistent tcgen05/TMEM/TMA implicit GEMM), %d launches per step" % len(conv),
                    "flops_per_step": conv_flops, "kernel_ms_per_step": conv_ms, "avg_launch_us": 1e3 * conv_ms / len(conv),
                    "share_of_step": conv_ms / step_ms, "other_layer_ms_per_step": other_ms,
                    "note": "algorithmic FLOPs (2*Cout*Cin*k^2*H*W); precision mode %d issues %d tensor-core MMAs per "
                            "algorithmic MAC; kernel time = sum over the conv launches of one step, CUDA events on the engine "
                            "stream between launches, per-layer median of 5 passes (serialised, one lane: no overlap between "
                            "consecutive or sibling layers is credited)"
                            % (args.precision, {0: 0, 1: 1, 2: 3, 3: 6}[args.precision])}
        cpu = None
        if not args.no_cpu_baseline:
            cpu, ref = cpu_baseline_full_frame(wl, W, hnp[0])
            cpu["parity_note"] = parity_note(wl, engs[1], hnp[0], ref)
        line = {"metric": wl.metric(), "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": {0: "f32", 1: "bf16", 2: "f16x2 (2 fp16 planes, 3 tcgen05 MMAs per MAC, fp32 accumulate)", 3: "bf16x3 (split, fp32 accumulate)"}[args.precision],
                "data": "synthetic",
                "config": {"workload": wl.desc,
                           "frames_per_step_per_gpu": B, "handles_per_gpu": NH, "precision_mode": args.precision, "sharding": "frames round-robin, one rank per GPU",
                           "l2": "%d distinct frames (%d MB) cycled > 126 MB L2; activations of one step >> L2" % (n_frames, n_frames * frame_bytes // 1000000),
                           "collective": "init broadcast of packed weights only (NCCL)" if world > 1 else "none"},
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * frame_bytes, "d2h_bytes_per_step": d2h,
                        "how": "pe_forward_frames (pinned host frames) + pe_fetch every step, %d handles per GPU, wall clock max over ranks" % NH},
                "gpu_launches": int(launches),
                "roofline": roofline}
        if cpu:
            line["cpu_baseline"] = cpu
        if replica is not None:
            line["replica_check"] = replica
        emit(line)
    for e in engs:
        e.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
