"""TEST INFRASTRUCTURE ONLY - the inputs on which tests/golden/ref_host.npz and ref_cuda.npz record what the reference's own code
computes.  tools/gen_ref_golden.py (which writes those files from oracle/_ref) and the tests that compare against them
(tests/test_oracle.py, test_host_pipeline.py, test_gpu_render.py) take their cases from here, so that the two cannot drift apart:
a case edited here without regenerating the files fails on a missing key or a hash that names the case.
"""
import ctypes as C
import hashlib
import os

import numpy as np

from oracle.orc import COCO_18, MPI_15

# OpenBLAS picks its sgemm kernel - and with it the summation order of every convolution of the oracle - from the CPU when it is
# loaded, unless OPENBLAS_CORETYPE names one.  The reference's convolution outputs were recorded with the SkylakeX kernel: the one
# kernel that computes the same bits in each OpenBLAS build the oracle may load (scipy's wheel, and OpenCV's older one, which names
# an unknown newer CPU "Prescott").  Only a CPU with these AVX-512 subsets can run it.
BLAS_CORE = "SkylakeX"
BLAS_CORE_CPU_FLAGS = ("avx512f", "avx512cd", "avx512bw", "avx512dq", "avx512vl")


def cpu_runs_blas_core():
    try:
        with open("/proc/cpuinfo") as f:
            flags = next((line.split(":", 1)[1].split() for line in f if line.startswith("flags")), [])
    except OSError:
        return False
    return all(fl in flags for fl in BLAS_CORE_CPU_FLAGS)


def pin_blas_core():
    """Make every OpenBLAS loaded from now on run BLAS_CORE where the CPU can (an OPENBLAS_CORETYPE already set is kept)."""
    if cpu_runs_blas_core():
        os.environ.setdefault("OPENBLAS_CORETYPE", BLAS_CORE)


def blas_core(path):
    """The kernel the OpenBLAS at `path` runs (scipy's wheel prefixes its symbols, OpenCV's does not)."""
    L = C.CDLL(path)
    for name in ("scipy_openblas_get_corename", "openblas_get_corename"):
        f = getattr(L, name, None)
        if f is not None:
            f.restype = C.c_char_p
            return f().decode()
    return None


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- reference host code (ref_host.npz)
IM2COL_CASES = [(3, 7, 9, 3, 1), (5, 11, 6, 7, 3), (4, 5, 5, 1, 0)]                                 # c, h, w, k, pad; rng seed 0
CONV_CASES = [(2, 3, 6, 4, 4, 3, 1), (1, 64, 23, 41, 64, 3, 1), (2, 128, 12, 21, 128, 7, 3), (1, 128, 12, 21, 512, 1, 0),
              (1, 185, 12, 21, 128, 7, 3)]                                                         # n, cin, h, w, cout, k, pad; seed 9
CONV_SAMPLE = 2048   # outputs stored per case besides the hash, at np.linspace(0, size - 1, n).astype(np.int64)
POOL_CASES = [(2, 3, 8, 10, 2, 2, 0), (1, 4, 7, 9, 2, 2, 0), (1, 2, 46, 82, 2, 2, 0), (1, 2, 9, 9, 3, 2, 1), (2, 1, 5, 5, 3, 2, 0)]   # seed 3
SCALE_CASES = [(656, 368, 1.0, 0.3, 3), (656, 368, 1.0, 0.15, 4), (496, 368, 1.0, 0.3, 2), (160, 96, 1.0, 0.3, 3), (992, 736, 1.0, 0.15, 4),
               (656, 368, 0.9, 0.05, 6)]                                                           # net_w, net_h, start, gap, scales
DISPLAY_CASES = [(1280, 720, 1280, 720), (640, 480, 1280, 720), (1920, 1080, 1280, 720), (333, 777, 656, 368), (1000, 10, 64, 64)]
PAD_CASE = (2, 90, 160, 48, 96, 3, 1.0, 0.3)              # frame seed, frame h, w, net_h, net_w, scales, start, gap
JSON_CASES = [(0, 18, 1.0), (1, 18, 0.5), (3, 15, 1.0), (7, 18, 0.3333333), (2, 18, 2.25)]           # people, parts, scale; seed 5
CONNECT_CASES = [(COCO_18, 320, 176, 8), (MPI_15, 240, 176, 5), (COCO_18, 656, 368, 22)]           # model, net_w, net_h, people
CONNECT_SEEDS = range(3)
SPECIAL_NETS = [(COCO_18, 320, 176), (MPI_15, 240, 176)]


def special_drops(num_parts):
    """Parts left out of every person of the special connect cases: nA==0 / nB==0 singleton rows, duplicates, nothing at all."""
    return ([2, 3, 4], [1], list(range(num_parts)), [0, 14, 15, 16, 17][:3])


def json_joints(rng, people, parts):
    j = (rng.random((people, parts, 3)) * np.array([1280, 720, 1])).astype(np.float32)
    if people:
        j[0, 1] = 0.0                                    # a missing part
        j[0, 2] = (1e-5, 123456.7, 1.0)                  # exponent and 6-digit rounding cases of operator<<(double/float)
    return j


KEY_TRIALS, KEY_SEED, KEY_LENGTH = 3, 21, 60
KEY_ALPHABET = "-=_+[]{};'" * 3 + ",." + "0123456789qwertyuiopas" + "g"

# ---- reference CUDA kernels (ref_cuda.npz)
CPM_NET, CPM_SCALES, CPM_THRESHOLDS = (COCO_18, 320, 176), (1, 3), (0.05, 0.5)
RENDER_CASES = [(COCO_18, 320, 176, 640, 352, [(0, 0), (0, 1), (1, 0), (18, 0), (19, 0), (20, 0), (21, 0), (39, 0)]),
                (MPI_15, 240, 176, 480, 352, [(0, 0), (1, 0), (15, 0), (16, 0), (17, 0), (44, 0)]),
                (COCO_18, 656, 368, 1280, 720, [(0, 1), (5, 0), (20, 0)])]   # model, net, display, (part_to_show, googly) views
RENDER_SEED, RENDER_PEOPLE = 21, 7
DEVICE_RENDER_CASES = [(COCO_18, 320, 176, 640, 352, [(0, 0), (0, 1), (3, 0), (19, 0), (20, 0), (25, 0)]),
                       (MPI_15, 240, 176, 480, 352, [(0, 0), (2, 0), (16, 0)])]
DEVICE_RENDER_SEED, DEVICE_RENDER_PEOPLE = 33, 6
