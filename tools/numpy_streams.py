"""Rate of the device NumPy-stream generator alone (rocco_b200_numpy_normals_dev), in normals/s on one GPU.

    python tools/numpy_streams.py [--count 500000000] [--reps 5] [--chunk-words 64]

Two legs, each timed with CUDA events around --reps calls after one warm-up call:
  * emit: normals [0, count) of default_rng(seed) written to a device buffer (8 B per normal);
  * skip: the same stream parsed up to normal `count` without writing (what a sample shard does to reach its first row).
One JSON line with the card's name and power limit, read in the same run.
"""
import argparse, ctypes, json, os, subprocess, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rocco_b200 import _lib

ap = argparse.ArgumentParser()
ap.add_argument("--count", type=int, default=500_000_000)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--seed", type=int, default=104729)
ap.add_argument("--chunk-words", type=int, default=64)
args = ap.parse_args()
lib = _lib.load()
_lib.require_device()
prev = lib.rocco_b200_numpy_streams_set_chunk_words(args.chunk_words)
out = torch.empty(args.count, dtype=torch.float64, device="cuda")
stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
words = ctypes.c_ulonglong(0)
s_lo, s_hi = args.seed & ((1 << 64) - 1), args.seed >> 64


def emit():
    _lib.check(lib.rocco_b200_numpy_normals_dev(s_lo, s_hi, 0, args.count, ctypes.c_void_p(out.data_ptr()), ctypes.byref(words),
                                                stream), "numpy normals")


def skip():
    _lib.check(lib.rocco_b200_numpy_normals_dev(s_lo, s_hi, args.count, 1, ctypes.c_void_p(out.data_ptr()), None, stream),
               "numpy normals")


def timed(fn):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / args.reps


emit_ms = timed(emit)
skip_ms = timed(skip)
lib.rocco_b200_numpy_streams_set_chunk_words(prev)
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                           str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = torch.cuda.get_device_name()
print(json.dumps({"gpu": card, "count": args.count, "chunk_words": args.chunk_words, "words_consumed": int(words.value),
                  "emit_ms": emit_ms, "emit_normals_per_s": args.count / (emit_ms * 1e-3),
                  "emit_GB_per_s_written": 8.0 * args.count / (emit_ms * 1e-3) / 1e9,
                  "skip_ms": skip_ms, "skip_normals_per_s": args.count / (skip_ms * 1e-3)}))
