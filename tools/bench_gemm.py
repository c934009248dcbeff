"""tcgen05 GEMM micro-benchmark on the shapes of one CLIP ViT-L/14 block at batch 32 (M = 8224) and of
ViT-B/16 at batch 256 (M = 50432): TFLOP/s per shape from CUDA events on the launching stream, SM clock
sampled by nvidia-smi during each shape's timed loop, and (yardstick only, never the product path)
torch.matmul / cuBLAS on the same shape under the same conditions.

    python tools/bench_gemm.py [--seconds 1.0]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vit-project_b200")]

import torch  # noqa: E402

import hba  # noqa: E402
from hba import ops  # noqa: E402
from hba.ops import HBA_ACT_QUICKGELU, Operand  # noqa: E402


class Clock:
    def __init__(self):
        self.rows = []
        self.p = subprocess.Popen(["nvidia-smi", "--id=0", "--query-gpu=clocks.sm,power.draw",
                                   "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                  stderr=subprocess.DEVNULL, text=True)
        threading.Thread(target=self._pump, daemon=True).start()

    def _pump(self):
        for line in self.p.stdout:
            try:
                a, b = line.split(",")
                self.rows.append((time.perf_counter(), float(a), float(b)))
            except ValueError:
                pass

    def window(self, t0, t1):
        r = [x for x in self.rows if t0 <= x[0] <= t1]
        if not r:
            return None, None
        return statistics.median(x[1] for x in r), max(x[2] for x in r)


def timed_loop(fn, seconds):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(5, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    return e0.elapsed_time(e1) / reps, t0, t1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--split", action="store_true")
    ap.add_argument("--no-cublas", action="store_true")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    sp = a.split
    shapes = [("qkv", 8224, 3072, 1024, "bf16"), ("out_proj+res", 8224, 1024, 1024, "res"),
              ("c_fc+quickgelu", 8224, 4096, 1024, "gelu"), ("c_proj+res", 8224, 1024, 4096, "res"),
              ("c_proj_noepi", 8224, 1024, 4096, "bf16"),
              ("vitb_qkv", 50432, 2304, 768, "bf16"), ("vitb_fc2+res", 50432, 768, 3072, "res"),
              ("square8k_bf16out", 8192, 8192, 8192, "bf16")]
    if a.only:
        shapes = [s for s in shapes if s[0] in a.only.split(",")]
    clk = Clock()
    out = {"split": sp, "shapes": {}}
    for name, M, N, K, kind in shapes:
        A = Operand.empty(M, K, sp, dev)
        B = Operand.empty(N, K, sp, dev)
        A.buf.normal_()
        B.buf.normal_(std=0.05)
        bias = torch.randn(N, device=dev)
        if kind == "bf16":
            kw = dict(bias=bias, out=Operand.empty(M, N, sp, dev))
        elif kind == "gelu":
            kw = dict(bias=bias, act=HBA_ACT_QUICKGELU, out=Operand.empty(M, N, sp, dev))
        elif kind == "res":
            kw = dict(bias=bias, residual=torch.randn(M, N, device=dev), out_f32=torch.empty(M, N, device=dev))
        else:
            kw = dict(out_f32=torch.empty(M, N, device=dev))
        ms, t0, t1 = timed_loop(lambda: ops.gemm(A, B, M, **kw), a.seconds)
        mhz, watts = clk.window(t0, t1)
        rec = {"M": M, "N": N, "K": K, "ms": ms, "tflops": 2.0 * M * N * K / ms / 1e9, "sm_mhz": mhz, "watts": watts}
        if mhz:
            rec["frac_of_clock_peak"] = rec["tflops"] * 1e12 / (148 * 8192 * mhz * 1e6)
        if not a.no_cublas and not sp:
            a16, b16 = A.buf[:, :K], B.buf[:, :K]
            c16 = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
            time.sleep(0.3)
            ms2, t0, t1 = timed_loop(lambda: torch.matmul(a16, b16.t(), out=c16), a.seconds)
            mhz2, w2 = clk.window(t0, t1)
            rec["cublas_plain_tflops"] = 2.0 * M * N * K / ms2 / 1e9
            rec["cublas_sm_mhz"], rec["cublas_watts"] = mhz2, w2
        out["shapes"][name] = rec
        del A, B, kw
        torch.cuda.empty_cache()
        time.sleep(0.3)
    clk.p.terminate()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
