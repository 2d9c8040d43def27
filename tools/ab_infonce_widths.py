"""Two builds of the library against each other on the fused InfoNCE (rc_infonce_bf16) at D = 128, 384 and 512, in one process.

Both libraries are loaded with ctypes.CDLL and called with identical arguments; the timed launches alternate between them
so that clock and neighbour drift spread over both.  D = 512 is the control: with two builds that run the same kernels
there, its old / new difference and spread are the noise of the measurement.  Cells: D x (bf16 x, fp32 x) x (forward only,
forward + backward), B = 64, 256 x 256 pixels, K = 256 (X is 1-8 GB: far larger than the 126 MB L2).  Each timing sample
is REPS back-to-back launches between two CUDA events, after a warm-up; a cell reports the median of ALTS samples per
library and their spread (max - min).  The pre-pass the library runs inside rc_infonce_bf16 (bf16 copy of an fp32 x, row
norms where the kernel needs them) is part of every launch.  The outputs of the two libraries (loss, lse, dX) are compared
at the same sizes against the project's bf16 tolerances (2e-3 on loss and lse, 2e-2 max-relative on dX).

    git worktree add /tmp/rc_old <commit> && make -C /tmp/rc_old/rangeclip_b200/csrc
    python tools/ab_infonce_widths.py /tmp/rc_old/rangeclip_b200/librangeclip_b200.so [NEW_LIB] [--alts 7] [--reps 20] [--out f.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rangeclip_b200 import _lib, ops  # noqa: E402

B, H, W, K = 64, 256, 256, 256
HW = H * W
WIDTHS = (128, 384, 512)
CONTROL_D = 512


def load(path):
    lib = C.CDLL(os.path.abspath(path))
    for name, argtypes in _lib.PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _lib._RESTYPES.get(name, C.c_int)
    return lib


def gpu_state():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else f"nvidia-smi failed: {q.stderr.strip()}"


class Arm:
    """One library's output buffers for one cell; launch() is one rc_infonce_bf16 call."""

    def __init__(self, name, lib, x, xdt, D, tb, ttb, y, w, bwd):
        self.name, self.lib, self.x, self.xdt, self.D, self.bwd = name, lib, x, xdt, D, bwd
        self.tb, self.ttb, self.y, self.w = tb, ttb, y, w
        dev = x.device
        self.ws_bytes = int(lib.rc_infonce_workspace_bytes(B, D, HW, K, xdt))
        self.ws = torch.empty(self.ws_bytes, device=dev, dtype=torch.uint8)
        self.acc = torch.zeros(4, device=dev, dtype=torch.float64)      # loss_sum, w_sum, dlogtau, w_sum_in
        self.acc[3] = w.double().sum()
        self.lse = torch.empty(B * HW, device=dev)
        self.dx = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16) if bwd else None
        self.st = torch.cuda.current_stream().cuda_stream

    def launch(self):
        a = self.acc
        s = self.lib.rc_infonce_bf16(self.x.data_ptr(), self.xdt, B, self.D, HW, self.tb.data_ptr(), self.ttb.data_ptr(), K,
                                     self.y.data_ptr(), self.w.data_ptr(), 1 / 0.07, self.lse.data_ptr(), a[0:].data_ptr(),
                                     a[1:].data_ptr(), a[3:].data_ptr(), None, self.dx.data_ptr() if self.bwd else None, None,
                                     a[2:].data_ptr() if self.bwd else None, self.ws.data_ptr(), self.ws_bytes, 0, self.st)
        if s != 0:
            raise RuntimeError(f"{self.name}: rc_infonce_bf16 D={self.D} failed ({s}): {self.lib.rc_last_error().decode()}")

    def outputs(self):
        self.acc[:3].zero_()
        self.launch()
        torch.cuda.synchronize()
        return dict(loss=float(self.acc[0] / self.acc[1]), lse=self.lse.clone(), dx=self.dx)

    def time(self, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            self.launch()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps


def maxrel(a, b):
    return float((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old_lib")
    ap.add_argument("new_lib", nargs="?", default=_lib.LIB_PATH)
    ap.add_argument("--alts", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    libs = {"old": load(args.old_lib), "new": load(args.new_lib)}
    dev = torch.device("cuda:0")
    head = {"gpu_before": gpu_state(), "torch_name": torch.cuda.get_device_name(0), "B": B, "H": H, "W": W, "K": K,
            "alts": args.alts, "reps": args.reps, "old_lib": args.old_lib, "new_lib": args.new_lib}
    print(json.dumps(head), flush=True)
    cells = []
    for D in WIDTHS:
        g = torch.Generator(device=dev).manual_seed(D)
        x32 = torch.randn(B, D, HW, device=dev, generator=g)
        t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
        tb, ttb = ops.text_to_bf16(t)
        y = torch.randint(-1, K, (B * HW,), device=dev, generator=g, dtype=torch.int32)
        w = torch.randint(0, 3, (B * HW,), device=dev, generator=g).float()
        for xname in ("bf16", "fp32"):
            x = x32.to(torch.bfloat16) if xname == "bf16" else x32
            xdt = _lib.RC_BF16 if xname == "bf16" else _lib.RC_F32
            for bwd in (False, True):
                arms = {n: Arm(n, l, x, xdt, D, tb, ttb, y, w, bwd) for n, l in libs.items()}
                out = {n: a.outputs() for n, a in arms.items()}
                o, nw = out["old"], out["new"]
                cmp = {"loss_rel": abs(nw["loss"] - o["loss"]) / abs(o["loss"]), "lse_maxrel": maxrel(nw["lse"], o["lse"])}
                if bwd:
                    cmp["dx_maxrel"] = maxrel(nw["dx"], o["dx"])
                cmp["within_tol"] = cmp["loss_rel"] <= 2e-3 and cmp["lse_maxrel"] <= 2e-3 and cmp.get("dx_maxrel", 0.0) <= 2e-2
                for a in arms.values():
                    for _ in range(3):
                        a.launch()
                torch.cuda.synchronize()
                ms = {n: [] for n in arms}
                for _ in range(args.alts):
                    for n, a in arms.items():
                        ms[n].append(a.time(args.reps))
                cell = {"D": D, "x": xname, "mode": "fwd_bwd" if bwd else "fwd", **cmp}
                for n, v in ms.items():
                    cell[f"{n}_ms"] = round(statistics.median(v), 4)
                    cell[f"{n}_spread_ms"] = round(max(v) - min(v), 4)
                    cell[f"{n}_runs"] = [round(u, 4) for u in v]
                cell["new_over_old"] = round(cell["new_ms"] / cell["old_ms"], 4)
                print(json.dumps(cell), flush=True)
                cells.append(cell)
                del arms, out, o, nw
                torch.cuda.empty_cache()
        del x32, x
        torch.cuda.empty_cache()
    # a cell passes when the new library is not slower than the old one by more than the control's relative spread
    for c in cells:
        ctl = next(k for k in cells if k["D"] == CONTROL_D and k["x"] == c["x"] and k["mode"] == c["mode"])
        noise = max(ctl["old_spread_ms"], ctl["new_spread_ms"], abs(ctl["new_ms"] - ctl["old_ms"])) / ctl["old_ms"]
        c["control_noise"] = round(noise, 4)
        c["not_slower"] = c["new_ms"] / c["old_ms"] - 1 <= noise
    summary = {**head, "gpu_after": gpu_state(), "all_within_tol": all(c["within_tol"] for c in cells),
               "all_not_slower": all(c["not_slower"] for c in cells), "cells": cells}
    print(json.dumps({k: summary[k] for k in ("gpu_after", "all_within_tol", "all_not_slower")}), flush=True)
    for c in cells:
        print(f"D={c['D']:4d} x={c['x']} {c['mode']:7s} old {c['old_ms']:.3f} ms (+-{c['old_spread_ms']:.3f})  new {c['new_ms']:.3f} ms "
              f"(+-{c['new_spread_ms']:.3f})  new/old {c['new_over_old']:.3f}  control noise {c['control_noise']:.3f}  "
              f"lse {c['lse_maxrel']:.1e} dx {c.get('dx_maxrel', float('nan')):.1e}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
