"""More than 256 contrast rows on the shared 2x2 embeddings, one process, CUDA events.

Three variants of the text loss's fwd+bwd, alternated after a warm-up of each shape, medians reported:
  kblocked_rep4  ops.infonce_raw(rows, rep=4) at K > 256: the four-target kernel over blocks of 256 candidate rows
                 (forward round for the per-block lse, then fwd+bwd launches with the lse given)
  upsampled      what compute_loss_shared2x2 did before at K > 256: F.interpolate(nearest, x2) of the rows, the
                 full-resolution K-blocked loss of that tensor, then the 2x2 sum of its dX (upsample_nearest2d_backward,
                 what autograd runs below the interpolation)
  floor_k256     one rc_infonce_bf16_rep4 launch at K = 256 (the targets folded into [0, 256))
plus the public compute_loss_shared2x2 step at K = 300 (reference contrast builder, text term only) against compute_loss on
the stock decoder tail (F.interpolate -> F.normalize).  Peak memory: torch.cuda.max_memory_allocated above what was
allocated before the call.  The outputs of kblocked_rep4 and upsampled are compared at the timed size.

B = 64, D = 512, 128^2 rows / 256^2 labels, bf16 rows, weights = the reference's 0.7 HW draws with replacement.

    python tools/bench_shared2x2_kblocked.py [--out profiles/r5_shared2x2_kblocked.json] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from unittest import mock

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rangeclip_b200 as R  # noqa: E402
from rangeclip_b200 import ops  # noqa: E402
from rangeclip_b200.losses import group_2x2  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def peak_bytes(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del out
    return peak


def alternate(arms, rounds, n):
    for fn in arms.values():          # warm-up: module load, workspace sizes, allocator
        fn()
        fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            ms[name].append(timed(fn, n))
    return {name: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for name, v in ms.items()}


def maxrel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def make_batch(dev, B, D, h, w, n_labels, seed):
    """Rows [B, D, h, w] bf16; full-resolution labels in 16x16 blocks from n_labels classes (-1 nowhere: every pixel has a
    label), weights = multiplicity of each pixel among 0.7 HW draws per image (model.py:220-228)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    H, W = 2 * h, 2 * w
    x = torch.randn(B, D, h, w, device=dev, generator=g).to(torch.bfloat16)
    lab = torch.randint(0, n_labels, (B, H // 16, W // 16), device=dev, generator=g)
    seg = lab.repeat_interleave(16, 1).repeat_interleave(16, 2).contiguous()
    draws = torch.randint(0, H * W, (B, int(0.7 * H * W)), device=dev, generator=g)
    wt = torch.zeros(B, H * W, device=dev)
    wt.scatter_add_(1, draws, torch.ones_like(draws, dtype=torch.float32))
    return x, seg.to(torch.int32), wt.view(B, H, W)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r5_shared2x2_kblocked.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_shared2x2_kblocked: needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    B, D, h, w = 64, 512, 128, 128
    H, W = 2 * h, 2 * w
    inv_tau = 1 / 0.07
    res = {"gpu": info, "B": B, "D": D, "rows": [h, w], "labels": [H, W], "x_dtype": "bfloat16", "loss": [], "step": None}
    for K in (300, 512):
        gt = torch.Generator(device=dev).manual_seed(7 + K)
        t = F.normalize(torch.randn(K, D, device=dev, generator=gt), dim=1)
        x, seg, wt = make_batch(dev, B, D, h, w, K, 11 + K)
        y_full, w_full = seg.reshape(B, -1), wt.reshape(B, -1)
        y4, w4 = group_2x2(seg), group_2x2(wt)
        y4_256 = torch.where(y4 >= 0, y4 % 256, y4)
        t256 = t[:256].contiguous()
        outs = {}

        def new():
            outs["kblocked_rep4"] = ops.infonce_raw(x, t, y4, w4, inv_tau, True, False, "auto", rep=4)
            return outs["kblocked_rep4"]

        def upsampled():
            up = F.interpolate(x, scale_factor=2, mode="nearest")
            r = ops.infonce_raw(up, t, y_full, w_full, inv_tau, True, False, "auto")
            del up
            r["dx"] = torch.ops.aten.upsample_nearest2d_backward(r["dx"], [H, W], [B, D, h, w], 2.0, 2.0)
            outs["upsampled"] = r
            return r

        def floor():
            return ops.infonce_raw(x, t256, y4_256, w4, inv_tau, True, False, "bf16", rep=4)

        arms = {"kblocked_rep4": new, "upsampled": upsampled, "floor_k256": floor}
        t_ms = alternate(arms, args.rounds, 3)
        row = {"K": K, "n_blocks": (K + 255) // 256}
        for name, fn in arms.items():
            row[name] = dict(t_ms[name], peak_mib=peak_bytes(fn) / 2**20)
        a, b = outs["kblocked_rep4"], outs["upsampled"]
        la, lb = float(a["loss_sum"] / a["w_sum"]), float(b["loss_sum"] / b["w_sum"])
        row["agreement"] = {"loss_rel": abs(la - lb) / abs(lb), "dx_maxrel": maxrel(a["dx"], b["dx"]),
                            "dlogtau_rel": abs(float(a["dlogtau"]) - float(b["dlogtau"])) / abs(float(b["dlogtau"])),
                            "lse_maxrel": maxrel(a["lse"], b["lse"].view(B, H, W)[:, ::2, ::2].reshape(-1))}
        row["speedup_vs_upsampled"] = t_ms["upsampled"]["median_ms"] / t_ms["kblocked_rep4"]["median_ms"]
        row["ratio_to_floor"] = t_ms["kblocked_rep4"]["median_ms"] / t_ms["floor_k256"]["median_ms"]
        print(json.dumps(row), flush=True)
        res["loss"].append(row)
        ag = row["agreement"]
        assert ag["loss_rel"] < 2e-3 and ag["dx_maxrel"] < 2e-2 and ag["dlogtau_rel"] < 2e-2 and ag["lse_maxrel"] < 1e-4, ag
        del x, seg, wt, y_full, w_full, y4, w4, y4_256, outs
        torch.cuda.empty_cache()

    # the public step at K = 300: G foreground labels in the batch + (300 - G) random distractors, text term only
    n_labels, C = 101, 2000          # labels 1..100 in the segmentation (0 = background)
    x, seg, _ = make_batch(dev, B, D, h, w, n_labels, 5)
    G = int(torch.unique(seg).gt(0).sum())
    kd = 300 - G
    text = torch.randn(C, D, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    sets = {"medium": {}, "hard": {}}
    kw = dict(W_image=0.0, W_smooth=0.0, k_distractors=kd, pct_medium=0.0, pct_hard=0.0, pct_rand=1.0)

    class Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(0.07)))
            self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(0.1)))

    model = Model().to(dev)
    got = {}

    def step(shared):
        def run():
            xg = x.detach().requires_grad_(True)
            model.zero_grad(set_to_none=True)
            np.random.seed(1); torch.manual_seed(1)
            if shared:
                total, loss_info = R.compute_loss_shared2x2(model, xg, seg, text, sets, None, None, **kw)
            else:
                up = F.normalize(F.interpolate(xg, scale_factor=2, mode="nearest"), dim=1)
                total, loss_info = R.compute_loss(model, up, seg, text, sets, None, None, **kw)
            total.backward()
            got[shared] = (loss_info, xg.grad, float(model.log_temperature_text.grad))
            return xg.grad
        return run

    with mock.patch("torch.nn.functional.interpolate", side_effect=RuntimeError("upsampled")):
        step(True)()               # the shared step never builds the upsampled tensor
    t_ms = alternate({"compute_loss_shared2x2": step(True), "stock_tail": step(False)}, args.rounds, 1)
    row = {"K": G + kd, "foreground_labels": G, "k_distractors": kd, "terms": "text only (W_image = W_smooth = 0)"}
    for name, shared in (("compute_loss_shared2x2", True), ("stock_tail", False)):
        row[name] = dict(t_ms[name], peak_mib=peak_bytes(step(shared)) / 2**20)
    (ia, ga, da), (ib, gb, db) = got[True], got[False]
    row["agreement"] = {"loss_rel": abs(ia["text_contrastive_loss"] - ib["text_contrastive_loss"]) / abs(ib["text_contrastive_loss"]),
                        "dx_maxrel": maxrel(ga, gb), "dlogtau_rel": abs(da - db) / abs(db)}
    row["speedup"] = t_ms["stock_tail"]["median_ms"] / t_ms["compute_loss_shared2x2"]["median_ms"]
    print(json.dumps(row), flush=True)
    res["step"] = row
    res["note"] = ("loss variants: fwd+bwd of the text InfoNCE with the gradient w.r.t. the rows, inputs resident (the 4.3 GB "
                   "upsampled bf16 tensor exceeds L2); step: compute_loss_shared2x2 on the bf16 rows against compute_loss "
                   "on F.normalize(F.interpolate(rows)), both with the reference contrast builder")
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"written": args.out}))
    ag = row["agreement"]
    assert ag["loss_rel"] < 2e-3 and ag["dx_maxrel"] < 2e-2 and ag["dlogtau_rel"] < 2e-2, ag


if __name__ == "__main__":
    main()
