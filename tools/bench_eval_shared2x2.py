"""Evaluation on the shared 2x2 embeddings against the stock decoder tail, one process, CUDA events.

(a) kernel: rc_eval_topk_hist_bf16 on the nearest-x2 upsampled bf16 tensor [B,D,2h,2w] against rc_eval_topk_bf16_rep4 on
    the rows [B,D,h,w]; metrics only (no id tensor), the histograms and counters of the two must be identical.
(b) public validation step: the stock tail (conv.float() -> F.interpolate -> F.normalize, then predict_and_accumulate)
    against predict_and_accumulate(conv, ..., shared2x2=True); reference candidate builder over the whole vocabulary.

B = 64, D = 512, 128^2 rows / 256^2 labels, K in {256, 1024}, k in {1, 5}, bf16 rows built from their labels in the style
of bench.py's evaluation config.  The two forms of each pair are alternated after a warm-up; medians are reported.  Mpix/s
counts full-resolution pixels; the tensor share is 2 K D flop per ranked row over 2250 TFLOP/s (dense BF16, data sheet).

    python tools/bench_eval_shared2x2.py [--out profiles/r4_eval_shared2x2.json] [--rounds 5]
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rangeclip_b200 import MetricAccumulator, ops, predict_and_accumulate  # noqa: E402

PEAK_BF16_TFLOPS = 2250.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def make_batch(dev, text, B, h, w, sigma, seed):
    """Labels in 32x32 full-resolution blocks drawn from the whole vocabulary; row (i, j) = text[label of (2i, 2j)] + noise
    (bench.py's eval config on the half-resolution rows), bf16."""
    C, D = text.shape
    g = torch.Generator(device=dev).manual_seed(seed)
    lab = torch.randint(0, C, (B, 2 * h // 32, 2 * w // 32), device=dev, generator=g)
    seg = lab.repeat_interleave(32, 1).repeat_interleave(32, 2).contiguous()
    conv = torch.empty(B, D, h, w, device=dev, dtype=torch.bfloat16)
    for b in range(B):
        conv[b] = (text[seg[b, ::2, ::2]].permute(2, 0, 1) + sigma * torch.randn(D, h, w, device=dev, generator=g)).to(torch.bfloat16)
    return conv, seg


def equivalences(C, dev, seed=5):
    E = torch.eye(C, dtype=torch.bool)
    pairs = torch.randperm(C, generator=torch.Generator().manual_seed(seed))[: C // 10]
    for a, b in zip(pairs[:-1].tolist(), pairs[1:].tolist()):
        E[a, b] = True
        E[b, a] = True
    return E.to(torch.uint8).to(dev), torch.argmax(E.to(torch.uint8), dim=1).to(dev)


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(arms, rounds, n):
    for fn in arms.values():          # warm-up: module load, workspace sizes
        fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            ms[name].append(timed(fn, n))
    return {name: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for name, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r4_eval_shared2x2.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval_shared2x2: needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    B, D, h, w = 64, 512, 128, 128
    H, W = 2 * h, 2 * w
    npix, nrows = B * H * W, B * h * w
    res = {"gpu": info, "B": B, "D": D, "rows": [h, w], "labels": [H, W], "kernel": [], "step": []}
    for K in (256, 1024):
        gt_ = torch.Generator(device=dev).manual_seed(99)
        text = F.normalize(torch.randn(K, D, device=dev, generator=gt_), dim=1)
        tb = ops.text_to_bf16(text)[0]
        idx = torch.arange(K, device=dev)
        E, cmap = equivalences(K, dev)
        conv, seg = make_batch(dev, text, B, h, w, 0.3, 500 + K)
        x_up = conv.repeat_interleave(2, 2).repeat_interleave(2, 3).contiguous()
        hists = {name: (torch.zeros(5, K, device=dev, dtype=torch.int64), torch.zeros(3, device=dev, dtype=torch.int64))
                 for name in ("upsampled", "rep4")}
        for k in (1, 5):
            def up():
                hh, cc = hists["upsampled"]
                hh.zero_(); cc.zero_()
                ops.eval_topk_hist(x_up, text, idx, k, seg, E, cmap, hh, cc, t_bf16=tb, want_ids=False)

            def rep4():
                hh, cc = hists["rep4"]
                hh.zero_(); cc.zero_()
                ops.eval_topk_rep4(conv, tb, idx, k, seg, E, cmap, hh, cc, want_ids=False)

            t = alternate({"upsampled": up, "rep4": rep4}, args.rounds, 5)
            same = all(torch.equal(hists["upsampled"][i], hists["rep4"][i]) for i in range(2))
            row = {"K": K, "k": k, "histograms_identical": same}
            for name, ranked in (("upsampled", npix), ("rep4", nrows)):
                ms = t[name]["median_ms"]
                tf = 2.0 * K * D * ranked / (ms * 1e-3) / 1e12
                row[name] = dict(t[name], mpix_s=npix / (ms * 1e-3) / 1e6, tensor_tflops=tf, tensor_share=tf / PEAK_BF16_TFLOPS)
            row["speedup"] = t["upsampled"]["median_ms"] / t["rep4"]["median_ms"]
            print(json.dumps(row), flush=True)
            res["kernel"].append(row)
            assert same, "rc_eval_topk_bf16_rep4 and the upsampled launch disagree"
        del x_up

        # (b) the public validation step, top-5, reference candidate builder over the whole vocabulary
        accs = {"stock_tail": MetricAccumulator(E, cmap, device=dev), "shared2x2": MetricAccumulator(E, cmap, device=dev)}

        def stock():
            random.seed(1)
            xn = F.normalize(F.interpolate(conv.float(), scale_factor=2, mode="nearest"), dim=1)
            predict_and_accumulate(xn, text, seg, accs["stock_tail"], K, 5, want_ids=False)

        def shared():
            random.seed(1)
            predict_and_accumulate(conv, text, seg, accs["shared2x2"], K, 5, want_ids=False, shared2x2=True)

        t = alternate({"stock_tail": stock, "shared2x2": shared}, args.rounds, 2)
        fin = {name: a.finalize(seg) for name, a in accs.items()}
        row = {"K": K, "k": 5, "speedup": t["stock_tail"]["median_ms"] / t["shared2x2"]["median_ms"],
               "hbm_bytes_not_materialised": {"upsampled_fp32": B * D * H * W * 4, "bf16_copy": B * D * H * W * 2}}
        for name in accs:
            row[name] = dict(t[name], mpix_s=npix / (t[name]["median_ms"] * 1e-3) / 1e6,
                             pixel_accuracy_t1=fin[name]["pixel_accuracy_t1"], pixel_accuracy_tk=fin[name]["pixel_accuracy_tk"])
        print(json.dumps(row), flush=True)
        res["step"].append(row)
        del conv, seg, accs
        torch.cuda.empty_cache()
    res["note"] = ("kernel: metrics only (no id tensor), inputs resident (the 4.3 GB upsampled tensor exceeds L2); step: "
                   "stock tail = conv.float() -> F.interpolate -> F.normalize -> predict_and_accumulate (fp32 rows: the fused "
                   "kernel's bf16 pre-pass), shared2x2 = predict_and_accumulate on the bf16 conv output")
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"written": args.out}))


if __name__ == "__main__":
    main()
