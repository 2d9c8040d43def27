"""Open-vocabulary scores against ids only, one process, CUDA events.

(a) full resolution: rc_eval_topk_bf16 (ids) against rc_eval_topk_scores_bf16 (ids, cosine, softmax probability) on the
    same bf16 rows, B = 64, 256^2, D = 512, K in {1024, 5632} (5632: the size of the SUN RGB-D pseudo-label vocabulary),
    k in {1, 5};
(b) shared 2x2: rc_eval_topk_bf16_rep4 (ids) against rc_eval_topk_scores_bf16_rep4 on the decoder's 128^2 rows, outputs at
    256^2, same K and k;
(c) eager PyTorch (F.normalize -> einsum -> softmax -> topk on a materialised [B, K, HW] fp32 logit tensor) at B = 8, the
    batch whose logits fit comfortably (8.6 GB at K = 5632; B = 64 would need 17 / 94 GB).

The rows are text rows of 32x32 label blocks plus noise (bench.py's evaluation config), so the number of top-k insertions is
that of a trained model rather than of random rows.  The two arms of each pair alternate after a warm-up; medians are
reported, and the ids of the two arms are compared.  x (4.3 GB) is far larger than the 126 MB L2.  Mpix/s counts output
pixels.

    python tools/bench_segment.py [--out profiles/r9_segment.json] [--rounds 7]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rangeclip_b200 import ops  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_device": torch.cuda.get_device_name(0)}


def make_rows(dev, text, B, h, w, block, sigma, seed):
    """Rows [B, D, h, w] bf16: text[label] + noise, labels constant on block x block squares of the row grid."""
    C, D = text.shape
    g = torch.Generator(device=dev).manual_seed(seed)
    lab = torch.randint(0, C, (B, h // block, w // block), device=dev, generator=g)
    lab = lab.repeat_interleave(block, 1).repeat_interleave(block, 2)
    x = torch.empty(B, D, h, w, device=dev, dtype=torch.bfloat16)
    for b in range(B):
        x[b] = (text[lab[b]].permute(2, 0, 1) + sigma * torch.randn(D, h, w, device=dev, generator=g)).to(torch.bfloat16)
    return x


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def alternate(arms, rounds, n):
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            ms[name].append(timed(fn, n))
    return {name: statistics.median(v) for name, v in ms.items()}, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r9_segment.json")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    D, tau = 512, 0.07
    lt = torch.tensor([math.log(tau)], device=dev)
    vocab = F.normalize(torch.randn(5632, D, device=dev), dim=1)
    rec = {"gpu": gpu_info(), "tau": tau, "D": D, "full": [], "shared2x2": [], "eager": []}

    x = make_rows(dev, vocab[:1024], 64, 256, 256, 32, 1.5, seed=1)
    for K in (1024, 5632):
        t = vocab[:K]
        imap = torch.arange(K, device=dev)
        tb = ops.text_to_bf16(t)[0]
        # the rows were drawn from the first 1024 labels: at K = 5632 the other labels are distractors
        for k in (1, 5):
            arms = {"ids": lambda: ops.eval_topk(x, t, imap, k, "bf16", t_bf16=tb),
                    "scores": lambda: ops.eval_topk_scores(x, tb, imap, k, lt)}
            med, raw = alternate(arms, args.rounds, args.iters)
            same = torch.equal(arms["ids"](), arms["scores"]()[0])
            n_px = x.shape[0] * x.shape[2] * x.shape[3]
            r = {"B": 64, "HW": "256x256", "K": K, "k": k, "ids_ms": med["ids"], "scores_ms": med["scores"],
                 "ratio": med["scores"] / med["ids"], "ids_mpix_s": n_px / med["ids"] / 1e3,
                 "scores_mpix_s": n_px / med["scores"] / 1e3, "ids_equal": same, "raw_ms": raw}
            print(json.dumps({kk: v for kk, v in r.items() if kk != "raw_ms"}), flush=True)
            rec["full"].append(r)
    del x
    torch.cuda.empty_cache()

    x2 = make_rows(dev, vocab[:1024], 64, 128, 128, 16, 1.5, seed=2)
    for K in (1024, 5632):
        t = vocab[:K]
        imap = torch.arange(K, device=dev)
        tb = ops.text_to_bf16(t)[0]
        for k in (1, 5):
            arms = {"ids": lambda: ops.eval_topk_rep4(x2, tb, imap, k),
                    "scores": lambda: ops.eval_topk_scores(x2, tb, imap, k, lt, shared2x2=True)}
            med, raw = alternate(arms, args.rounds, args.iters)
            same = torch.equal(arms["ids"](), arms["scores"]()[0])
            n_px = x2.shape[0] * 4 * x2.shape[2] * x2.shape[3]
            r = {"B": 64, "rows": "128x128", "out": "256x256", "K": K, "k": k, "ids_ms": med["ids"],
                 "scores_ms": med["scores"], "ratio": med["scores"] / med["ids"], "ids_mpix_s": n_px / med["ids"] / 1e3,
                 "scores_mpix_s": n_px / med["scores"] / 1e3, "ids_equal": same, "raw_ms": raw}
            print(json.dumps({kk: v for kk, v in r.items() if kk != "raw_ms"}), flush=True)
            rec["shared2x2"].append(r)
    del x2
    torch.cuda.empty_cache()

    x8 = make_rows(dev, vocab[:1024], 8, 256, 256, 32, 1.5, seed=3)
    for K in (1024, 5632):
        t = vocab[:K]
        tb = ops.text_to_bf16(t)[0]
        imap = torch.arange(K, device=dev)

        def eager(k=5):
            xn = F.normalize(x8.float(), dim=1).flatten(2)
            p = torch.softmax(torch.einsum("bdn,kd->bkn", xn, t) / tau, dim=1)
            return p.topk(k, dim=1)

        arms = {"eager": eager, "scores": lambda: ops.eval_topk_scores(x8, tb, imap, 5, lt)}
        med, raw = alternate(arms, args.rounds, args.iters)
        n_px = 8 * 256 * 256
        r = {"B": 8, "HW": "256x256", "K": K, "k": 5, "eager_ms": med["eager"], "scores_ms": med["scores"],
             "eager_mpix_s": n_px / med["eager"] / 1e3, "scores_mpix_s": n_px / med["scores"] / 1e3,
             "speedup": med["eager"] / med["scores"], "eager_peak_gb": None, "raw_ms": raw}
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        eager()
        torch.cuda.synchronize()
        r["eager_peak_gb"] = (torch.cuda.max_memory_allocated() - base) / 1e9
        print(json.dumps({kk: v for kk, v in r.items() if kk != "raw_ms"}), flush=True)
        rec["eager"].append(r)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
