"""Embedding widths 512 / 768 / 1024 (CLIP ViT-B/32, ViT-L/14, ViT-H/14) on the kernels that take them:

    python tools/bench_wide_embeddings.py [--rounds 5] [--out profiles/r7_wide_embeddings.json]

  infonce   the headline fwd+bwd launch (rc_infonce_bf16, TS kernel), B = 64, 256 x 256, bf16, K = 256;
            TFLOP/s = 4 K D B HW / t (the S GEMM and the dX GEMM, 2 flops per multiply-add)
  rep4      the four-target launch on the decoder's 128 x 128 rows (rc_infonce_bf16_rep4), B = 64, K = 256
  topk      top-5 over K = 1024 with the fused histograms (rc_eval_topk_hist_bf16), B = 64, 256 x 256: resident X at
            D = 512, streamed X (one L2 re-read of X per 256-row text block) at 768 / 1024
  area_f32  the area-image loss at n = 64 on the fp32 CUDA-core kernel (fwd+bwd)

The widths alternate within every round (no width runs all its repetitions back to back); each entry reports the median and
the spread of the per-round means (CUDA events, warm-up excluded; the inputs are larger than the L2).  The card's name,
power limit and maximum SM clock are read in the same run.  share_of_datasheet_peak: the launch's rate over the data
sheet's dense bf16 rate for one B200 (2250 TFLOP/s at 1000 W), which a card set to a lower power limit does not reach."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from rangeclip_b200 import MetricAccumulator, losses, ops  # noqa: E402

PEAK_BF16_TFLOPS = 2250.0
WIDTHS = (512, 768, 1024)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=pl, max_sm_clock=clk)
    except Exception as e:  # pragma: no cover
        return dict(name=torch.cuda.get_device_name(0), error=str(e))


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def make_cases(dev, g):
    cases = {}
    B, HW, K = 64, 256 * 256, 256
    y = torch.randint(0, K, (B * HW,), device=dev, generator=g, dtype=torch.int32)
    w = torch.ones(B * HW, device=dev)
    h4 = 128 * 128
    y4 = torch.randint(0, K, (B * h4, 4), device=dev, generator=g, dtype=torch.int32)
    w4 = torch.ones(B * h4, 4, device=dev)
    Kt = 1024
    seg = torch.randint(0, Kt, (B, 256, 256), device=dev, generator=g)
    for D in WIDTHS:
        x = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16)
        for b in range(B):
            x[b] = torch.randn(D, HW, device=dev, generator=g).to(torch.bfloat16)
        t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
        tb = ops.text_to_bf16(t)
        x4 = x.view(B, D, 4, h4)[:, :, 0].contiguous()
        tk = torch.nn.functional.normalize(torch.randn(Kt, D, device=dev, generator=g), dim=1)
        tkb = ops.text_to_bf16(tk)[0]
        acc = MetricAccumulator(torch.eye(Kt, dtype=torch.uint8), torch.arange(Kt), device=dev)
        hist = torch.zeros(5, Kt, device=dev, dtype=torch.int64)
        cnt = torch.zeros(3, device=dev, dtype=torch.int64)
        idx = torch.arange(Kt, device=dev)
        area = torch.randn(64, D, device=dev, generator=g)
        img = torch.randn(64, D, device=dev, generator=g)
        lt = torch.tensor(-2.3, device=dev, requires_grad=True)
        ar = area.clone().requires_grad_(True)

        def area_step(ar=ar, img=img, lt=lt):
            losses.image_contrastive_loss(ar, img, lt).backward()

        cases[D] = dict(
            infonce=lambda x=x, t=t, tb=tb: ops.infonce_raw(x, t, y, w, 1 / 0.07, True, False, "bf16", t_bf16=tb),
            rep4=lambda x4=x4, t=t, tb=tb: ops.infonce_raw(x4, t, y4, w4, 1 / 0.07, True, False, "bf16", t_bf16=tb, rep=4),
            topk=lambda x=x, tk=tk, tkb=tkb, hist=hist, cnt=cnt, idx=idx, acc=acc:
                ops.eval_topk_hist(x, tk, idx, 5, seg, acc.E, acc.cmap, hist, cnt, t_bf16=tkb, want_ids=False),
            area_f32=area_step,
        )
        del acc
    return cases, dict(B=B, HW=HW, K=K, K_topk=Kt, rows_rep4=B * h4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wide_embeddings: needs a CUDA device")
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    cases, shape = make_cases(dev, g)
    names = ("infonce", "rep4", "topk", "area_f32")
    for D in WIDTHS:                                  # warm-up: module loading, smem opt-in, allocator
        for n in names:
            for _ in range(2):
                cases[D][n]()
    torch.cuda.synchronize()
    samples = {(D, n): [] for D in WIDTHS for n in names}
    for r in range(a.rounds):
        order = WIDTHS if r % 2 == 0 else WIDTHS[::-1]
        for n in names:
            for D in order:
                samples[(D, n)].append(timed(cases[D][n], a.reps))
    res = dict(card=card(), shape=shape, rounds=a.rounds, reps=a.reps, peak_bf16_tflops_datasheet=PEAK_BF16_TFLOPS, results={})
    for D in WIDTHS:
        e = {}
        for n in names:
            s = samples[(D, n)]
            e[n] = dict(ms_median=round(statistics.median(s), 4), ms_min=round(min(s), 4), ms_max=round(max(s), 4))
        t = e["infonce"]["ms_median"] * 1e-3
        tf = 4 * shape["K"] * D * shape["B"] * shape["HW"] / t / 1e12
        e["infonce"]["tflops"] = round(tf, 1)
        e["infonce"]["share_of_datasheet_peak"] = round(tf / PEAK_BF16_TFLOPS, 3)
        t4 = e["rep4"]["ms_median"] * 1e-3
        e["rep4"]["tflops"] = round(4 * shape["K"] * D * shape["rows_rep4"] / t4 / 1e12, 1)
        e["topk"]["form"] = "resident X" if D <= 512 else "streamed X"
        res["results"][str(D)] = e
    for D in WIDTHS[1:]:
        res["results"][str(D)]["infonce"]["time_vs_512"] = round(
            res["results"][str(D)]["infonce"]["ms_median"] / res["results"]["512"]["infonce"]["ms_median"], 3)
        res["results"][str(D)]["topk"]["time_vs_512"] = round(
            res["results"][str(D)]["topk"]["ms_median"] / res["results"]["512"]["topk"]["ms_median"], 3)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
