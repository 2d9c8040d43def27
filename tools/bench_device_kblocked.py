"""The sync-free text loss above 256 contrast rows (device contrast builder, K-blocked rounds with K and tau in device
memory), one process, CUDA events, medians of alternated rounds.

Public compute_loss_shared2x2 step, text term only (W_image = W_smooth = 0), fwd + bwd (loss.backward()):
  reference        contrast_builder="reference" (host round trips), K = G + 200 distractors
  device_256       contrast_builder="device", max_contrast=256: the one-launch form, distractors trimmed to fit
  device_512       max_contrast=512: two K-blocked launches per round, every distractor kept
  device_1024      max_contrast=1024: four launches per round, the last two empty
  device_512_graph the device_512 call and its backward captured in one CUDA graph, replayed
plus peak memory (torch.cuda.max_memory_allocated above what was allocated before the call), and the one-target form
(compute_loss on full-resolution rows [B, D, 256, 256]) with the reference builder and at max_contrast=512.
The rounds themselves, on one contrast set drawn by the device builder at capacity 512: the device-parameter rounds
(infonce_raw(..., dev_blocks=True)) against the host-parameter rounds on the same K rows -- times and output agreement.

B = 64, D = 512, 128^2 rows / 256^2 labels, bf16 rows; labels 1..100 in 16x16 blocks (G = 100 present), 200 random
distractors from C = 2000 (K = 300).

    python tools/bench_device_kblocked.py [--out profiles/r6_device_kblocked.json] [--rounds 5]
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rangeclip_b200 as R  # noqa: E402
from rangeclip_b200 import ops  # noqa: E402
from rangeclip_b200.losses import group_2x2  # noqa: E402
from tools.bench_shared2x2_kblocked import alternate, gpu_info, make_batch, maxrel, peak_bytes  # noqa: E402


class Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(0.07)))
        self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(0.1)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r6_device_kblocked.json"))
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_device_kblocked: needs a CUDA device")
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    B, D, h, w = 64, 512, 128, 128
    H, W = 2 * h, 2 * w
    n_labels, C, n_dis = 101, 2000, 200
    x, seg, _ = make_batch(dev, B, D, h, w, n_labels, 5)
    G = int(torch.unique(seg).gt(0).sum())
    text = torch.randn(C, D, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    sets = {"medium": {}, "hard": {}}
    kw = dict(W_image=0.0, W_smooth=0.0, k_distractors=n_dis, pct_medium=0.0, pct_hard=0.0, pct_rand=1.0)
    model = Model().to(dev)
    res = {"gpu": info, "B": B, "D": D, "rows": [h, w], "labels": [H, W], "x_dtype": "bfloat16", "foreground_labels": G,
           "k_distractors": n_dis, "C": C, "terms": "text only (W_image = W_smooth = 0), fwd + bwd"}
    got = {}

    def step(builder, cap, rows=x, fn=R.compute_loss_shared2x2, tag=None):
        def run():
            xg = rows.detach().requires_grad_(True)
            model.zero_grad(set_to_none=True)
            np.random.seed(1); torch.manual_seed(1)
            total, loss_info = fn(model, xg, seg, text, sets, None, None, contrast_builder=builder, max_contrast=cap, **kw)
            total.backward()
            got[tag] = (loss_info, total)
            return xg.grad
        return run

    # CUDA graph of the device_512 step: loss and the gradients of x and log tau in one graph
    xg_graph = x.detach().requires_grad_(True)
    params = [xg_graph, model.log_temperature_text]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            total_g, _ = R.compute_loss_shared2x2(model, xg_graph, seg, text, sets, None, None, contrast_builder="device",
                                                  max_contrast=512, **kw)
            torch.autograd.grad(total_g, params)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        total_g, info_g = R.compute_loss_shared2x2(model, xg_graph, seg, text, sets, None, None, contrast_builder="device",
                                                   max_contrast=512, **kw)
        grads_g = torch.autograd.grad(total_g, params)

    arms = {"reference": step("reference", 256, tag="reference"), "device_256": step("device", 256, tag="device_256"),
            "device_512": step("device", 512, tag="device_512"), "device_1024": step("device", 1024, tag="device_1024"),
            "device_512_graph": graph.replay}
    t_ms = alternate(arms, args.rounds, 3)
    rows = {}
    for name, fn in arms.items():
        rows[name] = dict(t_ms[name], peak_mib=peak_bytes(fn) / 2**20)
    for name in ("reference", "device_256", "device_512", "device_1024"):
        rows[name]["text_loss"] = float(got[name][1].detach())
    rows["device_512_graph"]["text_loss"] = float(total_g)
    # the contrast sets the device builder drew (same seeds for every capacity)
    for cap in (256, 512, 1024):
        np.random.seed(1); torch.manual_seed(1)
        _, aux = R.text_contrastive_loss(x, seg, text, sets, model.log_temperature_text.detach(), 0.7, n_dis, 0.0, 0.0, 1.0,
                                         "auto", return_aux=True, shared2x2=True, contrast_builder="device", max_contrast=cap)
        K, flags, n_present, n_d = aux["contrast_info"].tolist()
        rows[f"device_{cap}"].update(K=K, builder_flags=flags, present=n_present, distractors=n_d)
    res["shared2x2_step"] = rows
    print(json.dumps(rows), flush=True)

    # one target per row: compute_loss on full-resolution rows
    x_full = torch.nn.functional.interpolate(x, scale_factor=2, mode="nearest")
    arms1 = {"reference": step("reference", 256, rows=x_full, fn=R.compute_loss, tag="full_reference"),
             "device_512": step("device", 512, rows=x_full, fn=R.compute_loss, tag="full_device_512")}
    t1 = alternate(arms1, args.rounds, 1)
    res["one_target_step_256x256"] = {name: dict(t1[name], peak_mib=peak_bytes(fn) / 2**20) for name, fn in arms1.items()}
    print(json.dumps(res["one_target_step_256x256"]), flush=True)
    del x_full
    torch.cuda.empty_cache()

    # the rounds on one contrast set: device parameters at capacity 512 against host parameters on its K rows
    np.random.seed(1); torch.manual_seed(1)
    rand_idx = torch.randint(0, H * W, (B, int(0.7 * H * W)), device=dev)
    target_flat = seg.reshape(B, -1)
    counts = ops.sample_label_counts(target_flat, rand_idx, C)
    label_map, contrast, kinfo = ops.contrast_build(counts, None, None, 0, n_dis, 512, 1234)
    wt, y = ops.sample_weights(target_flat, rand_idx, label_map)
    t_norm, tb, ttb = ops.text_prepare(text, contrast, want_f32=True, want_bf16=True)
    y4, w4 = group_2x2(y.view(B, H, W)), group_2x2(wt.view(B, H, W))
    K = int(kinfo[0])
    log_tau = model.log_temperature_text.detach().reshape(1).float()
    inv_tau = math.exp(-float(log_tau))
    outs = {}

    def dev_rounds():
        outs["dev"] = ops.infonce_raw(x, t_norm, y4, w4, 0.0, True, False, "bf16", rep=4, t_bf16=(tb, ttb), k_dev=kinfo,
                                      log_tau_dev=log_tau, dev_blocks=True)
        return outs["dev"]

    def host_rounds():
        outs["host"] = ops.infonce_raw(x, t_norm[:K], y4, w4, inv_tau, True, False, "auto", rep=4)
        return outs["host"]

    t2 = alternate({"device_rounds_cap512": dev_rounds, f"host_rounds_K{K}": host_rounds}, args.rounds, 3)
    a, b = outs["dev"], outs["host"]
    agreement = {"loss_rel": abs(float(a["loss_sum"] / a["w_sum"]) - float(b["loss_sum"] / b["w_sum"])) / abs(float(b["loss_sum"] / b["w_sum"])),
                 "lse_maxrel": maxrel(a["lse"], b["lse"]), "dx_maxrel": maxrel(a["dx"].float(), b["dx"].float()),
                 "dlogtau_rel": abs(float(a["dlogtau"]) - float(b["dlogtau"])) / abs(float(b["dlogtau"]))}
    res["rounds"] = {"K": K, "capacity": 512, **t2, "agreement": agreement}
    print(json.dumps(res["rounds"]), flush=True)
    res["note"] = ("step times: device events around 3 calls each (1 for the one-target form), arms alternated per round, "
                   "inputs resident; reference = host contrast builder; the device rows never synchronise; the graph replays "
                   "the device_512 step (loss + torch.autograd.grad of x and log tau)")
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"written": args.out}))
    assert torch.isfinite(grads_g[0]).all()
    assert agreement["loss_rel"] < 1e-5 and agreement["lse_maxrel"] < 1e-5 and agreement["dx_maxrel"] < 1e-2, agreement


if __name__ == "__main__":
    main()
