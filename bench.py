#!/usr/bin/env python
"""Benchmark of the DepthCLIP loss / evaluation hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W                 # this repo's CUDA path; headline = configs[1]
    python bench.py --impl reference --gpus N --steps K ...       # reference arm: the reference's CPU path, host cores
    python bench.py --workload full_step --gpus N ...             # configs[2]: reference backbone + fused losses under DDP
    python bench.py --gpus 1 --steps K --dump-outputs DIR         # + the last timed step's outputs as DIR/<name>.npy

Headline workload (one "step" = one fused forward+backward pass over one batch): B=64 images of 256x256 pixel
embeddings, D=512, bf16, K=256 text rows (63 ground-truth labels + 193 curriculum distractors), sampling weights as in
model.py:220-228.  Prints ONE JSON line; the other BASELINE configs ride along as extra keys of that line
(with_dtext, hybrid, api_device, area = configs[3], eval = configs[4], gpu_eager = the reference's own eager CUDA
path on the same GPU, cpu_baseline / cpu_eval / cpu_full_step = configs[0] on the host cores)."""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG = dict(B=64, H=256, W=256, D=512, K=256, C=1024, G=63, tau=0.07, pct_sampling=0.7)
METRIC = "pixel_text_infonce_fwd_bwd_throughput"
UNIT = "Mpix/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY section 8d)
# ------------------------------------------------------------------------------------------------

def make_labels(B, H, W, G, gen):
    """Per image an 8x8 grid of 32x32 blocks; labels from a pool of G foreground ids, id 0 once."""
    gh, gw = H // 32, W // 32
    pick = torch.randint(1, G + 1, (B, gh, gw), generator=gen)
    pick[:, 0, 0] = 0
    return pick.repeat_interleave(32, 1).repeat_interleave(32, 2).contiguous()


def make_device_workload(device, seed, B):
    c = CFG
    g = torch.Generator(device=device).manual_seed(seed)
    D, H, W, K, C = c["D"], c["H"], c["W"], c["K"], c["C"]
    x = torch.empty(B, D, H, W, device=device, dtype=torch.bfloat16)
    for b in range(B):                                    # unit-norm rows, generated per image to bound memory
        xb = torch.randn(D, H, W, device=device, generator=g)
        x[b] = (xb / xb.norm(dim=0, keepdim=True)).to(torch.bfloat16)
    text = torch.nn.functional.normalize(torch.randn(C, D, device=device, generator=g), dim=1)
    seg = make_labels(B, H, W, c["G"], torch.Generator().manual_seed(seed)).to(device)
    # contrast set: the G ground-truth ids + (K - G) distractor ids  (curriculum 0/0.75/0.25, Q3 dict form)
    gt_ids = torch.arange(1, c["G"] + 1, device=device)
    rest = torch.arange(c["G"] + 1, C, device=device)
    distract = rest[torch.randperm(rest.numel(), device=device, generator=g)[: K - c["G"]]]
    contrast = torch.unique(torch.cat([gt_ids, distract]))
    assert contrast.numel() == K
    n_samples = int(c["pct_sampling"] * H * W)
    rand_idx = torch.randint(0, H * W, (B, n_samples), device=device, generator=g)
    return dict(x=x, text=text, seg=seg, contrast=contrast, rand_idx=rand_idx)


def similarity_sets(contrast_ids, G, C):
    """Dict-form hard sets (Q3's intended path): every GT label lists the benchmark's distractor ids, so that the
    reference's own builder (model.py:240-268) yields exactly the K contrast rows of the device workload."""
    gt = set(range(1, G + 1))
    dis = [int(v) for v in contrast_ids if int(v) not in gt]
    sets = {"medium": {}, "hard": {i: [] for i in range(C)}}
    for lab in gt:
        sets["hard"][lab] = dis
    return sets


class TemperatureHolder(torch.nn.Module):
    """The two learnable temperatures of DepthUNet (model.py:77-78) without the backbone."""

    def __init__(self, tau_text, tau_image=0.1):
        super().__init__()
        self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(tau_text)))
        self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(tau_image)))


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    """SM clock / power / throttle reasons sampled every 20 ms DURING the timed region (NVML)."""

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)
        self.max_mhz = None

    def _run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            while not self.stop.is_set():
                self.rows.append((float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), N.nvmlDeviceGetPowerUsage(h) / 1e3,
                                  int(N.nvmlDeviceGetCurrentClocksEventReasons(h))))
                self.stop.wait(0.02)
        except Exception as e:  # pragma: no cover
            self.rows.append((float("nan"), float("nan"), -1))
            self.err = repr(e)

    def __enter__(self):
        self.t.start()
        time.sleep(0.05)
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        rows = [r for r in self.rows if r[2] >= 0]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"]}
        sm = sorted(r[0] for r in rows)
        bits = 0
        for r in rows:
            bits |= r[2]
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "power_w_max": max(r[1] for r in rows),
                "samples": len(rows), "reasons": [n for b_, n in names.items() if bits & b_]}


# ------------------------------------------------------------------------------------------------
# The reference's own op sequence, device-agnostic.  On CUDA tensors it is the "GPU eager incumbent" (SURVEY 8d:
# "also time the reference's GPU eager path (fp32 and autocast-fp16) on the same B200 -- it is the real incumbent").
# ------------------------------------------------------------------------------------------------

def eager_text_infonce(pixel_embeddings, target_indices, text, rand_indices, contrast, log_tau):
    """model.py:204-228 (gather with replacement, drop label 0) and :272-291 (normalize, matmul, /tau, CE)."""
    B, D, H, W = pixel_embeddings.shape
    pred_flat = pixel_embeddings.view(B, D, -1)
    target_flat = target_indices.view(B, -1)
    pred_samples = torch.gather(pred_flat, 2, rand_indices.unsqueeze(1).expand(-1, D, -1))
    label_samples = torch.gather(target_flat, 1, rand_indices)
    valid = label_samples > 0
    pred_samples = pred_samples.permute(0, 2, 1)[valid].view(-1, D)
    label_samples = label_samples[valid].view(-1)
    t = torch.nn.functional.normalize(text[contrast], p=2, dim=1)
    pred_samples = torch.nn.functional.normalize(pred_samples, p=2, dim=1)
    mapping = torch.full((text.shape[0],), -1, dtype=torch.long, device=text.device)
    mapping[contrast] = torch.arange(contrast.shape[0], device=text.device)
    mapped = mapping[label_samples]
    logits = pred_samples @ t.T
    logits = logits / torch.exp(log_tau)
    return torch.nn.functional.cross_entropy(logits, mapped)


def eager_eval_batch(x, text, seg, E, cmap, state, k=5):
    """predict tail (model.py:164-173: normalize, einsum, topk) + metric accumulation (validate.py:88-139) in the
    reference's own form: python loops over the labels of the batch, two .item() per label."""
    B, D, H, W = x.shape
    xn = torch.nn.functional.normalize(x, dim=1).view(B, D, -1)
    tn = torch.nn.functional.normalize(text, dim=1)
    logits = torch.einsum("bdn,cd->bcn", xn, tn).view(B, -1, H, W)
    topk = logits.topk(k, dim=1).indices
    gt = seg.reshape(-1)
    tk = topk.permute(0, 2, 3, 1).reshape(-1, k)
    top1 = tk[:, 0]
    state["c1"] += E[gt, top1].sum().item()
    state["tot"] += gt.numel()
    state["ck"] += E[gt.unsqueeze(1), tk].any(dim=1).sum().item()
    ge, p1 = cmap[gt], cmap[top1]
    labels = torch.unique(torch.cat([ge, p1]))
    for lab in labels:
        pm, gm = p1 == lab, ge == lab
        state["i1"][lab.item()] = state["i1"].get(lab.item(), 0) + (pm & gm).sum().item()
        state["u1"][lab.item()] = state["u1"].get(lab.item(), 0) + (pm | gm).sum().item()
    tke = cmap[tk]
    oracle_pred = top1.clone()
    for lab in labels:
        hit = (ge == lab) & (tke == lab).any(dim=1)
        oracle_pred[hit] = lab
    for lab in labels:
        pm, gm = oracle_pred == lab, ge == lab
        state["ik"][lab.item()] = state["ik"].get(lab.item(), 0) + (pm & gm).sum().item()
        state["uk"][lab.item()] = state["uk"].get(lab.item(), 0) + (pm | gm).sum().item()


def new_eval_state():
    return dict(c1=0, ck=0, tot=0, i1={}, u1={}, ik={}, uk={})


def make_equivalences(C, seed=5):
    """Symmetric synonym pairs on 10 % of the ids as a NON-transitive chain (a~b, b~c, a!~c; SURVEY Q9), and the
    row-min class map of dataloader.py:191-202."""
    E = torch.eye(C, dtype=torch.bool)
    pairs = torch.randperm(C, generator=torch.Generator().manual_seed(seed))[: C // 10]
    for a_, b_ in zip(pairs[:-1].tolist(), pairs[1:].tolist()):
        E[a_, b_] = True
        E[b_, a_] = True
    cmap = torch.argmax(E.to(torch.uint8), dim=1)
    return E, cmap


def make_eval_batch(device, text, B, H, W, sigma, seed):
    """SURVEY 8d config 4: X = normalize(text[gt] + sigma * randn), labels = 8x8 blocks drawn from the whole vocabulary."""
    C, D = text.shape
    g = torch.Generator(device=device).manual_seed(seed)
    lab = torch.randint(0, C, (B, H // 32, W // 32), device=device, generator=g)
    seg = lab.repeat_interleave(32, 1).repeat_interleave(32, 2).contiguous()
    x = torch.empty(B, D, H, W, device=device, dtype=torch.bfloat16)
    for b in range(B):
        xb = text[seg[b]].permute(2, 0, 1) + sigma * torch.randn(D, H, W, device=device, generator=g)
        x[b] = (xb / xb.norm(dim=0, keepdim=True)).to(torch.bfloat16)
    return x, seg


# ------------------------------------------------------------------------------------------------
# CPU baselines: the UNMODIFIED reference from baseline/_ref when it is staged, else the oracle port
# ------------------------------------------------------------------------------------------------

def reference_available():
    return os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "RangeCLIP"))


def bare_reference_model(tau=0.07):
    """The reference DepthUNet without its backbone: only compute_loss / its parameters are exercised."""
    from tools.stage_reference import import_reference_model
    DepthUNet = import_reference_model()
    m = DepthUNet.__new__(DepthUNet)
    torch.nn.Module.__init__(m)
    m.device = torch.device("cpu")
    m.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(tau)))
    m.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(0.1)))
    return m


def cpu_text_step(Bc, seed=0):
    """One fwd+bwd of the pixel-text InfoNCE on CPU at the headline shape: the reference's own compute_loss (text term
    only, its own torch.randint draw) when baseline/_ref is staged, else the oracle port of the same op sequence."""
    c = CFG
    g = torch.Generator().manual_seed(seed)
    D, H, W, K, C = c["D"], c["H"], c["W"], c["K"], c["C"]
    x = torch.nn.functional.normalize(torch.randn(Bc, D, H, W, generator=g), dim=1).requires_grad_(True)
    text = torch.nn.functional.normalize(torch.randn(C, D, generator=g), dim=1)
    seg = make_labels(Bc, H, W, c["G"], g)
    contrast = torch.unique(torch.cat([torch.arange(1, c["G"] + 1), torch.arange(c["G"] + 1, c["G"] + 1 + K - c["G"])]))
    if reference_available():
        model = bare_reference_model(c["tau"])
        sets = similarity_sets(contrast.tolist(), c["G"], C)

        def step():
            x.grad = None
            loss, _ = model.compute_loss(x, seg, text, sets, None, None, W_text=1.0, W_image=0.0, W_smooth=0.0,
                                         percent_image_sampling=c["pct_sampling"], k_distractors=K - c["G"], pct_medium=0.0,
                                         pct_hard=1.0, pct_rand=0.0)
            loss.backward()
            return float(loss.detach())
        return step, Bc * H * W, "reference"
    from oracle import rangeclip_oracle as O
    rand_idx = torch.randint(0, H * W, (Bc, int(c["pct_sampling"] * H * W)), generator=g)
    log_tau = torch.log(torch.tensor(c["tau"])).requires_grad_(True)

    def step():
        x.grad = None
        loss = O.text_infonce_sampled(x, seg, text, rand_idx, contrast, log_tau)
        loss.backward()
        return float(loss.detach())
    return step, Bc * H * W, "port"


def time_host(step, steps, warmup):
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def time_cpu(Bc, steps, warmup):
    torch.set_num_threads(os.cpu_count() or 1)
    step, pix, kind = cpu_text_step(Bc)
    t = time_host(step, steps, warmup)
    return pix / t / 1e6, t, torch.get_num_threads(), kind


def cpu_eval_baseline(Bc=2, C=1024):
    """configs[4] on the host cores, bounded: predict tail + metric loops of the reference form on Bc maps, K = 1024."""
    from oracle import rangeclip_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    c = CFG
    g = torch.Generator().manual_seed(3)
    text = torch.nn.functional.normalize(torch.randn(C, c["D"], generator=g), dim=1)
    x, seg = make_eval_batch(torch.device("cpu"), text, Bc, c["H"], c["W"], 0.3, 11)
    x = x.float()
    E, cmap = make_equivalences(C)
    En, cn = E.numpy(), cmap.numpy()
    reduced = list(range(C))

    def step():
        st = O.MetricState()
        topk, _, _ = O.predict_tail(x, text, reduced, 5)
        O.metrics_accumulate(st, seg.numpy().reshape(-1), topk.permute(0, 2, 3, 1).reshape(-1, 5).numpy(), En, cn)
        return st.total
    t = time_host(step, 2, 1)
    return {"value": Bc * c["H"] * c["W"] / t / 1e6, "unit": "Mpix/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{Bc} maps 256x256, D=512, K=1024, top-5: predict tail (model.py:164-173) + metric loops (validate.py:88-139), torch/numpy CPU fp32, median of 2",
            "s_per_step": t}


def cpu_full_step_baseline(Bc=4):
    """configs[0]: the reference DepthUNet (ResNet-18-UNet+ASPP, random init) forward + hybrid loss + backward on the
    host cores, B=4, 256x256, D=512, C=33 candidate texts (K=32 foreground labels), one object per image."""
    if not reference_available():
        return {"unavailable": "baseline/_ref not staged (tools/stage_reference.py)"}
    from tools.stage_reference import import_reference_model
    torch.set_num_threads(os.cpu_count() or 1)
    DepthUNet = import_reference_model()
    torch.manual_seed(0)
    model = DepthUNet('resnet', torch.device("cpu"), embedding_dim=512, use_batch_norm=True, activation_func='relu')
    g = torch.Generator().manual_seed(1)
    depth = torch.rand(Bc, 1, 256, 256, generator=g) + 0.5
    C = 33
    text = torch.nn.functional.normalize(torch.randn(C, 512, generator=g), dim=1)
    seg = torch.randint(0, C, (Bc, 8, 8), generator=g).repeat_interleave(32, 1).repeat_interleave(32, 2).contiguous()
    sets = {"medium": [[] for _ in range(C)], "hard": [[] for _ in range(C)]}
    img = torch.nn.functional.normalize(torch.randn(Bc, 512, generator=g), dim=1)

    def step():
        model.zero_grad(set_to_none=True)
        emb, _, _ = model(depth)
        area = torch.stack([(emb[b] * (seg[b] == seg[b, 128, 128])[None]).sum(dim=(1, 2)) / (seg[b] == seg[b, 128, 128]).sum()
                            for b in range(Bc)]).detach()          # dataloader.py:286-304 (detached, Q4)
        loss, _ = model.compute_loss(emb, seg, text, sets, area, img, k_distractors=50)
        loss.backward()
        return float(loss.detach())
    t = time_host(step, 2, 1)
    return {"value": Bc * 256 * 256 / t / 1e6, "unit": "Mpix/s", "cores": torch.get_num_threads(), "kind": "reference",
            "sample": f"configs[0]: unmodified reference DepthUNet fwd + hybrid loss (text+image+smooth) + bwd, B={Bc}, 256x256, D=512, C=33, CPU fp32, median of 2",
            "s_per_step": t}


# ------------------------------------------------------------------------------------------------
# main
# ------------------------------------------------------------------------------------------------

def dist_env():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    c = CFG
    Bc = 2
    steps, warmup = max(1, min(args.steps, 5)), max(1, min(args.warmup, 1))
    val, t, cores, kind = time_cpu(Bc, steps, warmup)
    how = "the unmodified reference DepthUNet.compute_loss from baseline/_ref" if kind == "reference" else "the oracle port"
    sample = (f"B={Bc} of the B={c['B']} batch per step (same 256x256, D=512, K=256, 0.7 sampling), {how}, torch CPU fp32")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: pixel-text InfoNCE fwd+bwd, 256x256, D=512, K=256", "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def section(fn):
    """Secondary sections never take the headline line down with them."""
    try:
        return fn()
    except Exception as e:  # noqa: BLE001
        torch.cuda.empty_cache()
        return {"error": repr(e)[:300]}


DUMP_PIXELS = 8192


def dump_outputs(out_dir, dx, lse, acc):
    """Write what the headline step returns to its caller, from its last timed run, as DIR/<name>.npy: the loss and
    weight sums and dlogtau (float64), the log-sum-exp of every pixel row (float32), and dX (float32) at DUMP_PIXELS
    pixels drawn with a fixed seed, all D channels each (dx_sample[i] is pixel dx_sample_pixels[i] = b * HW + p).
    About 34 MB at the headline shape, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    B, D, HW = dx.shape
    pix = np.sort(np.random.default_rng(0).choice(B * HW, size=min(DUMP_PIXELS, B * HW), replace=False))
    pix_d = torch.from_numpy(pix).to(dx.device)
    out = {"loss_sum": acc[0], "w_sum": acc[1], "dlogtau": acc[2], "lse": lse,
           "dx_sample": dx[pix_d // HW, :, pix_d % HW].float(), "dx_sample_pixels": pix.astype(np.float64)}
    for name, v in out.items():
        if isinstance(v, torch.Tensor):
            v = v.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), v)


def run_gpu(args):
    import torch.distributed as dist
    from rangeclip_b200 import _lib, ops
    import rangeclip_b200 as R
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: keep NCCL's version banner / debug output on stderr
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=device)
    c = CFG
    B, D, H, W, K = c["B"], c["D"], c["H"], c["W"], c["K"]
    HW, M = H * W, c["B"] * H * W
    wl = make_device_workload(device, 1234 + rank, B)
    x, text, seg = wl["x"], wl["text"], wl["seg"]
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    inv_tau = 1.0 / c["tau"]
    pk = peaks()

    # per-step inputs that the loss wrapper derives from (seg, rand_idx, contrast): part of the step
    label_map = torch.full((c["C"],), -1, dtype=torch.int32, device=device)
    label_map[wl["contrast"]] = torch.arange(K, device=device, dtype=torch.int32)
    _, tb, ttb = ops.text_prepare(text, wl["contrast"], want_f32=False, want_bf16=True)
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, _lib.RC_BF16))
    ws = torch.empty(ws_bytes, device=device, dtype=torch.uint8)
    dx = torch.empty(B, D, HW, device=device, dtype=torch.bfloat16)
    lse = torch.empty(M, device=device, dtype=torch.float32)
    acc = torch.zeros(4, device=device, dtype=torch.float64)

    kernel_events = []

    def step(flags=0, record=False, dt=None, wsp=None, wsb=None):
        """sampling weights -> weight sum -> fused fwd+bwd kernel (row norms, loss, lse, dX, dlogtau)."""
        w, y = ops.sample_weights(seg.view(B, HW), wl["rand_idx"], label_map)
        acc.zero_()
        _lib.check(L.rc_weight_sum(w.data_ptr(), y.data_ptr(), M, acc[3:].data_ptr(), st), "rc_weight_sum")
        if record:      # CUDA events on the launch stream around the dominant kernel, inside the timed region
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        _lib.check(L.rc_infonce_bf16(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), K,
                                     y.data_ptr(), w.data_ptr(), inv_tau, lse.data_ptr(), acc[0:].data_ptr(),
                                     acc[1:].data_ptr(), acc[3:].data_ptr(), None, dx.data_ptr(), None if dt is None else dt.data_ptr(),
                                     acc[2:].data_ptr(), (wsp if wsp is not None else ws).data_ptr(), wsb if wsb is not None else ws_bytes,
                                     flags, st), "rc_infonce_bf16")
        if record:
            e1.record()
            kernel_events.append((e0, e1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup=3):
        """ms per call of fn: CUDA events on the launch stream, barrier + synchronize on both sides, max over ranks."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t) / steps

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    n0 = _lib.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    with ClockSampler(local) as clk:
        barrier()
        ev[0].record()
        for _ in range(args.steps):
            step(record=True)
        ev[1].record()
        barrier()
    launches = _lib.launch_count() - n0
    ms = ev[0].elapsed_time(ev[1])
    tmax = torch.tensor([ms], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax)
    loss = float(acc[0] / acc[1])
    value = world * M * args.steps / (ms * 1e-3) / 1e6
    if args.dump_outputs and rank == 0:      # before the sections below reuse dx / lse / acc
        dump_outputs(args.dump_outputs, dx, lse, acc)

    # ---- dominant kernel: average launch duration from the CUDA events recorded inside the timed region
    k_ms = sum(e0.elapsed_time(e1) for e0, e1 in kernel_events) / max(1, len(kernel_events))
    flops = 4.0 * M * K * D                      # S = X T^T and dX = P T: 2 GEMM units (dText: see with_dtext)
    achieved = flops / (k_ms * 1e-3) / 1e12
    long_region = ms > 2000.0
    peak = pk["tf_sust"] if long_region else pk["tf_burst"]
    traffic = None
    for tp in ("r2_traffic.json", "r1_traffic.json"):
        tp = os.path.join(ROOT, "profiles", tp)
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("infonce_umma_pair_kernel_bytes_per_launch")
            break
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "infonce_umma_pair_kernel<true>", "kernel_ms": k_ms,
                "peak_source": f"{pk['src']} {'sustained' if long_region else 'burst'} cuBLAS bf16",
                "algorithmic_flops_per_launch": flops}

    # ---- the same step on the TS-mode kernel (softmax tile as a tensor-memory operand; RC_INFONCE_TS_KERNEL)
    def ts_section():
        t = timed(lambda: step(flags=8), args.steps)
        return {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "loss": float(acc[0] / acc[1]),
                "tflops": flops / (t * 1e-3) / 1e12, "kernel": "infonce_ts_kernel (csrc/infonce_ts.cu), flag RC_INFONCE_TS_KERNEL"}
    ts_kernel = section(ts_section)

    # ---- the step with dText (north_star: "a matching fused backward produces dPixelEmb and dText"): 3 GEMM units
    def dtext_section():
        wsb = int(L.rc_infonce_workspace_bytes_dt(B, D, HW, K, _lib.RC_BF16))
        wsp = torch.empty(wsb, device=device, dtype=torch.uint8)
        dt = torch.zeros(K, D, device=device, dtype=torch.float32)
        t = timed(lambda: (dt.zero_(), step(dt=dt, wsp=wsp, wsb=wsb)), max(3, args.steps // 2))
        fl = 6.0 * M * K * D
        a = fl / (t * 1e-3) / 1e12
        return {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "tflops": a, "frac": a / pk["tf_burst"],
                "algorithmic_flops_per_step": fl, "dtext_abs_sum": float(dt.abs().sum()),
                "note": "fused kernel also stores G = rs (P - onehot) (bf16 [B][HW][Kp]); split-K tcgen05 GEMM dT = G^T X"}
    with_dtext = section(dtext_section)

    model = TemperatureHolder(c["tau"]).to(device)
    sets = similarity_sets(wl["contrast"].tolist(), c["G"], c["C"])

    def api_loss(xd, sd, W_image=0.0, W_smooth=0.0, area=None, img=None, precision="auto", builder="reference"):
        return R.compute_loss(model, xd, sd, text, sets, area, img, W_text=1.0, W_image=W_image, W_smooth=W_smooth,
                              percent_image_sampling=c["pct_sampling"], k_distractors=K - c["G"], pct_medium=0.0, pct_hard=1.0,
                              pct_rand=0.0, precision=precision, contrast_builder=builder)

    # ---- end to end through the public drop-in API with HOST buffers (pinned), loss read back
    e2e = None
    if not args.no_e2e:
        xh = x.cpu().pin_memory()
        segh = seg.cpu().pin_memory()
        e_steps = max(2, min(args.steps, 5))
        h2d = xh.numel() * 2 + segh.numel() * 8
        d2h = 6 * 4

        # as a DataLoader with pinned memory does: the copy of step i + 1 runs on a side stream while step i computes;
        # every step's inputs cross PCIe inside the timed region and every step's loss_info is read back
        copy_stream = torch.cuda.Stream(device=device)

        def fetch():
            with torch.cuda.stream(copy_stream):
                xd = xh.to(device, non_blocking=True)
                sd = segh.to(device, non_blocking=True)
                ev = torch.cuda.Event(); ev.record(copy_stream)
            return xd, sd, ev

        def e2e_step(batch, prefetch):
            xd, sd, ev = batch
            nxt = fetch() if prefetch else None
            torch.cuda.current_stream().wait_event(ev)
            xd.record_stream(torch.cuda.current_stream()); sd.record_stream(torch.cuda.current_stream())
            total, info = api_loss(xd.requires_grad_(True), sd)
            total.backward()
            return info["total_loss"], nxt

        np.random.seed(0); torch.manual_seed(0)
        e2e_step(fetch(), False)
        barrier()
        t0 = time.perf_counter()
        batch = fetch()
        for i in range(e_steps):
            _, batch = e2e_step(batch, i + 1 < e_steps)
        barrier()
        dt_e = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt_e, op=dist.ReduceOp.MAX)
        e2e = {"value": world * M * e_steps / float(dt_e) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e_steps,
               "api": "rangeclip_b200.compute_loss(...)+backward, pinned host X/seg copied on a side stream (next step's copy overlaps this step's kernels), loss_info read back"}
        del xh, segh

    # ---- the public API with X resident on the device: what the host-side set builders and the autograd plumbing cost
    def api_device_section():
        xg = x.detach().requires_grad_(True)

        params = [xg] + list(model.parameters())

        def f():      # autograd.grad: the gradient tensors themselves (backward() on a LEAF x adds autograd's own 4.3 GB copy into x.grad)
            total, info = api_loss(xg, seg)
            return torch.autograd.grad(total, params, allow_unused=True)
        np.random.seed(0); torch.manual_seed(0)
        t = timed(f, max(3, args.steps // 2), 2)
        return {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "kernel_step_ms": ms / args.steps,
                "overhead_ms": t - ms / args.steps,
                "api": "compute_loss(text term)+backward, bf16 X on the device, contrast-set builder + loss_info readback inside"}
    api_device = section(api_device_section)

    # ---- the same call with the device-side contrast-set builder (SURVEY 8f-2): no host synchronisation inside compute_loss
    def api_sync_free_section():
        xg = x.detach().requires_grad_(True)
        params = [xg] + list(model.parameters())
        info_box = []

        def f():
            total, info = api_loss(xg, seg, builder="device")
            info_box[:] = [info]
            return torch.autograd.grad(total, params, allow_unused=True)
        np.random.seed(0); torch.manual_seed(0)
        t = timed(f, max(3, args.steps // 2), 2)
        li = info_box[0]
        return {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "kernel_step_ms": ms / args.steps,
                "overhead_ms": t - ms / args.steps, "over_kernel_step": t / (ms / args.steps), "loss": li["total_loss"],
                "api": "compute_loss(text term, contrast_builder='device')+backward, bf16 X on the device: label histogram -> "
                       "rc_contrast_build -> rc_infonce_bf16_dyn, loss_info fetched lazily (read once after the timed loop)"}
    api_sync_free = section(api_sync_free_section)

    # ---- the sync-free call + backward captured in ONE CUDA graph (possible because nothing in it talks to the host): replay cost
    def api_graph_section():
        xg = x.detach().requires_grad_(True)
        params = [xg] + list(model.parameters())
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                total, _info = api_loss(xg, seg, builder="device")
                torch.autograd.grad(total, params, allow_unused=True)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            total, info = api_loss(xg, seg, builder="device")
            grads = torch.autograd.grad(total, params, allow_unused=True)
        t = timed(graph.replay, max(3, args.steps // 2), 2)
        out = {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "over_kernel_step": t / (ms / args.steps),
               "loss": info["total_loss"], "api": "torch.cuda.graph over compute_loss(contrast_builder='device') + autograd.grad; replay only"}
        del graph, grads, total
        return out
    api_graph = section(api_graph_section)

    # ---- hybrid loss (text + area-image + smoothness) through compute_loss, device-resident X, bf16 and fp32 X
    def hybrid_section():
        from rangeclip_b200 import pool_objects_per_image
        g = torch.Generator(device=device).manual_seed(77)
        img = torch.nn.functional.normalize(torch.randn(B, D, device=device, generator=g), dim=1)
        labels = seg[:, 128, 128].tolist()
        out = {}
        for name, xin in (("bf16", x), ("fp32", None)):
            if xin is None:
                xin = x.float()
            xg = xin.detach().requires_grad_(True)

            params = [xg] + list(model.parameters())

            def f():
                with torch.no_grad():      # dataloader.py:205: prepare_image_contrast_data is @torch.no_grad (Q4)
                    area = pool_objects_per_image(xg, seg, list(range(B)), labels)
                total, info = api_loss(xg, seg, W_image=0.5, W_smooth=2e2, area=area, img=img)
                torch.autograd.grad(total, params, allow_unused=True)
                return info
            np.random.seed(0); torch.manual_seed(0)
            t = timed(f, max(5, args.steps // 2), 2)
            info = f()
            out[name] = {"ms_per_step": t, "value": world * M / (t * 1e-3) / 1e6, "unit": UNIT, "total_loss": info["total_loss"],
                         "text": info["text_contrastive_loss"], "image": info["image_contrastive_loss"], "smooth": info["smoothness_loss"]}
            del xg, xin
            torch.cuda.empty_cache()
        out["fp32_over_bf16"] = out["fp32"]["ms_per_step"] / out["bf16"]["ms_per_step"]
        out["note"] = ("compute_loss(W_text=1, W_image=0.5, W_smooth=200)+backward, one object per image (n=B), X on the device; "
                       "fp32 X = what the reference decoder emits (decoder.py:115): one pre-pass gives the bf16 copy, the smoothness sums "
                       "and the 4-bit difference signs (rc_infonce_prepass_tv), the backward runs from those signs (rc_tv_bwd_codes)")
        return out
    hybrid = None if args.no_hybrid else section(hybrid_section)

    # ---- the contrast set beyond one launch's 256 rows (model.py:268: K is data dependent; predict default 300 negatives)
    def kcliff_section():
        out = {"K256_ms": ms / args.steps}
        for K2 in (300, 512):
            g = torch.Generator(device=device).manual_seed(K2)
            t2 = torch.nn.functional.normalize(torch.randn(K2, D, device=device, generator=g), dim=1)
            y2 = torch.randint(0, K2, (M,), device=device, generator=g, dtype=torch.int32)
            w2 = torch.ones(M, device=device)
            t = timed(lambda: ops.infonce_raw(x, t2, y2, w2, inv_tau, True, False, "auto"), 3, 1)
            out[f"K{K2}_ms"] = t
            out[f"K{K2}_over_K256"] = t / (ms / args.steps)
            del t2, y2, w2
        torch.cuda.empty_cache()
        return out
    kcliff = None if args.no_kcliff else section(kcliff_section)

    # ---- configs[3]: area-image alignment stress, 64 object masks per image, B=64: masked pooling + image InfoNCE n=4096
    def area_section():
        n_obj = 64
        seg64 = (torch.arange(64, device=device).view(8, 8) + 1).repeat_interleave(32, 0).repeat_interleave(32, 1)[None].expand(B, H, W).contiguous()
        lut = torch.full((B, 65), -1, dtype=torch.int32, device=device)
        lut[:, 1:] = torch.arange(B * n_obj, device=device, dtype=torch.int32).view(B, n_obj)
        n = B * n_obj
        out = {}
        for name, xin in (("bf16", x), ("fp32", x[: B // 2].float())):
            Bx = xin.shape[0]
            esz = xin.element_size()
            t_f = timed(lambda: ops.pool_forward(xin, seg64[:Bx], lut[:Bx], True, Bx * n_obj), 5, 2)
            pooled, cnt = ops.pool_forward(xin, seg64[:Bx], lut[:Bx], True, Bx * n_obj)
            gup = torch.randn(Bx * n_obj, D, device=device)
            t_b = timed(lambda: ops.pool_backward(gup, cnt, seg64[:Bx], lut[:Bx], True, tuple(xin.shape), xin.dtype), 5, 2)
            px = Bx * HW
            out[name] = {"B": Bx, "fwd_ms": t_f, "bwd_ms": t_b,
                         "fwd_GBs": px * (D * esz + 8) / (t_f * 1e-3) / 1e9, "bwd_GBs": px * (D * esz + 8) / (t_b * 1e-3) / 1e9,
                         "fwd_frac_of_hbm": px * (D * esz + 8) / (t_f * 1e-3) / 1e9 / pk["hbm"],
                         "bwd_frac_of_hbm": px * (D * esz + 8) / (t_b * 1e-3) / 1e9 / pk["hbm"]}
            del pooled, cnt, gup
        del xin
        torch.cuda.empty_cache()
        pooled, _ = ops.pool_forward(x, seg64, lut, True, n)
        g = torch.Generator(device=device).manual_seed(31)
        imgs = torch.nn.functional.normalize(torch.randn(n, D, device=device, generator=g), dim=1)
        area = pooled.detach().requires_grad_(True)

        def f():
            area.grad = None
            R.image_contrastive_loss(area, imgs, model.log_temperature_image).backward()
        t_i = timed(f, 5, 2)

        def f_eager():
            area.grad = None
            a = torch.nn.functional.normalize(area, dim=1)
            i_ = torch.nn.functional.normalize(imgs, dim=1)
            torch.nn.functional.cross_entropy(a @ i_.T / torch.exp(model.log_temperature_image), torch.arange(n, device=device)).backward()
        t_e = timed(f_eager, 5, 2)
        out["image_infonce_n4096"] = {"ms": t_i, "eager_torch_ms": t_e, "n": n,
                                      "note": "model.py:304-321 fwd+bwd, tensor cores over blocks of 256 candidates vs eager cuBLAS+softmax"}
        out["peak_hbm_GBs"] = pk["hbm"]
        out["note"] = "algorithmic bytes per pixel D*elt + 8 (labels); 64 masks = the 32x32 blocks of every image"
        return out
    area_cfg = None if args.no_area else section(area_section)

    # ---- evaluation workload (configs[4]): top-5 over a K=1024 vocabulary + equivalence-aware histograms,
    #      5000 maps = 78 batches of 64 + 1 of 8, round-robin over ranks, ONE all-reduce of the int64 state
    ev = None
    eager_eval = None
    if not args.no_eval:
        from rangeclip_b200 import MetricAccumulator
        from rangeclip_b200.distributed import all_reduce_metrics, shard_batches
        Ce = 1024
        ge = torch.Generator(device=device).manual_seed(99)
        text_e = torch.nn.functional.normalize(torch.randn(Ce, D, device=device, generator=ge), dim=1)
        _, tbe, _ = ops.text_prepare(text_e, None, want_f32=False, want_bf16=True)
        idx_map = torch.arange(Ce, device=device)
        E, cmap = make_equivalences(Ce)
        n_batches = 79
        mine = list(shard_batches(n_batches, rank, world))
        # two resident batches of embeddings built FROM their labels (SURVEY 8d config 4: ~50 % top-1), re-used round robin
        pool_b = [make_eval_batch(device, text_e, B, H, W, 0.3, 500 + i) for i in range(2)]
        acc_m = MetricAccumulator(E, cmap, device=device)

        def eval_batch(gb):
            nb_ = B if gb < n_batches - 1 else 8
            xe, se = pool_b[gb % 2]
            # one fused kernel per batch: top-5 on the tensor cores, ids -> class histograms in registers (no id tensor)
            acc_m.update_from_embeddings(xe[:nb_], text_e, idx_map, se[:nb_], 5, batch_index=gb, t_bf16=tbe, want_ids=False)
            return nb_ * HW

        eval_batch(0); acc_m = MetricAccumulator(E, cmap, device=device)
        barrier()
        ee = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ee[0].record()
        pix = 0
        for gb in mine:
            pix += eval_batch(gb)
        all_reduce_metrics(acc_m)
        ee[1].record()
        barrier()
        tm = torch.tensor([ee[0].elapsed_time(ee[1])], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        fin = acc_m.finalize(pool_b[(n_batches - 1) % 2][1][:8])
        tot_pix = (78 * B + 8) * HW
        ev = {"value": tot_pix / (float(tm) * 1e-3) / 1e6, "unit": "Mpix/s", "ms": float(tm), "maps": 78 * B + 8, "K": Ce, "top_k": 5,
              "total_pixels_counted": fin["total_pixels"], "pixel_accuracy_t1": fin["pixel_accuracy_t1"],
              "pixel_accuracy_tk": fin["pixel_accuracy_tk"], "mIoU_t1": fin["mIoU_t1"], "mIoU_tk": fin["mIoU_tk"],
              "tensor_tflops": 2.0 * Ce * D * tot_pix / (float(tm) * 1e-3) / 1e12,
              "frac_of_burst_peak": 2.0 * Ce * D * tot_pix / (float(tm) * 1e-3) / 1e12 / pk["tf_burst"],
              "frac_of_sustained_peak": 2.0 * Ce * D * tot_pix / (float(tm) * 1e-3) / 1e12 / pk["tf_sust"],
              "note": "78x64+8 synthetic maps, X = normalize(text[gt] + 0.3 randn) (two resident batches re-used), synonym chain on 10% of the ids; "
                      "fused tcgen05 top-5 + equivalence-aware histograms (one kernel per batch) + fold, one int64 all-reduce at the end"}
        assert fin["total_pixels"] == tot_pix

        # the top-k kernel alone (rc_eval_topk_bf16, ids written) on one resident batch: what the scan / MMA halves sustain
        def eval_kernel_section():
            xe, _ = pool_b[0]
            out = {}
            for kk in (5, 1):
                # a kernel timed ALONE is compared with the burst peak: let the 0.3 s evaluation loop above drain out of the power window
                torch.cuda.synchronize(); time.sleep(1.5)
                t = timed(lambda: ops.eval_topk(xe, text_e, idx_map, kk, "bf16", t_bf16=tbe), 5, 2)
                tf = 2.0 * Ce * D * B * HW / (t * 1e-3) / 1e12
                out[f"top{kk}"] = {"ms": t, "value": B * HW / (t * 1e-3) / 1e6, "unit": "Mpix/s", "tflops": tf, "frac_of_burst_peak": tf / pk["tf_burst"]}
            out["note"] = "eval_topk_umma_kernel (CTA-pair form) on one batch of 64 maps, K=1024, ids [B,k,HW] int64 written; 1.5 s idle before each timing (burst regime; the 5000-map loop above is the sustained one)"
            return out
        ev["kernel"] = section(eval_kernel_section)

        # the reference's eager CUDA evaluation of ONE batch (predict tail + python metric loops with .item() syncs)
        def eager_eval_section():
            xe, se = pool_b[0]
            Ed, cd = E.to(device), cmap.to(device)
            out = {}
            for name, ac in (("fp32", False), ("autocast_fp16", True)):
                def f():
                    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=ac):
                        eager_eval_batch(xe.float(), text_e, se, Ed, cd, new_eval_state())
                f()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                t = time.perf_counter() - t0
                out[name] = {"ms_per_batch": t * 1e3, "value": B * HW / t / 1e6, "unit": "Mpix/s"}
                torch.cuda.empty_cache()
            out["note"] = "model.py:164-173 + validate.py:88-139 as written (einsum -> [B,K,HW] logits -> topk -> per-label python loops), one batch of 64 maps, K=1024"
            return out
        if rank == 0 and not args.no_eager:
            eager_eval = section(eager_eval_section)
            if isinstance(eager_eval, dict) and "fp32" in eager_eval:
                eager_eval["ours_over_eager_fp32"] = ev["value"] / world / eager_eval["fp32"]["value"]
                eager_eval["ours_over_eager_autocast"] = ev["value"] / world / eager_eval["autocast_fp16"]["value"]
        del pool_b
        torch.cuda.empty_cache()

    # ---- the reference's eager CUDA text loss on the same GPU (the incumbent): fp32 and autocast-fp16, largest B that fits
    def gpu_eager_section():
        out = {}
        log_tau = torch.log(torch.tensor(c["tau"], device=device)).requires_grad_(True)
        for name, ac in (("fp32", False), ("autocast_fp16", True)):
            Bg = B
            while Bg >= 4:
                try:
                    xg = x[:Bg].float().requires_grad_(True)
                    sg, rg = seg[:Bg], wl["rand_idx"][:Bg]

                    def f():
                        xg.grad = None
                        with torch.autocast("cuda", dtype=torch.float16, enabled=ac):
                            l_ = eager_text_infonce(xg, sg, text, rg, wl["contrast"], log_tau)
                        l_.backward()
                        return l_
                    t = timed(f, 3, 1) if world == 1 else None
                    if t is None:
                        f(); torch.cuda.synchronize(); t0 = time.perf_counter(); f(); torch.cuda.synchronize(); t = (time.perf_counter() - t0) * 1e3
                    out[name] = {"B": Bg, "ms_per_step": t, "value": Bg * HW / (t * 1e-3) / 1e6, "unit": UNIT, "loss": float(f().detach())}
                    del xg
                    torch.cuda.empty_cache()
                    break
                except torch.OutOfMemoryError:
                    xg = None
                    torch.cuda.empty_cache()
                    Bg //= 2
        out["note"] = ("model.py:204-228,272-291 op sequence on CUDA tensors (gather with replacement, normalize, matmul, /tau, CE) + autograd, "
                       "fp32 X as the decoder emits it; per-GPU numbers")
        return out
    gpu_eager = None
    if rank == 0 and not args.no_eager:
        gpu_eager = section(gpu_eager_section)
    barrier()
    vs_gpu_eager = None
    if isinstance(gpu_eager, dict) and "fp32" in gpu_eager:
        vs_gpu_eager = {"kernel_step_over_eager_fp32": (value / world) / gpu_eager["fp32"]["value"],
                        "kernel_step_over_eager_autocast_fp16": (value / world) / gpu_eager["autocast_fp16"]["value"]}
        if isinstance(hybrid, dict) and "fp32" in hybrid:
            vs_gpu_eager["note"] = "apples to apples at the API level (fp32 X in, fp32 dX out): see hybrid.fp32 / api_device vs gpu_eager"

    # ---- the same loss when X comes out of the reference decoder (nearest x2 of a 128x128 map, quirk Q8; SURVEY 8f-1):
    #      one embedding row per 2x2 block with its four targets -- informational, not the headline (configs[1] is
    #      defined on independent per-pixel embeddings)
    shared = None
    if not args.no_shared:
        from rangeclip_b200.losses import group_2x2
        xl = x[:, :, ::2, ::2].contiguous()                  # [B, D, 128, 128]: the tensor before decoder.py:113
        hw = xl.shape[2] * xl.shape[3]
        dxl = torch.empty(B, D, hw, device=device, dtype=torch.bfloat16)
        lsel = torch.empty(B * hw, device=device, dtype=torch.float32)
        wsl_bytes = int(L.rc_infonce_workspace_bytes(B, D, hw, K, _lib.RC_BF16))
        wsl = torch.empty(wsl_bytes, device=device, dtype=torch.uint8)

        def shared_step():
            w, y = ops.sample_weights(seg.view(B, HW), wl["rand_idx"], label_map)
            acc.zero_()
            _lib.check(L.rc_weight_sum(w.data_ptr(), y.data_ptr(), M, acc[3:].data_ptr(), st), "rc_weight_sum")
            y4, w4 = group_2x2(y.view(B, H, W)), group_2x2(w.view(B, H, W))
            _lib.check(L.rc_infonce_bf16_rep4(xl.data_ptr(), _lib.RC_BF16, B, D, hw, tb.data_ptr(), ttb.data_ptr(), K,
                                              y4.data_ptr(), w4.data_ptr(), inv_tau, lsel.data_ptr(), acc[0:].data_ptr(),
                                              acc[1:].data_ptr(), acc[3:].data_ptr(), None, dxl.data_ptr(), None,
                                              acc[2:].data_ptr(), wsl.data_ptr(), wsl_bytes, 0, st), "rc_infonce_bf16_rep4")

        ts = timed(shared_step, args.steps)
        shared = {"value": world * M / (ts * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ts,
                  "loss": float(acc[0] / acc[1]),
                  "note": "full-resolution pixels per second when X = nearest_x2 of a 128x128 decoder output: "
                          "rc_infonce_bf16_rep4 on the 128x128 distinct rows (sampling weights + 2x2 grouping inside the step)"}
        del xl, dxl, lsel, wsl

    cpu = cpu_eval = cpu_full = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, t, cores, kind = time_cpu(2, 3, 1)
        how = "unmodified reference compute_loss (baseline/_ref)" if kind == "reference" else "oracle port"
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"B=2 of the B=64 batch (256x256, D=512, K=256, 0.7 sampling), {how}, torch CPU fp32, median of 3",
               "s_per_step": t}
        cpu_eval = section(cpu_eval_baseline)
        cpu_full = section(cpu_full_step_baseline)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "configs[1]: pixel-text InfoNCE fwd+bwd, B=64/GPU, 256x256, D=512, K=256 (63 GT + 193 distractors), "
                                   "0.7 sampling with replacement", "outputs": "loss, lse, dX (bf16), dlogtau",
                       "l2": "inputs (4.3 GB bf16 per step) exceed the 126 MB L2; no flush needed",
                       "step": "rc_sample_weights + rc_weight_sum + fused tcgen05 kernel (row norms, S GEMM, softmax/CE, dX GEMM, projection)"},
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "ts_kernel": ts_kernel, "with_dtext": with_dtext, "api_device": api_device, "api_sync_free": api_sync_free, "api_graph": api_graph, "hybrid": hybrid, "kcliff": kcliff,
            "area": area_cfg, "eval": ev, "gpu_eager": gpu_eager, "vs_gpu_eager": vs_gpu_eager, "gpu_eager_eval": eager_eval,
            "cpu_eval": cpu_eval, "cpu_full_step": cpu_full, "shared2x2": shared, "loss": loss,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="infonce", choices=["infonce", "full_step"])
    for flag in ("e2e", "cpu", "eval", "shared", "hybrid", "area", "eager", "kcliff"):
        ap.add_argument(f"--no-{flag}", action="store_true")
    ap.add_argument("--batch", type=int, default=64, help="full_step: images per GPU")
    ap.add_argument("--variant", default="shared2x2", choices=["shared2x2", "full", "eager"], help="full_step: loss path")
    ap.add_argument("--phase", default="step", choices=["step", "backbone", "nosync"], help="full_step: what is timed")
    ap.add_argument("--builder", default="device", choices=["device", "reference"],
                    help="full_step: contrast-set builder of compute_loss (device = sync-free, SURVEY 8f-2; reference = host RNG parity)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "infonce" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the headline workload (--workload infonce --impl ours)")
    if args.workload == "full_step":
        from tools.full_step import run_full_step
        run_full_step(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
