"""Embeddings wider than 512 channels: D = 768 (CLIP ViT-L/14) and 1024 (ViT-H/14) through the tensor-core InfoNCE kernels,
the streamed-X tensor-core top-k and the wide form of the fp32 CUDA-core kernels (640 < D <= 1024 included).

Most checks here are the suite's own checks at D = 512, run again at the new widths: the per-row fp64 bounds of
oracle/infonce_rows.py for every InfoNCE form, the tie-aware top-k with its fused histograms, the R = 4 top-k against the
upsampled launch, and the sync-free public loss against the oracle.  New here: TS against SS bit for bit at the new widths,
the fp32 kernels' 1e-5 contract at D in {640, 768, 1024}, the public calls at D = 768, and one launch whose X has more than
2^31 elements."""
import functools
import math
import os
import sys

import pytest
import torch

from oracle import infonce_rows as OR
from oracle import rangeclip_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import test_gpu_dev_kblocked as dev_kb            # noqa: E402  (the D = 512 checks, reused at the new widths)
import test_gpu_device_builder as dev_builder     # noqa: E402
import test_gpu_eval_shared2x2 as eval2x2         # noqa: E402
import test_gpu_infonce_rows as rows              # noqa: E402
import test_gpu_shared2x2_kblocked as shared2x2_kb  # noqa: E402

pytestmark = pytest.mark.gpu

WIDE = [768, 1024]
TS, SS = 0, 32


def dev():
    return torch.device("cuda:0")


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------------------------
# tensor-core InfoNCE: every form against the per-row fp64 bounds
# ---------------------------------------------------------------------------------------------------------------------
# (form, B, D, HW, K, R): B = 1, HW = 328 is three tiles (an odd number of tile pairs with B = 1), HW = 200 a partial tile
FORMS = [(f, B, D, HW, K, R) for D in WIDE for (f, B, HW, K, R) in [
    ("ts", 1, 328, 200, 1), ("ts", 2, 200, 256, 4),
    ("ss", 1, 328, 130, 1), ("ss", 2, 136, 256, 4),
    ("fwd", 1, 328, 256, 1), ("fwd", 1, 200, 70, 4),
    ("dyn", 1, 328, 150, 1), ("dyn", 2, 200, 256, 4),
    ("f32x", 1, 328, 200, 1),
]]


@pytest.mark.parametrize("tau", [0.07, 0.02])
@pytest.mark.parametrize("form", FORMS, ids=rows._form_id)
def test_rows_single_launch_wide(form, tau):
    rows.test_rows_single_launch(form, tau)


KB_FORMS = [("kblocked", 2, 768, 200, 300, 1), ("kblocked", 1, 1024, 200, 700, 4), ("kblocked", 2, 1024, 72, 300, 4),
            ("kblocks", 1, 768, 256, 700, 1), ("kblocks", 1, 1024, 512, 300, 1)]


@pytest.mark.parametrize("tau", [0.07, 0.02])
@pytest.mark.parametrize("form", KB_FORMS, ids=rows._form_id)
def test_rows_kblocked_wide(form, tau):
    rows.test_rows_kblocked(form, tau)


@pytest.mark.parametrize("tau", [0.07, 0.02])
@pytest.mark.parametrize("rep,D,K", [(1, 768, 300), (4, 768, 700), (1, 1024, 700), (4, 1024, 300)])
def test_dev_kblocked_rows_wide(rep, D, K, tau):
    """K-blocked rounds with K and log tau in device memory"""
    dev_kb.test_dev_rounds_rows_inside_the_fp64_bound(rep, D, K, tau)


@pytest.mark.parametrize("D", WIDE)
@pytest.mark.parametrize("rep", [1, 4])
def test_dev_kblocked_equals_host_rounds_and_empty_blocks_are_inert(rep, D):
    """device K against host K at K = 300 and 700; valid K = 300 at capacity 512 and 1024 (blocks 2, 3 empty): identical"""
    for K in (300, 700):
        dev_kb.test_dev_rounds_equal_the_host_parameter_rounds(rep, D, K)
    B, HW = 2, 136
    x, t, y, w = OR.make_case(B, D, HW, 300, rep, seed=41 + rep + D)
    xd, yd, wd = x.to(dev()).to(torch.bfloat16), y.to(dev()), w.to(dev())
    log_tau = math.log(0.07)
    dev_kb._assert_identical(dev_kb._dev_rounds(xd, t, yd, wd, 512, log_tau), dev_kb._dev_rounds(xd, t, yd, wd, 1024, log_tau))


@pytest.mark.parametrize("tau", [0.07, 0.02])
@pytest.mark.parametrize("D", WIDE)
@pytest.mark.parametrize("rep", [1, 4])
def test_ts_equals_ss_bit_for_bit(rep, D, tau):
    """the TS and SS backward kernels give the same dX and lse bits at the new widths (one launch and K-blocked rounds)"""
    from rangeclip_b200 import ops
    B, HW = 1, 328
    for K in (200, 300):
        x, t, y, w = OR.make_case(B, D, HW, K, rep, seed=D + K + rep)
        xd, td, yd, wd = x.to(dev()).to(torch.bfloat16), t.to(dev()), y.to(dev()), w.to(dev())
        prec = "bf16" if K <= 256 else "kblocked"
        r = [ops.infonce_raw(xd, td, yd, wd, 1 / tau, True, False, prec, rep=rep, flags=f) for f in (TS, SS)]
        torch.cuda.synchronize()
        if K <= 256:
            assert torch.equal(r[0]["dx"].view(torch.int16), r[1]["dx"].view(torch.int16))
            assert torch.equal(r[0]["lse"].view(torch.int32), r[1]["lse"].view(torch.int32))
            for k in ("loss_sum", "w_sum", "dlogtau"):
                assert float(r[0][k]) == float(r[1][k]), k


# ---------------------------------------------------------------------------------------------------------------------
# fp32 CUDA-core kernels, 512 < D <= 1024
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tau", [0.07, 0.02])
@pytest.mark.parametrize("D", [640, 768, 1024, 516])
def test_fp32_kernel_wide(D, tau):
    """loss, lse, dX, dText and dlogtau of rc_infonce_f32 against fp64 at 1e-5 relative"""
    from rangeclip_b200 import ops
    B, HW, K = 2, 72, 60
    x, t, y, w = OR.make_case(B, D, HW, K, 1, seed=77 + D)
    r = ops.infonce_raw(x.to(dev()), t.to(dev()), y.to(dev()), w.to(dev()), 1 / tau, True, True, "fp32")
    torch.cuda.synchronize()
    assert r["precision"] == "fp32"
    ref = rows._ref(x, t, y, w, 1 / tau)
    dx = rows._rows(r["dx"], B, D, HW)
    rows._check_rows(f"simt D={D} tau={tau} dx", (dx - ref["dx"]).norm(dim=1), OR.dx_bound_f32(ref, D))
    rows._check_rows(f"simt D={D} tau={tau} lse", (r["lse"].double().cpu() - ref["lse"]).abs(), 1e-5 * (ref["lse"].abs() + 1))
    assert abs(float(r["loss_sum"]) - float(ref["loss_sum"])) <= 1e-5 * abs(float(ref["loss_sum"]))
    dlt_scale = float(ref["cj"].abs().sum())                                 # dlogtau = -sum_rows cj: relative to its terms
    assert abs(float(r["dlogtau"]) - float(ref["dlogtau"])) <= 1e-5 * dlt_scale
    assert maxrel(r["dt"], ref["dt"]) < 1e-5
    # the public fp32 entry (x's rows as the fp64 oracle of the rangeclip model file sees them)
    ref2 = O.infonce_dense(rows._rows(x, B, D, HW), t, y, w, 1 / tau)
    assert abs(float(r["loss_sum"] / r["w_sum"]) - float(ref2["loss"])) <= 1e-5 * abs(float(ref2["loss"]))


@pytest.mark.parametrize("D", [640, 768, 1024])
@pytest.mark.parametrize("k", [1, 5])
def test_fp32_topk_wide(D, k):
    """rc_eval_topk_f32: ids against the fp64 ranking, tie-aware"""
    from rangeclip_b200 import ops
    g = torch.Generator().manual_seed(D + k)
    B, H, W, K = 2, 8, 12, 300
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1)
    x = t[torch.randint(0, K, (B, H, W), generator=g)].permute(0, 3, 1, 2) + 0.5 * torch.randn(B, D, H, W, generator=g)
    idx = torch.arange(K) * 3
    out = ops.eval_topk(x.to(dev()), t.to(dev()), idx.to(dev()), k, "fp32").cpu()
    logits = torch.einsum("bdn,cd->bcn", torch.nn.functional.normalize(x.double(), dim=1).reshape(B, D, H * W), t.double())
    ref_v = logits.topk(k, dim=1).values                                     # [B, k, HW]
    got = torch.gather(logits, 1, (out.reshape(B, k, H * W) // 3))
    assert bool(((got - ref_v).abs() < 1e-5).all())                          # the same values in the same order (ties either way)
    assert bool((out.reshape(B, k, -1).sort(dim=1).values.diff(dim=1) != 0).all()) if k > 1 else True


# ---------------------------------------------------------------------------------------------------------------------
# tensor-core top-k with X streamed
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,D,H,W,C,neg", [(2, 768, 16, 16, 1024, 300), (1, 1024, 16, 24, 150, 50), (1, 768, 8, 16, 40, 300),
                                           (3, 1024, 16, 16, 1400, 1100)])
def test_topk_streamed_x_device_candidates(B, D, H, W, C, neg):
    """ids tie-aware against fp64 for K up to 1024 top-5 and K <= 256, single-CTA (one tile) and CTA-pair (odd tile counts),
    the device-sized candidate set, and the fused histograms bit-identical to those of the returned ids"""
    dev_builder.test_predict_with_device_side_candidate_set(B, D, H, W, C, neg)


@pytest.mark.parametrize("B,D,h,w,K,k,xdtype,bad_gt", [
    (1, 768, 8, 16, 1024, 5, torch.bfloat16, False),
    (3, 1024, 12, 16, 1024, 5, torch.bfloat16, True),
    (1, 768, 24, 16, 1024, 1, torch.float32, False),
    (2, 1024, 10, 20, 200, 5, torch.bfloat16, True),
    (2, 768, 16, 16, 300, 3, torch.float32, True),
])
def test_topk_streamed_x_rep4_equals_upsampled_launch(B, D, h, w, K, k, xdtype, bad_gt):
    eval2x2.test_rep4_bit_exact_against_upsampled_launch(B, D, h, w, K, k, xdtype, bad_gt)


@pytest.mark.parametrize("D", WIDE)
@pytest.mark.parametrize("k", [1, 5])
def test_topk_streamed_x_host_k_against_fp64(D, k):
    """K = 1024 top-1 / top-5 through rc_eval_topk_bf16: tie-aware against fp64 on the operands the tensor cores see"""
    from rangeclip_b200 import ops
    g = torch.Generator().manual_seed(D * 3 + k)
    B, H, W, K = 3, 16, 16, 1024
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1)
    tb = t.to(torch.bfloat16).float()
    x = (tb[torch.randint(0, K, (B, H, W), generator=g)].permute(0, 3, 1, 2) + 0.3 * torch.randn(B, D, H, W, generator=g))
    x = x.to(torch.bfloat16).float()
    out = ops.eval_topk(x.to(dev()).to(torch.bfloat16), t.to(dev()), torch.arange(K, device=dev()), k, "bf16").cpu()
    logits = torch.einsum("bdn,cd->bcn", x.double().reshape(B, D, H * W), tb.double())
    ref_v = logits.topk(k, dim=1).values
    got = torch.gather(logits, 1, out.reshape(B, k, H * W))
    scale = logits.abs().amax(dim=1, keepdim=True)
    assert bool(((got - ref_v).abs() <= 1e-5 * scale).all())


# ---------------------------------------------------------------------------------------------------------------------
# public calls at D = 768
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shared", [False, True])
def test_compute_loss_device_builder_d768(monkeypatch, shared):
    """compute_loss / compute_loss_shared2x2 with contrast_builder="device" under the sync check, against the oracle"""
    monkeypatch.setattr(dev_builder, "_case", functools.partial(dev_builder._case, D=768))
    dev_builder.test_compute_loss_device_builder_matches_oracle_and_never_syncs(shared)


@pytest.mark.parametrize("shared", [False, True])
def test_compute_loss_device_builder_max_contrast_512_d768(monkeypatch, shared):
    """max_contrast = 512: the K-blocked rounds with the row count in device memory, against the oracle"""
    monkeypatch.setattr(dev_kb, "_case", functools.partial(dev_kb._case, D=768))
    dev_kb.test_compute_loss_device_builder_above_256_rows(shared)


@pytest.mark.parametrize("C,kd", [(400, 100), (700, 500)], ids=["K<=256", "K>256"])
def test_compute_loss_shared2x2_never_upsamples_d768(C, kd):
    """compute_loss_shared2x2 at D = 768, one launch and K blocks: equal to compute_loss on the upsampled embeddings (the same
    draw), with F.interpolate patched to raise and the peak memory below the upsampled tensor's size"""
    shared2x2_kb.test_compute_loss_shared2x2_above_256_contrast_rows(768, C, kd, 64)


@pytest.mark.parametrize("n", [64, 1024])
def test_image_contrastive_loss_d768(n):
    """the area-image loss at n = 64 (fp32 kernel, 1e-5) and n = 1024 (tensor cores in K blocks, 2e-3 / 2e-2)"""
    from rangeclip_b200 import losses
    D = 768
    g = torch.Generator().manual_seed(n)
    area = torch.randn(n, D, generator=g)
    img = torch.randn(n, D, generator=g)
    if n >= 512:                                          # the tensor cores see bf16 operands
        area = area.to(torch.bfloat16).float()
        img = torch.nn.functional.normalize(img, dim=1).to(torch.bfloat16).float()
    log_tau = torch.tensor(math.log(0.1), device=dev(), requires_grad=True)
    ad = area.to(dev()).requires_grad_(True)
    loss = losses.image_contrastive_loss(ad, img.to(dev()), log_tau)
    loss.backward()
    torch.cuda.synchronize()
    ref = O.infonce_dense(area, torch.nn.functional.normalize(img, dim=1), torch.arange(n), torch.ones(n), 10.0)
    tol_l, tol_g = (1e-5, 1e-5) if n < 512 else (2e-3, 2e-2)
    assert abs(float(loss) - float(ref["loss"])) <= tol_l * abs(float(ref["loss"]))
    assert maxrel(ad.grad, ref["dx"]) < tol_g
    assert abs(float(log_tau.grad) - float(ref["dlogtau"])) <= max(tol_g, 1e-4) * abs(float(ref["dlogtau"]))


@pytest.mark.parametrize("builder", ["reference", "device"])
def test_predict_and_accumulate_shared2x2_d768(builder):
    """predict_and_accumulate(..., shared2x2=True): ids and histograms equal those of the upsampled embeddings"""
    import random as pyrandom
    from rangeclip_b200 import MetricAccumulator, evaluation
    B, D, h, w, C = 2, 768, 12, 16, 400
    g = torch.Generator().manual_seed(9)
    text = torch.randn(C, D, generator=g)
    seg = torch.randint(0, 60, (B, 2 * h, 2 * w), generator=g)
    x = (torch.nn.functional.normalize(text, dim=1)[seg[:, ::2, ::2]].permute(0, 3, 1, 2)
         + 0.3 * torch.randn(B, D, h, w, generator=g)).to(torch.bfloat16)
    xd, td, sd = x.to(dev()), text.to(dev()), seg.to(dev())
    E = torch.eye(C, dtype=torch.uint8)
    cmap = torch.arange(C)
    acc_a, acc_b = MetricAccumulator(E, cmap, device=dev()), MetricAccumulator(E, cmap, device=dev())
    pyrandom.seed(3)
    ids_a, _ = evaluation.predict_and_accumulate(xd, td, sd, acc_a, 100, 5, candidate_builder=builder, shared2x2=True)
    x_up = torch.nn.functional.interpolate(xd.float(), scale_factor=2, mode="nearest").to(torch.bfloat16)
    pyrandom.seed(3)
    ids_b, _ = evaluation.predict_and_accumulate(x_up, td, sd, acc_b, 100, 5, candidate_builder=builder)
    torch.cuda.synchronize()
    assert torch.equal(ids_a, ids_b)
    assert torch.equal(acc_a.acc, acc_b.acc) and torch.equal(acc_a.counters, acc_b.counters)


# ---------------------------------------------------------------------------------------------------------------------
# more than 2^31 elements in X
# ---------------------------------------------------------------------------------------------------------------------
def test_more_than_2_31_elements():
    """B = 33, D = 1024, 256 x 256 in bf16 (2.2e9 elements, 4.4 GB), fwd+bwd: sampled rows, the last image's last rows
    included, against fp64; rows of weight 0 get exactly zero dX"""
    from rangeclip_b200 import ops
    B, D, HW, K, tau = 33, 1024, 256 * 256, 64, 0.07
    assert B * D * HW > 2 ** 31
    g = torch.Generator(device=dev()).manual_seed(1)
    x = torch.randn(B, D, HW, device=dev(), dtype=torch.bfloat16, generator=g)
    t = torch.nn.functional.normalize(torch.randn(K, D, device=dev(), generator=g), dim=1).to(torch.bfloat16).float()
    y = torch.randint(-1, K, (B * HW,), device=dev(), dtype=torch.int32, generator=g)
    w = torch.randint(0, 3, (B * HW,), device=dev(), generator=g).float()
    r = ops.infonce_raw(x, t, y, w, 1 / tau, True, False, "bf16")
    torch.cuda.synchronize()
    lse, dx = r["lse"], r["dx"]
    W_tot = float((w * (y >= 0)).double().sum())
    last = torch.arange(B * HW - 300, B * HW, device=dev())
    sample = torch.cat([torch.randint(0, B * HW, (3000,), device=dev(), generator=g), last,
                        torch.arange(HW - 100, HW + 100, device=dev()),
                        (2 ** 31 // (D * HW)) * HW + torch.arange(-100, 100, device=dev())])      # the image that starts at 2^31
    b, p = sample // HW, sample % HW
    xs = x[b, :, p].double()                                                 # [n, D]
    xh = xs / xs.norm(dim=1, keepdim=True).clamp_min(1e-12)
    z = xh @ t.double().T / tau
    lse_ref = torch.logsumexp(z, dim=1)
    ys, ws = y[sample].long(), (w[sample] * (y[sample] >= 0)).double()
    P = torch.softmax(z, dim=1)
    P[torch.arange(len(sample)), ys.clamp_min(0)] -= (ys >= 0).double()
    dz = P * (ws / W_tot)[:, None] / tau
    dxh = dz @ t.double()
    dx_ref = (dxh - xh * (xh * dxh).sum(1, keepdim=True)) / xs.norm(dim=1, keepdim=True)
    assert bool(((lse[sample].double() - lse_ref).abs() <= 2e-3 * lse_ref.abs().clamp_min(1.0)).all())
    got = dx[b, :, p].double()
    live = ws > 0
    err = (got - dx_ref).norm(dim=1)[live] / dx_ref.norm(dim=1)[live]
    assert float(err.max()) < 2e-2, float(err.max())
    assert bool((got[~live] == 0).all())
    assert int((~live).sum()) > 100
