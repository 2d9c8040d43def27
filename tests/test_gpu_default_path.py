"""GPU tests of what round 1 left unpinned (VERDICT r1, "Next round" item 1):
  * the DEFAULT path of compute_loss -- tensor cores, fused text + smoothness backward, bf16 gradient widened in one
    pass -- against fixtures produced by the unmodified reference at D = 256 / 512, plain and inside torch.autocast;
  * one-image parity at BASELINE widths (HW = 65 536, D = 512, K = 256; K = 1024 evaluation; 64 masks at 256x256);
  * a second backward through the same graph (ADVICE r1: the saved gradient must stay intact);
  * the kernels as registered PyTorch custom operators (torch.ops.rangeclip.*: opcheck, fake tensors, torch.compile);
  * sharded validation through the drop-in: two processes on one GPU (gloo), every rank equals the single-process run.
Tolerances: 2e-2 max-relative on gradients and 2e-3 on losses for the bf16 tensor-core path (BASELINE.json north_star),
integer metrics bit-exact."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import rangeclip_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BF16_MAXREL = 2e-2
BF16_LOSS_RTOL = 2e-3


def dev():
    return torch.device("cuda:0")


def maxrel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


class _Model(torch.nn.Module):
    def __init__(self, tau_text=0.07, tau_image=0.1):
        super().__init__()
        self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(tau_text)))
        self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(tau_image)))


def _sets(g):
    C = g["text"].shape[0]
    hard = {i: [int(v) for v in g["hard"][i]] for i in range(C)}
    med = {i: [int(v) for v in g["medium"][i]] for i in range(C)}
    return {"medium": med, "hard": hard}


def _run_compute_loss(g, X, model, precision="auto", autocast=False, **kw):
    import rangeclip_b200 as R
    from unittest import mock
    area = torch.tensor(g["area"]).to(dev()) if g["area"].size else None
    img = torch.tensor(g["img"]).to(dev()) if g["img"].size else None
    rand_idx = torch.tensor(g["rand_idx"]).to(dev())
    seed = int(g["seed"])
    np.random.seed(seed); torch.manual_seed(seed); random.seed(seed)
    with mock.patch("torch.randint", lambda *a, **k: rand_idx), torch.autocast("cuda", enabled=autocast):
        return R.compute_loss(model, X, torch.tensor(g["seg"]).to(dev()), torch.tensor(g["text"]).to(dev()), _sets(g), area, img,
                              W_image=float(g["W_image"]), W_smooth=float(g["W_smooth"]),
                              percent_image_sampling=float(g["pct_sampling"]), k_distractors=int(g["k_distractors"]),
                              pct_medium=float(g["pcts"][0]), pct_hard=float(g["pcts"][1]), pct_rand=float(g["pcts"][2]),
                              precision=precision, **kw)


@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("xdtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", ["d256", "d512"])
def test_compute_loss_default_path_vs_reference(golden_dir, case, xdtype, autocast):
    """compute_loss(precision="auto") takes the tcgen05 kernel and the fused text + smoothness backward at D = 256 / 512;
    the fixtures are the reference's own totals / dX / dlogtau on bf16-exact inputs (tests/golden/make_golden.py).
    The reference trainer always calls it inside autocast (train_util.py:299): both contexts are covered."""
    g = np.load(os.path.join(golden_dir, f"loss_{case}.npz"))
    model = _Model().to(dev())
    X = torch.tensor(g["X"]).to(dev()).to(xdtype).requires_grad_(True)
    total, info = _run_compute_loss(g, X, model, "auto", autocast)
    total.backward()
    assert X.grad.dtype == xdtype
    assert abs(float(total) - float(g["total"])) <= BF16_LOSS_RTOL * abs(float(g["total"]))
    assert abs(info["text_contrastive_loss"] - float(g["text_loss"])) <= BF16_LOSS_RTOL * abs(float(g["text_loss"]))
    assert abs(info["image_contrastive_loss"] - float(g["image_loss"])) <= BF16_LOSS_RTOL * abs(float(g["image_loss"]))
    assert abs(info["smoothness_loss"] - float(g["smooth_loss"])) <= BF16_LOSS_RTOL * abs(float(g["smooth_loss"]))
    assert maxrel(X.grad.float().cpu(), g["dX"]) < BF16_MAXREL
    assert abs(float(model.log_temperature_text.grad) - float(g["dlogtau_text"])) <= BF16_MAXREL * abs(float(g["dlogtau_text"]))
    assert abs(float(model.log_temperature_image.grad) - float(g["dlogtau_image"])) <= BF16_MAXREL * abs(float(g["dlogtau_image"]))


@pytest.mark.parametrize("fused", [True, False])
def test_second_backward_sees_the_same_gradient(golden_dir, fused):
    """retain_graph / autograd.grad followed by backward: the saved dX is read-only, every backward returns
    upstream * dX again (ADVICE r1: the in-place late scaling returned dx*g^2 on the second pass)."""
    g = np.load(os.path.join(golden_dir, "loss_d256.npz"))
    model = _Model().to(dev())
    X = torch.tensor(g["X"]).to(dev()).to(torch.bfloat16).requires_grad_(True)
    total, _ = _run_compute_loss(g, X, model, "auto", False) if fused else (None, None)
    if not fused:       # text term alone: the rangeclip::infonce node
        import rangeclip_b200 as R
        from unittest import mock
        rand_idx = torch.tensor(g["rand_idx"]).to(dev())
        np.random.seed(1); torch.manual_seed(1)
        with mock.patch("torch.randint", lambda *a, **k: rand_idx):
            total = R.text_contrastive_loss(X, torch.tensor(g["seg"]).to(dev()), torch.tensor(g["text"]).to(dev()), _sets(g),
                                            model.log_temperature_text, k_distractors=int(g["k_distractors"]))
    (g1,) = torch.autograd.grad(total * 0.5, X, retain_graph=True)
    (g2,) = torch.autograd.grad(total * 0.5, X, retain_graph=True)
    assert torch.equal(g1, g2)
    total.backward()
    assert maxrel(X.grad.float().cpu(), 2.0 * g1.float().cpu()) < 1e-2        # bf16 rounding of the scaled copies only
    assert float(X.grad.float().abs().max()) > 0


def test_pair_kernels_one_image_full_width_vs_oracle():
    """HW = 65 536, D = 512, K = 256 (one image of BASELINE configs[1]) against the fp64 oracle: loss, lse, dX, dlogtau
    from the TS-mode kernel, the same from the shared-memory-operand kernel, and dText from the tensor-core dText path."""
    from rangeclip_b200 import ops
    D, HW, K, tau = 512, 65536, 256, 0.07
    g = torch.Generator().manual_seed(4242)
    x = torch.nn.functional.normalize(torch.randn(1, D, HW, generator=g), dim=1).to(torch.bfloat16)
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1)
    y = torch.randint(0, K, (HW,), generator=g, dtype=torch.int32)
    w = torch.randint(0, 3, (HW,), generator=g).float()
    y[torch.rand(HW, generator=g) < 0.1] = -1
    tb = t.to(torch.bfloat16).float()                  # what the tensor cores see
    rows = x[0].float().t().contiguous()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = O.infonce_dense(rows, tb, y.long(), w, 1.0 / tau)
    dx_ref = ref["dx"].t().float()
    xd = x.view(1, D, 256, 256).to(dev())
    for flags, want_dt in ((0, False), (8, False), (0, True)):
        r = ops.infonce_raw(xd, tb.to(dev()), y.to(dev()), w.to(dev()), 1.0 / tau, True, want_dt, "bf16", flags=flags)
        loss = float(r["loss_sum"] / r["w_sum"])
        assert abs(loss - float(ref["loss"])) <= BF16_LOSS_RTOL * abs(float(ref["loss"])), (flags, want_dt)
        valid = (w > 0) & (y >= 0)
        assert float((r["lse"].cpu()[valid] - ref["lse"].float()[valid]).abs().max()) < 2e-3 * float(ref["lse"].abs().max())
        assert maxrel(r["dx"].float().cpu().view(D, HW), dx_ref) < BF16_MAXREL, (flags, want_dt)
        assert abs(float(r["dlogtau"]) - float(ref["dlogtau"])) <= BF16_MAXREL * abs(float(ref["dlogtau"]))
        if want_dt:
            assert maxrel(r["dt"].cpu(), ref["dt"].float()) < BF16_MAXREL


def test_fused_top5_histograms_one_map_k1024_vs_oracle():
    """One 256x256 map against a K = 1024 vocabulary (BASELINE configs[4]): the fused tcgen05 top-5 + histogram kernel
    against the oracle's metric accumulation fed the kernel's own ids (bit-exact), and the ids against the oracle's fp64
    logits tie-aware (every disagreement is a gap below the bf16 resolution of a cosine)."""
    from rangeclip_b200 import ops
    C, D, H, W, k = 1024, 512, 256, 256, 5
    g = torch.Generator().manual_seed(77)
    eq = {i: {i} for i in range(C)}
    pairs = torch.randperm(C, generator=g)[:102].tolist()
    for a, b in zip(pairs[:-1], pairs[1:]):            # a non-transitive synonym chain over 10 % of the ids (Q9)
        eq[a].add(b); eq[b].add(a)
    E = O.build_equivalence_tensor(eq, C); cmap = O.build_equivalence_class_map(E)
    text = torch.nn.functional.normalize(torch.randn(C, D, generator=g), dim=1)
    seg = torch.randint(0, C, (1, H // 16, W // 16), generator=g).repeat_interleave(16, 1).repeat_interleave(16, 2).contiguous()
    x = torch.nn.functional.normalize(text[seg].permute(0, 3, 1, 2) + 0.3 * torch.randn(1, D, H, W, generator=g), dim=1).to(torch.bfloat16)
    hist = torch.zeros(5, C, device=dev(), dtype=torch.int64); cnt = torch.zeros(3, device=dev(), dtype=torch.int64)
    idx = torch.arange(C, device=dev())
    ids = ops.eval_topk_hist(x.to(dev()), text.to(dev()), idx, k, seg.to(dev()), torch.tensor(E).to(dev()).to(torch.uint8),
                             torch.tensor(cmap).to(dev()), hist, cnt).cpu()
    st = O.MetricState()
    O.metrics_accumulate(st, seg.numpy().reshape(-1), ids.permute(0, 2, 3, 1).reshape(-1, k).numpy(), E, cmap)
    fin_o = O.metrics_finalize(st, seg.numpy().reshape(-1), cmap)
    from rangeclip_b200 import MetricAccumulator
    acc = MetricAccumulator(torch.tensor(E), torch.tensor(cmap), device=dev())
    acc.update(seg.to(dev()), ids.to(dev()))
    fin = acc.finalize(seg.to(dev()))
    assert int(cnt[2]) == H * W and fin["total_pixels"] == H * W
    assert [int(v) for v in cnt.tolist()] == [st.correct_top1, st.correct_topk, st.total]
    for name in ("mIoU_t1", "mIoU_tk", "pixel_accuracy_t1", "pixel_accuracy_tk"):
        assert fin[name] == fin_o[name], name
    assert 0.1 < fin["pixel_accuracy_t1"] < 0.95          # the hit and the miss branches are both exercised
    # tie-aware id check on a strided sample of pixels (fp64 logits on bf16-rounded operands)
    sel = torch.arange(0, H * W, 97)
    xr = x[0].float().view(D, -1)[:, sel].t().double()
    logits = torch.nn.functional.normalize(xr, dim=1) @ text.to(torch.bfloat16).double().t()
    got = ids[0].view(k, -1)[:, sel].t()
    top = logits.topk(k, dim=1)
    for r_ in range(sel.numel()):
        for j in range(k):
            if int(got[r_, j]) != int(top.indices[r_, j]):
                assert abs(float(logits[r_, got[r_, j]]) - float(top.values[r_, j])) < 4e-3, (r_, j)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pooling_64_masks_256x256_vs_oracle(dtype):
    """BASELINE configs[3] per image: 64 object masks (the 32x32 blocks) of one 256x256 map, D = 512."""
    import rangeclip_b200 as R
    D, H, W = 512, 256, 256
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, D, H, W, generator=g).to(dtype)
    seg = (torch.arange(64).view(8, 8) + 1).repeat_interleave(32, 0).repeat_interleave(32, 1)[None].contiguous()
    labels = list(range(1, 65))
    ref = O.area_pool_per_image(x.float(), seg, [0] * 64, labels)
    out = R.pool_objects_per_image(x.to(dev()), seg.to(dev()), [0] * 64, labels)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert maxrel(out.float().cpu(), ref) < tol
    xg = x.to(dev()).requires_grad_(True)
    up = torch.randn(64, D, generator=g)
    (R.pool_objects_per_image(xg, seg.to(dev()), [0] * 64, labels, differentiable=True).float() * up.to(dev())).sum().backward()
    gref = (up / 1024.0)[seg[0].reshape(-1) - 1].t().reshape(1, D, H, W)          # every mask has 32*32 pixels
    assert maxrel(xg.grad.float().cpu(), gref) < (1e-6 if dtype == torch.float32 else 1e-2)


def test_shared2x2_falls_back_when_the_four_target_kernel_does_not_apply():
    """ADVICE r1: more than 256 contrast rows (their number is data dependent) or D outside (256, 512) must not abort the
    training step: compute_loss_shared2x2 then takes the loss of the upsampled tensor through the ordinary path."""
    import rangeclip_b200 as R
    from unittest import mock
    for D, C, kd, H in ((64, 40, 12, 16), (256, 400, 300, 32)):
        g = torch.Generator().manual_seed(D + C)
        e = torch.randn(2, D, H // 2, H // 2, generator=g).to(dev())
        seg = torch.randint(0, 9, (2, H // 4, H // 4), generator=g).repeat_interleave(4, 1).repeat_interleave(4, 2).to(dev())
        text = torch.randn(C, D, generator=g).to(dev())
        sets = {"medium": {}, "hard": {}}
        rand_idx = torch.randint(0, H * H, (2, int(0.7 * H * H)), generator=g).to(dev())
        res = []
        for shared in (True, False):
            model = _Model().to(dev())
            x = e.clone().requires_grad_(True)
            np.random.seed(3); torch.manual_seed(3)
            with mock.patch("torch.randint", lambda *a, **k: rand_idx):
                if shared:
                    total, info = R.compute_loss_shared2x2(model, x, seg, text, sets, None, None, W_image=0.0, W_smooth=0.0, k_distractors=kd,
                                                           pct_medium=0.0, pct_hard=0.0, pct_rand=1.0)
                else:
                    up = torch.nn.functional.normalize(torch.nn.functional.interpolate(x, scale_factor=2, mode="nearest"), dim=1)
                    total, info = R.compute_loss(model, up, seg, text, sets, None, None, W_image=0.0, W_smooth=0.0, k_distractors=kd,
                                                 pct_medium=0.0, pct_hard=0.0, pct_rand=1.0)
            total.backward()
            res.append((float(total), x.grad.float().cpu()))
        assert abs(res[0][0] - res[1][0]) <= 2e-3 * abs(res[1][0])
        assert maxrel(res[0][1], res[1][1]) < BF16_MAXREL


def test_text_prepare_out_of_range_index_yields_nan_rows():
    """ADVICE r1: the reference raises at candidate_text_embeddings[index_tensor]; the kernel marks the row instead of
    reading out of bounds."""
    from rangeclip_b200 import ops
    text = torch.randn(10, 64, device=dev())
    t32, tb, ttb = ops.text_prepare(text, torch.tensor([0, 3, 10, -2, 9, -1], device=dev()), want_f32=True, want_bf16=True)
    assert torch.isnan(t32[2]).all() and torch.isnan(t32[3]).all()
    assert torch.isfinite(t32[[0, 1, 4]]).all() and torch.isnan(tb[2].float()).all()
    assert float(t32[5].abs().sum()) == 0.0 and float(tb[5].float().abs().sum()) == 0.0      # -1 = pad entry of rc_contrast_build: a zero row
    assert torch.allclose(t32[1], torch.nn.functional.normalize(text[3], dim=0), atol=1e-6)


# ------------------------------------------------------------------------------------------------
# the kernels as PyTorch custom operators
# ------------------------------------------------------------------------------------------------

def _small_infonce_args(D=256, HW=64, K=40, requires_grad=True):
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, D, 8, HW // 8, generator=g).to(torch.bfloat16).to(dev()).requires_grad_(requires_grad)
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1).to(dev())
    y = torch.randint(0, K, (2 * HW,), generator=g, dtype=torch.int32).to(dev())
    w = torch.ones(2 * HW, device=dev())
    log_tau = torch.log(torch.tensor(0.07, device=dev())).requires_grad_(requires_grad)
    return x, t, log_tau, y, w


def test_custom_ops_are_registered_and_pass_opcheck():
    import rangeclip_b200  # noqa: F401  (registers torch.ops.rangeclip.*)
    for name in ("infonce", "pixel_losses", "smoothness", "tv_bwd", "scale_to", "scale_", "masked_pool", "masked_pool_bwd",
                 "sample_weights", "text_prepare", "eval_topk", "eval_hist", "eval_topk_hist", "eval_fold"):
        assert hasattr(torch.ops.rangeclip, name), name
    x, t, log_tau, y, w = _small_infonce_args()
    tests = ("test_schema", "test_faketensor", "test_autograd_registration")
    torch.library.opcheck(torch.ops.rangeclip.infonce.default, (x, t, log_tau, y, w, True, False, "auto", 1, None, None), test_utils=tests)
    torch.library.opcheck(torch.ops.rangeclip.infonce.default, (x, t, log_tau, y, w, True, False, "kblocked", 1, None, None),
                          test_utils=tests)
    torch.library.opcheck(torch.ops.rangeclip.smoothness.default, (x, 10.0, 12.0), test_utils=tests)
    torch.library.opcheck(torch.ops.rangeclip.scale_to.default, (x.detach(), torch.tensor(0.5, device=dev()), 0), test_utils=tests)
    seg = torch.randint(0, 5, (2, 8, 8), device=dev())
    lut = torch.tensor([-1, 0, 1, 2, 3], dtype=torch.int32, device=dev())
    torch.library.opcheck(torch.ops.rangeclip.masked_pool.default, (x, [seg], lut, False, 4), test_utils=tests)


def test_torch_compile_does_not_break_inside_the_loss_ops():
    """torch.compile(fullgraph=True): Dynamo + AOTAutograd trace through the registered operators (fake tensors, autograd
    formulas) without a graph break; backend aot_eager keeps Triton / inductor out of it."""
    from rangeclip_b200 import ops
    x, t, log_tau, y, w = _small_infonce_args()

    def f(x, t, log_tau, y, w):
        text, smooth = ops.pixel_losses(x, t, log_tau, y, w)
        return text + 200.0 * smooth

    eager = f(x, t, log_tau, y, w)
    (gx_e, gl_e) = torch.autograd.grad(eager, (x, log_tau))
    cf = torch.compile(f, backend="aot_eager", fullgraph=True)
    out = cf(x, t, log_tau, y, w)
    (gx_c, gl_c) = torch.autograd.grad(out, (x, log_tau))
    assert torch.allclose(out, eager) and torch.equal(gx_c, gx_e) and torch.allclose(gl_c, gl_e)


# ------------------------------------------------------------------------------------------------
# sharded validation through the drop-in (two processes, one GPU, gloo)
# ------------------------------------------------------------------------------------------------

_WORKER = r"""
import json, os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
import rangeclip_b200 as R
from rangeclip_b200.distributed import shard_batches
g = np.load({fixture!r})
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
if world > 1:
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"], rank=rank, world_size=world)
dev = torch.device("cuda:0")
E, cmap = torch.tensor(g["E"]), torch.tensor(g["cmap"])
gen = torch.Generator().manual_seed(123)
segs = [torch.tensor(s) for s in g["seg"]] + [torch.tensor(g["seg"][0]).flip(1), torch.tensor(g["seg"][1]).flip(2)]
topks = [torch.tensor(t) for t in g["topk"]] + [torch.tensor(g["topk"][1]), torch.tensor(g["topk"][0])]
order = [0, 3, 1, 4, 2]                     # five batches; the reference's last-batch label filter bites on batch 2
batches = [dict(depth=torch.zeros(2, 1, 16, 16), image=torch.zeros(2, 3, 16, 16), segmentation=segs[i],
                object_bbox=torch.zeros(2, 4, dtype=torch.long), object_label="x", _topk=topks[i]) for i in order]
mine = [batches[i] for i in shard_batches(len(batches), rank, world)]

class FakeModel:
    def __init__(self): self.i = 0
    def eval(self): return self
    def predict(self, depth_maps, candidate_text_embeddings, segmentation, num_negatives, top_k):
        t = mine[self.i]["_topk"].to(dev); self.i += 1
        return t, torch.zeros(2, 4, 16, 16, device=dev), torch.tensor(0.07)
    def compute_loss(self, **kw): return torch.tensor(0.0), {{"total_loss": 1.0 + rank}}

best = R.validate_model(FakeModel(), None, None, None, [str(i) for i in range(int(g["C"]))], E, cmap, None,
                        dict(pct_medium=0.0, pct_hard=0.5, pct_rand=0.5), mine, 0, {{"step": -1, "loss": float("inf")}}, dev,
                        all_reduce=world > 1)
out = {{k: best[k] for k in ("mIoU_t1", "mIoU_tk", "pixel_accuracy_t1", "pixel_accuracy_tk", "loss")}}
json.dump(out, open({out!r} + str(rank) + "_" + str(world) + ".json", "w"))
if world > 1:
    dist.destroy_process_group()
"""


def test_validate_model_two_ranks_equal_one_rank(golden_dir, tmp_path):
    """validate_model(all_reduce=True) on two ranks (gloo, both on cuda:0, real kernels) returns on EVERY rank the four
    floats of the single-process run over the same five batches -- global batch indices for the first-seen order and the
    globally last batch's class filter (VERDICT r1 weak #5 / ADVICE r1)."""
    fixture = os.path.join(golden_dir, "metrics.npz")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT, fixture=fixture, out=str(tmp_path / "res_")))
    env = dict(os.environ, PORT=str(29600 + os.getpid() % 300))
    subprocess.run([sys.executable, str(script)], env=dict(env, RANK="0", WORLD_SIZE="1"), check=True, timeout=300)
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), WORLD_SIZE="2")) for r in range(2)]
    for p in procs:
        assert p.wait(timeout=300) == 0
    one = json.load(open(str(tmp_path / "res_") + "0_1.json"))
    for r in range(2):
        two = json.load(open(str(tmp_path / "res_") + f"{r}_2.json"))
        for key in ("mIoU_t1", "mIoU_tk", "pixel_accuracy_t1", "pixel_accuracy_tk"):
            assert two[key] == one[key], (r, key, two[key], one[key])
    assert one["mIoU_tk"] > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_normalize_rows_matches_f_normalize(dtype):
    """rangeclip::normalize_rows (the decoder tail's F.normalize, decoder.py:114, one kernel each way) against PyTorch."""
    from rangeclip_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(2, 96, 8, 12, generator=g) * (0.2 + torch.rand(2, 1, 8, 12, generator=g))).to(dtype)
    x[0, :, 0, 0] = 0                                   # a zero row: eps path (F.normalize clamps the norm at 1e-12)
    up = torch.randn(2, 96, 8, 12, generator=g)
    xr = x.float().clone().requires_grad_(True)
    ref = torch.nn.functional.normalize(xr, p=2, dim=1)
    (ref * up).sum().backward()
    xd = x.detach().clone().to(dev()).requires_grad_(True)
    out = ops.normalize_rows(xd)
    assert out.dtype == torch.float32
    (out * up.to(dev())).sum().backward()
    assert xd.grad.dtype == dtype
    assert maxrel(out.detach().cpu(), ref.detach()) < 1e-6
    assert maxrel(xd.grad.float().cpu(), xr.grad) < (1e-5 if dtype == torch.float32 else 1e-2)
