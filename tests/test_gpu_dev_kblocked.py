"""The sync-free K-blocked InfoNCE: the device contrast builder above 256 rows.  The K-blocked rounds are shaped for the
contrast set's capacity (up to 1024 rows, four launches of 256) and every launch (rc_infonce_bf16_dyn_kblock) reads from
device memory how many of its rows are valid, and log(tau).  Checked here: the rounds against the host-parameter rounds on
the same rows and against the fp64 row bounds of oracle/infonce_rows.py; empty blocks change nothing; TS and SS agree bit
for bit; the public loss with contrast_builder="device" above 256 rows matches the oracle, never synchronises and is
captured in a CUDA graph; opcheck of the operator form."""
import math

import numpy as np
import pytest
import torch

from oracle import infonce_rows as OR
from oracle import rangeclip_oracle as O

pytestmark = pytest.mark.gpu

BF16_MAXREL = 2e-2        # the project's bf16 gates (BASELINE.json): max-relative on gradients, relative on the loss
BF16_LOSS_RTOL = 2e-3
TS, SS = 0, 32


def dev():
    return torch.device("cuda:0")


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _kinfo(K):
    return torch.tensor([K, 0, 0, 0], dtype=torch.int32, device=dev())


def _padded(t, cap):
    """t [K, D] -> [cap, D] with zero pad rows (what rc_text_prepare gives the builder's -1 entries)"""
    tp = torch.zeros(cap, t.shape[1], device=dev())
    tp[:t.shape[0]] = t.to(dev())
    return tp


def _dev_rounds(x, t, y, w, cap, log_tau):
    """the sync-free K-blocked rounds on the first K = t.shape[0] rows of a set of capacity `cap`"""
    from rangeclip_b200 import ops
    rep = 4 if y.dim() == 2 else 1
    r = ops.infonce_raw(x, _padded(t, cap), y, w, 0.0, True, False, "bf16", rep=rep, k_dev=_kinfo(t.shape[0]),
                        log_tau_dev=torch.tensor([log_tau], dtype=torch.float32, device=dev()), dev_blocks=True)
    torch.cuda.synchronize()
    return r


def _host_rounds(x, t, y, w, inv_tau):
    from rangeclip_b200 import ops
    rep = 4 if y.dim() == 2 else 1
    r = ops.infonce_raw(x, t.to(dev()), y, w, inv_tau, True, False, "auto", rep=rep)
    assert r["precision"] == "bf16-kblocked"
    torch.cuda.synchronize()
    return r


def _dev_inv_tau(log_tau):
    """the kernels' inv_tau = expf(-log tau) of the fp32 log tau"""
    return math.exp(-float(torch.tensor(log_tau, dtype=torch.float32)))


def _assert_close(a, b):
    """device expf against the host exponent: the only difference between the two forms"""
    assert abs(float(a["loss_sum"]) - float(b["loss_sum"])) <= 1e-5 * abs(float(b["loss_sum"]))
    assert maxrel(a["lse"], b["lse"]) < 1e-5
    assert abs(float(a["dlogtau"]) - float(b["dlogtau"])) <= 1e-4 * abs(float(b["dlogtau"]))
    assert maxrel(a["dx"].float(), b["dx"].float()) < 1e-2
    assert float(a["w_sum"]) == float(b["w_sum"])


def _assert_identical(a, b):
    for k in ("loss_sum", "w_sum", "dlogtau"):
        assert float(a[k]) == float(b[k]), k
    assert torch.equal(a["lse"].view(torch.int32), b["lse"].view(torch.int32))
    assert torch.equal(a["dx"].view(torch.int16), b["dx"].view(torch.int16))


def _rows(a, B, D, HW):
    return a.detach().reshape(B, D, HW).permute(0, 2, 1).reshape(B * HW, D).double().cpu()


def _check_rows(name, err, bound):
    err, bound = err.double(), bound.double()
    assert bool(torch.isfinite(err).all()), f"{name}: non-finite rows"
    ratio = err / bound
    bad = torch.nonzero(ratio > 1).flatten()
    assert bad.numel() == 0, f"{name}: {bad.numel()} rows out of bound, worst ratio {float(ratio.max()):.3g}"
    return float(ratio.max())


def _check_row_bounds(tag, r, ref, B, D, HW, K):
    """every row's lse and dX, the loss sum and dlogtau inside the fp64 bounds of the K-blocked rounds (dX accumulated in
    the kernel, one bf16 store per block)"""
    nb = (K + 255) // 256
    lse = r["lse"].double().cpu()
    wl = _check_rows(f"{tag} lse", (lse - ref["lse"]).abs(), OR.lse_bound(ref, D, 256, nb))
    sp = OR.store_points_kblocked(ref, True)
    dx = _rows(r["dx"].float(), B, D, HW)
    wd = _check_rows(f"{tag} dx", (dx - ref["dx"]).norm(dim=1), OR.dx_bound(ref, D, 256, store_points=sp, lse_given=True, nb=nb))
    loss_b, dlt_b = OR.sums_bounds(ref, D, 256, 64 * nb, nb, True)
    assert abs(float(r["loss_sum"]) - float(ref["loss_sum"])) <= loss_b
    assert abs(float(r["dlogtau"]) - float(ref["dlogtau"])) <= dlt_b
    print(f"\n[rows] {tag}: worst error / bound lse {wl:.3f}, dx {wd:.3f}")


@pytest.mark.parametrize("K", [257, 300, 512, 700, 1024])
@pytest.mark.parametrize("D", [256, 512])
@pytest.mark.parametrize("rep", [1, 4])
def test_dev_rounds_equal_the_host_parameter_rounds(rep, D, K):
    """capacity = K: the same blocks as the host-parameter rounds, K and log tau from device memory"""
    B, HW = 2, 136
    x, t, y, w = OR.make_case(B, D, HW, K, rep, seed=rep * 7 + D + K)
    xd, yd, wd = x.to(dev()).to(torch.bfloat16), y.to(dev()), w.to(dev())
    log_tau = math.log(0.07)
    a = _dev_rounds(xd, t, yd, wd, K, log_tau)
    assert a["precision"] == "bf16-kblocked"
    b = _host_rounds(xd, t, yd, wd, _dev_inv_tau(log_tau))
    _assert_close(a, b)


@pytest.mark.parametrize("tau", [0.07, 0.0291, 0.01])
@pytest.mark.parametrize("rep,D,K", [(1, 256, 300), (1, 512, 1024), (4, 256, 700), (4, 512, 512), (1, 256, 257)])
def test_dev_rounds_rows_inside_the_fp64_bound(rep, D, K, tau):
    B, HW = 2, 136
    x, t, y, w = OR.make_case(B, D, HW, K, rep, seed=rep * 11 + D + K)
    log_tau = math.log(tau)
    r = _dev_rounds(x.to(dev()).to(torch.bfloat16), t, y.to(dev()), w.to(dev()), K, log_tau)
    ref = OR.reference(_rows(x, B, D, HW), t, y, w, _dev_inv_tau(log_tau))
    _check_row_bounds(f"dev-kblocked R={rep} D={D} K={K} tau={tau}", r, ref, B, D, HW, K)


@pytest.mark.parametrize("rep", [1, 4])
def test_empty_blocks_are_inert(rep):
    """valid K = 300 at capacity 512 and 1024: the launches of blocks 2 and 3 return at once, nothing changes a bit; valid
    K = 100 at capacity 512 (block 1 empty) against the one-launch form at capacity 256"""
    from rangeclip_b200 import ops
    B, D, HW = 2, 256, 136
    x, t, y, w = OR.make_case(B, D, HW, 300, rep, seed=41 + rep)
    xd, yd, wd = x.to(dev()).to(torch.bfloat16), y.to(dev()), w.to(dev())
    log_tau = math.log(0.07)
    _assert_identical(_dev_rounds(xd, t, yd, wd, 512, log_tau), _dev_rounds(xd, t, yd, wd, 1024, log_tau))
    x, t, y, w = OR.make_case(B, D, HW, 100, rep, seed=43 + rep)
    xd, yd, wd = x.to(dev()).to(torch.bfloat16), y.to(dev()), w.to(dev())
    a = _dev_rounds(xd, t, yd, wd, 512, log_tau)
    b = ops.infonce_raw(xd, _padded(t, 256), yd, wd, 0.0, True, False, "bf16", rep=rep, k_dev=_kinfo(100),
                        log_tau_dev=torch.tensor([log_tau], dtype=torch.float32, device=dev()))
    assert b["precision"] == "bf16"
    torch.cuda.synchronize()
    _assert_close(a, b)


def _launch(L, x, tb, ttb, Kb, kd, k0, y_rel, w, lt, lse, dx, flags, rep):
    from rangeclip_b200 import _lib
    B, D, HW = x.shape
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, Kb, _lib.RC_BF16))
    ws = torch.empty(ws_bytes, device=dev(), dtype=torch.uint8)
    acc = torch.zeros(4, device=dev(), dtype=torch.float64)
    acc[3] = w.double().sum()
    _lib.check(L.rc_infonce_bf16_dyn_kblock(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), Kb, kd.data_ptr(),
                                            k0, y_rel.data_ptr(), w.data_ptr(), lt.data_ptr(), rep, lse.data_ptr(),
                                            acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr() if dx is not None else None,
                                            None, dx.data_ptr() if dx is not None else None,
                                            acc[2:].data_ptr() if dx is not None else None, ws.data_ptr(), ws_bytes, flags,
                                            torch.cuda.current_stream().cuda_stream), "rc_infonce_bf16_dyn_kblock")
    torch.cuda.synchronize()
    return dict(lse=lse, dx=dx, loss_sum=acc[0], w_sum=acc[1], dlogtau=acc[2])


@pytest.mark.parametrize("rep", [1, 4])
@pytest.mark.parametrize("k0", [0, 256])
def test_ts_equals_ss_in_the_backward_round(rep, k0):
    """one block of the backward round (lse given, dX added to an existing gradient), TS against SS: dX, lse and the sums
    bit for bit; an empty block (valid rows <= k0) leaves dX, lse and the sums untouched on both kernels"""
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    B, D, HW, K = 2, 512, 136, 300
    x, t, y, w = OR.make_case(B, D, HW, K, rep, seed=53 + rep + k0)
    xd = x.to(dev()).to(torch.bfloat16)
    yd, wd = y.to(dev()), w.to(dev())
    wd = (wd * (yd >= 0)).contiguous()
    Kb = 256
    tb, ttb = ops.text_to_bf16(_padded(t, 512)[k0:k0 + Kb])
    y_rel = (yd - k0).contiguous()
    lt = torch.tensor([math.log(0.05)], dtype=torch.float32, device=dev())
    M = B * HW
    base = torch.randn(xd.shape, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).to(dev())
    lse_in = torch.randn(M, generator=torch.Generator().manual_seed(4)).to(dev()) + 30.0
    fl = 1 | ops.RC_INFONCE_KEEP_WEIGHT | ops.RC_INFONCE_LSE_GIVEN | ops.RC_INFONCE_ACCUMULATE_DX
    r = [_launch(L, xd, tb, ttb, Kb, _kinfo(K), k0, y_rel, wd, lt, lse_in.clone(), base.clone(), fl | extra, rep)
         for extra in (TS, SS)]
    assert torch.equal(r[0]["dx"].view(torch.int16), r[1]["dx"].view(torch.int16))
    assert torch.equal(r[0]["lse"].view(torch.int32), r[1]["lse"].view(torch.int32))
    for k in ("loss_sum", "w_sum", "dlogtau"):
        assert float(r[0][k]) == float(r[1][k]), k
    assert not torch.equal(r[0]["dx"], base)
    # the forward round's lse, SS forward kernel (the round-1 form of a backward launch runs TS / SS: same bits)
    lse_f = [_launch(L, xd, tb, ttb, Kb, _kinfo(K), k0, y_rel, wd, lt, torch.empty(M, device=dev()), torch.empty_like(xd),
                     1 | ops.RC_INFONCE_KEEP_WEIGHT | extra, rep)["lse"] for extra in (TS, SS)]
    f = _launch(L, xd, tb, ttb, Kb, _kinfo(K), k0, y_rel, wd, lt, torch.empty(M, device=dev()), None,
                1 | ops.RC_INFONCE_KEEP_WEIGHT, rep)
    assert torch.equal(lse_f[0].view(torch.int32), lse_f[1].view(torch.int32))
    assert maxrel(f["lse"], lse_f[0]) < 1e-6
    # empty block: valid rows = 200 - 256 < 0 (k0 = 256) -- nothing is written or added, on both kernels
    if k0 > 0:
        for extra in (TS, SS):
            e = _launch(L, xd, tb, ttb, Kb, _kinfo(200), k0, y_rel, wd, lt, lse_in.clone(), base.clone(), fl | extra, rep)
            assert torch.equal(e["dx"].view(torch.int16), base.view(torch.int16))
            assert float(e["loss_sum"]) == 0.0 and float(e["w_sum"]) == 0.0 and float(e["dlogtau"]) == 0.0
        sentinel = torch.full((M,), 7.0, device=dev())
        e = _launch(L, xd, tb, ttb, Kb, _kinfo(200), k0, y_rel, wd, lt, sentinel, None, 1 | ops.RC_INFONCE_KEEP_WEIGHT, rep)
        assert bool((e["lse"] == 7.0).all()) and float(e["loss_sum"]) == 0.0


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(0.07)))
        self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(0.1)))


def _case(B=2, D=256, H=32, W=32, C=600, n_labels=130, seed=3):
    """about 120 present labels among C = 600 (labels 0..n_labels-1 in the segmentation, 0 is background)"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, H, W, generator=g).to(torch.bfloat16).float()
    seg = torch.randint(0, n_labels, (B, H, W), generator=g)
    text = torch.randn(C, D, generator=g)
    rng = np.random.default_rng(seed)
    sets = {"hard": {c: [int(v) for v in rng.choice(C, 8, replace=False)] for c in range(C)},
            "medium": {c: [int(v) for v in rng.choice(C, 8, replace=False)] for c in range(C)}}
    return x, seg, text, sets


KW = dict(W_text=1.0, W_image=0.0, W_smooth=0.0, percent_image_sampling=0.7, k_distractors=250, pct_medium=0.2, pct_hard=0.5,
          pct_rand=0.3, contrast_builder="device")


@pytest.mark.parametrize("shared", [False, True])
def test_compute_loss_device_builder_above_256_rows(shared):
    """max_contrast=512: every distractor kept (flags 0, K > 256), no synchronisation, loss and gradients equal to the
    oracle's for the set drawn; the same inputs at max_contrast=256 still trim (flag 2)"""
    import rangeclip_b200 as R
    from rangeclip_b200 import losses
    x, seg, text, sets = _case()
    model = _Model().to(dev())
    if shared:
        seg = torch.nn.functional.interpolate(seg[:, None].float(), scale_factor=2, mode="nearest")[:, 0].long()
    xd = x.to(dev()).to(torch.bfloat16).requires_grad_(True)
    segd, textd = seg.to(dev()), text.to(dev())
    fn = R.compute_loss_shared2x2 if shared else R.compute_loss
    kw = dict(KW, max_contrast=512)
    torch.manual_seed(11)
    total, info = fn(model, xd, segd, textd, sets, None, None, **kw)        # warm-up: allocator, CSR cache, module loading
    total.backward()
    torch.cuda.synchronize()
    xd.grad = None; model.zero_grad()
    torch.manual_seed(11)
    torch.cuda.set_sync_debug_mode("error")
    try:
        total, info = fn(model, xd, segd, textd, sets, None, None, **kw)
        total.backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert isinstance(info, losses.LazyLossInfo)
    torch.manual_seed(11)
    _, aux = losses.text_contrastive_loss(xd.detach(), segd, textd, sets, model.log_temperature_text.detach(), 0.7, 250, 0.2, 0.5,
                                          0.3, "auto", return_aux=True, shared2x2=shared, contrast_builder="device",
                                          max_contrast=512)
    K, flags, n_present, n_dis = aux["contrast_info"].tolist()
    assert flags == 0 and K > 256 and n_dis == 250 and K == n_present + 250 and n_present > 100, (K, flags, n_present, n_dis)
    contrast = aux["contrast_indices"][:K].cpu()
    assert bool((aux["contrast_indices"][K:] == -1).all())
    xin = x if not shared else torch.nn.functional.interpolate(x, scale_factor=2, mode="nearest")
    Bq, D = xin.shape[0], xin.shape[1]
    w = O.sampling_weights(seg, aux["rand_indices"].cpu())
    lm = torch.full((text.shape[0],), -1, dtype=torch.long)
    lm[contrast] = torch.arange(K)
    yy = lm[seg.reshape(Bq, -1)]
    yy[seg.reshape(Bq, -1) == 0] = -1
    rows = xin.permute(0, 2, 3, 1).reshape(-1, D)
    ref = O.infonce_dense(rows, torch.nn.functional.normalize(text[contrast], dim=1), yy.reshape(-1), w.reshape(-1), 1 / 0.07)
    assert abs(float(total) - float(ref["loss"])) <= BF16_LOSS_RTOL * abs(float(ref["loss"]))
    assert abs(info["total_loss"] - float(ref["loss"])) <= BF16_LOSS_RTOL * abs(float(ref["loss"]))
    dx_ref = ref["dx"].reshape(Bq, xin.shape[2], xin.shape[3], D).permute(0, 3, 1, 2)
    if shared:
        dx_ref = dx_ref.reshape(Bq, D, x.shape[2], 2, x.shape[3], 2).sum(dim=(3, 5))
    assert maxrel(xd.grad.float(), dx_ref) < BF16_MAXREL
    assert abs(float(model.log_temperature_text.grad) - float(ref["dlogtau"])) <= BF16_MAXREL * abs(float(ref["dlogtau"]))
    # the default capacity keeps its meaning: the same draw at 256 rows trims distractors
    torch.manual_seed(11)
    _, aux256 = losses.text_contrastive_loss(xd.detach(), segd, textd, sets, model.log_temperature_text.detach(), 0.7, 250, 0.2,
                                             0.5, 0.3, "auto", return_aux=True, shared2x2=shared, contrast_builder="device",
                                             max_contrast=256)
    K2, flags2, _, _ = aux256["contrast_info"].tolist()
    assert K2 == 256 and flags2 == 2


@pytest.mark.parametrize("shared", [False, True])
def test_no_foreground_pixels_give_a_zero_loss_without_a_sync(shared):
    import rangeclip_b200 as R
    x, seg, text, sets = _case()
    seg = torch.zeros_like(seg)
    if shared:
        seg = torch.zeros(seg.shape[0], 2 * seg.shape[1], 2 * seg.shape[2], dtype=seg.dtype)
    model = _Model().to(dev())
    xd = x.to(dev()).to(torch.bfloat16).requires_grad_(True)
    segd, textd = seg.to(dev()), text.to(dev())
    fn = R.compute_loss_shared2x2 if shared else R.compute_loss
    kw = dict(KW, max_contrast=512)
    total, _ = fn(model, xd, segd, textd, sets, None, None, **kw)           # warm-up
    total.backward()
    torch.cuda.synchronize()
    xd.grad = None; model.zero_grad()
    torch.cuda.set_sync_debug_mode("error")
    try:
        total, info = fn(model, xd, segd, textd, sets, None, None, **kw)
        total.backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert float(total) == 0.0
    assert torch.isfinite(xd.grad).all() and float(xd.grad.float().abs().max()) == 0.0
    assert float(model.log_temperature_text.grad) == 0.0


def test_sync_free_compute_loss_above_256_rows_is_cuda_graph_capturable():
    """compute_loss(contrast_builder="device", max_contrast=512) + backward in ONE CUDA graph: replays draw new sets (K
    varies around 256 + present labels), stay finite and near the eager loss"""
    import rangeclip_b200 as R
    from rangeclip_b200 import losses as LS
    x, seg, text, sets = _case(B=2, D=256, H=32, W=32, seed=5)
    model = _Model().to(dev())
    xd = x.to(dev()).to(torch.bfloat16).requires_grad_(True)
    segd, textd = seg.to(dev()), text.to(dev())
    kw = dict(KW, max_contrast=512)
    params = [xd, model.log_temperature_text]
    eager = []
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            total, info = R.compute_loss(model, xd, segd, textd, sets, None, None, **kw)
            torch.autograd.grad(total, params)
            eager.append(float(total))
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    captured = {}
    real = LS.text_contrastive_loss

    def spy(*a, **k):                    # keeps the captured call's contrast_info, to see K move from replay to replay
        out = real(*a, **k)
        captured["info"] = out[1]["contrast_info"]
        return out

    graph = torch.cuda.CUDAGraph()
    LS.text_contrastive_loss = spy
    try:
        with torch.cuda.graph(graph):
            total, info = R.compute_loss(model, xd, segd, textd, sets, None, None, **kw)
            gx, gtau = torch.autograd.grad(total, params)
    finally:
        LS.text_contrastive_loss = real
    losses, ks = [], []
    for _ in range(4):
        graph.replay()
        torch.cuda.synchronize()
        losses.append(float(total))
        ks.append(int(captured["info"][0]))
        assert info["total_loss"] == pytest.approx(float(total), rel=1e-6)
        assert torch.isfinite(gx).all() and float(gx.float().abs().sum()) > 0 and torch.isfinite(gtau)
    assert all(k > 256 for k in ks), ks
    assert len(set(losses)) > 1
    mean_eager = sum(eager) / len(eager)
    assert all(abs(l - mean_eager) < 0.1 * abs(mean_eager) for l in losses), (losses, eager)


@pytest.mark.parametrize("rep", [1, 4])
def test_opcheck_infonce_device_blocks(rep):
    import rangeclip_b200  # noqa: F401  (registers torch.ops.rangeclip.*)
    B, D, HW, K = 1, 512, 128, 300
    x, t, y, w = OR.make_case(B, D, HW, K, rep, seed=9 + rep)
    xd = x.view(B, D, 8, 16).to(dev()).requires_grad_(True)
    log_tau = torch.tensor(math.log(0.07), device=dev(), requires_grad=True)
    args = (xd, _padded(t, 512), log_tau, y.to(dev()), w.to(dev()), True, False, "bf16", rep, None, None, _kinfo(K), True)
    torch.library.opcheck(torch.ops.rangeclip.infonce.default, args,
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
    if rep == 1:
        args = (xd, _padded(t, 512), log_tau, y.to(dev()), w.to(dev()), True, False, "bf16", None, None, _kinfo(K), True)
        torch.library.opcheck(torch.ops.rangeclip.pixel_losses.default, args,
                              test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
