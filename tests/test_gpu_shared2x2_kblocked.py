"""More than 256 contrast rows on the shared 2x2 embeddings: the four-target InfoNCE kernel in blocks of 256 candidate rows
(ops.infonce_kblocked_raw(rep=4): a forward round for the per-block logsumexp, then fwd+bwd launches with the row's lse given).

Checked against an autograd reference of the loss on normalize(nearest_x2(x)) (decoder.py:113-114), against the path it
replaces (the full-resolution K-blocked loss of the upsampled tensor), TS kernel against SS kernel bit for bit, and through
the public compute_loss_shared2x2.  bf16 tensor-core contract: 2e-3 relative on the loss, 2e-2 max-relative on dX and
dlogtau; the lse comes from fp32 logits and sums."""
import math
from unittest import mock

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF16_MAXREL = 2e-2
LOSS_REL = 2e-3
LSE_MAXREL = 1e-4
TS, SS = 0, 32      # the default backward kernel (TS), RC_INFONCE_SS_KERNEL


def dev():
    return torch.device("cuda:0")


def maxrel(a, b):
    a = np.asarray(a.detach().double().cpu() if torch.is_tensor(a) else a, dtype=np.float64)
    b = np.asarray(b.detach().double().cpu() if torch.is_tensor(b) else b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _case(B, D, h, w, K, seed):
    """x [B, D, h, w] (bf16-exact values), t [K, D] normalised (bf16-exact), full-resolution targets y / weights wt [B, 2h, 2w]
    with ignored pixels, duplicate and mixed labels in a block, blocks whose targets lie in different candidate blocks, and
    blocks of zero weight."""
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(B, D, h, w, generator=g) * (0.5 + torch.rand(B, 1, h, w, generator=g))).to(torch.bfloat16).float()
    t = F.normalize(torch.randn(K, D, generator=g), dim=1).to(torch.bfloat16).float()
    M = B * h * w
    y4 = torch.randint(0, K, (M, 1), generator=g, dtype=torch.int32).repeat(1, 4)     # mostly one label per block ...
    mixed = torch.rand(M, 4, generator=g) < 0.3                                         # ... some mixed, with duplicates
    y4 = torch.where(mixed, torch.randint(0, K, (M, 4), generator=g, dtype=torch.int32), y4)
    y4[torch.rand(M, 4, generator=g) < 0.15] = -1
    y4[torch.rand(M, generator=g) < 0.05] = -1                                          # blocks without a target
    w4 = torch.randint(0, 4, (M, 4), generator=g).float()
    w4[torch.rand(M, generator=g) < 0.05] = 0.0                                         # blocks of zero weight
    y4[0] = torch.tensor([0, K - 1, K // 2, K // 3])           # four targets in (up to) four candidate blocks
    y4[1] = torch.tensor([K - 1, 3, K - 1, 3])                 # duplicates across two blocks
    w4[0] = torch.tensor([1.0, 2.0, 3.0, 1.0])
    w4[1] = torch.tensor([2.0, 1.0, 1.0, 3.0])
    y4[2] = torch.tensor([-1, K - 1, -1, 7])
    w4[2] = torch.tensor([3.0, 1.0, 0.0, 2.0])                 # an ignored target with a non-zero weight
    H, W = 2 * h, 2 * w
    y = y4.view(B, h, w, 2, 2).permute(0, 1, 3, 2, 4).reshape(B, H, W)
    wt = w4.view(B, h, w, 2, 2).permute(0, 1, 3, 2, 4).reshape(B, H, W)
    return x, t, y, wt


def _group(t):
    from rangeclip_b200.losses import group_2x2
    return group_2x2(t)


def _reference(x, t, y, wt, log_tau):
    """float64 autograd of sum_p w_p (lse_p - z_p,y_p) / sum w on normalize(nearest_x2(x)): loss, per-row lse, dX, dlogtau."""
    xr = x.to(dev()).double().requires_grad_(True)
    lt = torch.tensor(float(log_tau), device=dev(), dtype=torch.float64, requires_grad=True)
    up = F.normalize(F.interpolate(xr, scale_factor=2, mode="nearest"), dim=1)
    z = torch.einsum("bdhw,kd->bhwk", up, t.to(dev()).double()) * torch.exp(-lt)
    lse = torch.logsumexp(z, dim=-1)
    yd, wd = y.to(dev()).long(), wt.to(dev()).double() * (y.to(dev()) >= 0)
    zy = torch.gather(z, -1, yd.clamp_min(0)[..., None])[..., 0]
    loss = (wd * (lse - zy)).sum() / wd.sum()
    loss.backward()
    return dict(loss=float(loss), lse=lse.detach()[:, ::2, ::2].reshape(-1), dx=xr.grad, dlogtau=float(lt.grad))


CASES = [
    # B, D, h, w, K, x dtype
    (2, 512, 16, 16, 257, torch.bfloat16),    # one-row last block
    (1, 256, 10, 12, 300, torch.float32),     # 120 rows: not a multiple of 128
    (1, 512, 20, 32, 512, torch.bfloat16),    # 5 tiles: an odd number of tile pairs
    (2, 512, 12, 20, 600, torch.float32),     # 240 rows per image
    (2, 256, 16, 16, 1100, torch.bfloat16),   # 5 blocks: dX summed on the host
    (1, 512, 9, 24, 1100, torch.float32),
]


@pytest.mark.parametrize("B,D,h,w,K,xdtype", CASES)
def test_kblocked_rep4_matches_the_autograd_reference(B, D, h, w, K, xdtype):
    from rangeclip_b200 import ops
    tau = 0.07
    x, t, y, wt = _case(B, D, h, w, K, seed=B * 7 + D + K + h)
    ref = _reference(x, t, y, wt, math.log(tau))
    xd = x.to(dev()).to(xdtype)
    y4, w4 = _group(y.to(dev())), _group(wt.to(dev()))
    r = ops.infonce_raw(xd, t.to(dev()), y4, w4, 1.0 / tau, True, False, "auto", rep=4)
    assert r["precision"] == "bf16-kblocked"
    loss = float(r["loss_sum"] / r["w_sum"])
    assert float(r["w_sum"]) == float((wt * (y >= 0)).sum())
    assert abs(loss - ref["loss"]) <= LOSS_REL * abs(ref["loss"]), (loss, ref["loss"])
    assert maxrel(r["lse"], ref["lse"]) < LSE_MAXREL, maxrel(r["lse"], ref["lse"])
    assert r["dx"].dtype == xdtype and r["dx"].shape == xd.shape
    assert maxrel(r["dx"], ref["dx"]) < BF16_MAXREL, maxrel(r["dx"], ref["dx"])
    assert abs(float(r["dlogtau"]) - ref["dlogtau"]) <= BF16_MAXREL * abs(ref["dlogtau"])
    # forward only: the same loss from the first round alone
    r0 = ops.infonce_raw(xd, t.to(dev()), y4, w4, 1.0 / tau, False, False, "auto", rep=4)
    assert abs(float(r0["loss_sum"] / r0["w_sum"]) - loss) <= 1e-6 * abs(loss)
    # the public autograd op with an upstream gradient of 3 (grad_scale != 1)
    xg = xd.clone().requires_grad_(True)
    lt = torch.tensor(math.log(tau), device=dev(), requires_grad=True)
    out = ops.infonce(xg, t.to(dev()), lt, y4, w4, rep=4)
    (3 * out).backward()
    assert abs(float(out) - ref["loss"]) <= LOSS_REL * abs(ref["loss"])
    assert maxrel(xg.grad, 3 * ref["dx"]) < BF16_MAXREL, maxrel(xg.grad, 3 * ref["dx"])
    assert abs(float(lt.grad) - 3 * ref["dlogtau"]) <= BF16_MAXREL * abs(3 * ref["dlogtau"])


def test_all_zero_weights_give_a_zero_loss_and_gradient():
    from rangeclip_b200 import ops
    x, t, y, wt = _case(1, 512, 8, 16, 300, seed=5)
    r = ops.infonce_raw(x.to(dev()).to(torch.bfloat16), t.to(dev()), _group(y.to(dev())), torch.zeros(128, 4, device=dev()),
                        1 / 0.07, True, False, "auto", rep=4)
    assert float(r["w_sum"]) == 0.0 and float(r["loss_sum"]) == 0.0
    assert float(r["dx"].float().abs().max()) == 0.0 and float(r["dlogtau"]) == 0.0
    assert bool(torch.isfinite(r["lse"]).all())


@pytest.mark.parametrize("D,K,xdtype", [(512, 300, torch.bfloat16), (256, 600, torch.float32), (512, 1100, torch.bfloat16)])
def test_kblocked_rep4_matches_the_upsampled_kblocked_loss(D, K, xdtype):
    """The path it replaces: interpolate, the full-resolution K-blocked loss, then the 2x2 sum of its dX."""
    from rangeclip_b200 import ops
    B, h, w = 2, 16, 24
    x, t, y, wt = _case(B, D, h, w, K, seed=D + K)
    xd = x.to(dev()).to(xdtype)
    up = F.interpolate(xd, scale_factor=2, mode="nearest")
    r1 = ops.infonce_raw(up, t.to(dev()), y.to(dev()).reshape(B, -1), wt.to(dev()).reshape(B, -1), 1 / 0.07, True, False, "auto")
    r4 = ops.infonce_raw(xd, t.to(dev()), _group(y.to(dev())), _group(wt.to(dev())), 1 / 0.07, True, False, "auto", rep=4)
    assert r1["precision"] == r4["precision"] == "bf16-kblocked"
    assert float(r1["w_sum"]) == float(r4["w_sum"])
    l1, l4 = float(r1["loss_sum"] / r1["w_sum"]), float(r4["loss_sum"] / r4["w_sum"])
    assert abs(l4 - l1) <= LOSS_REL * abs(l1)
    lse1 = r1["lse"].view(B, 2 * h, 2 * w)[:, ::2, ::2].reshape(-1)
    assert maxrel(r4["lse"], lse1) < LSE_MAXREL
    dsum = r1["dx"].float().view(B, D, h, 2, w, 2).sum(dim=(3, 5))
    assert maxrel(r4["dx"], dsum) < BF16_MAXREL, maxrel(r4["dx"], dsum)
    assert abs(float(r4["dlogtau"]) - float(r1["dlogtau"])) <= BF16_MAXREL * abs(float(r1["dlogtau"]))


def _launch_block(L, x, tb, ttb, Kb, y_rel, w4, lse, dx, flags):
    from rangeclip_b200 import _lib
    B, D, h, w = x.shape
    HW = h * w
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, Kb, _lib.RC_BF16))
    ws = torch.empty(ws_bytes, device=dev(), dtype=torch.uint8)
    acc = torch.zeros(4, device=dev(), dtype=torch.float64)
    acc[3] = w4.double().sum()
    _lib.check(L.rc_infonce_bf16_rep4(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), Kb, y_rel.data_ptr(),
                                      w4.data_ptr(), 1 / 0.07, lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(),
                                      acc[3:].data_ptr() if dx is not None else None, None,
                                      dx.data_ptr() if dx is not None else None, None,
                                      acc[2:].data_ptr() if dx is not None else None, ws.data_ptr(), ws_bytes, flags,
                                      torch.cuda.current_stream().cuda_stream), "rc_infonce_bf16_rep4")
    torch.cuda.synchronize()
    return dict(lse=lse, dx=dx, loss_sum=acc[0], w_sum=acc[1], dlogtau=acc[2])


def _assert_sums_equal(a, b, keys):
    for k in keys:
        u, v = float(a[k]), float(b[k])
        assert abs(u - v) <= 1e-12 * max(1.0, abs(v)), (k, u, v)


@pytest.mark.parametrize("s0", [0, 256])
def test_ts_equals_ss_kblocked_rep4_rounds(s0):
    """Both rounds of one candidate block (s0 = 0: a full block with targets beyond it; s0 = 256: the short last block of
    K = 300 with targets before it): the forward round's lse and sums, and the accumulate round's dX (TMA reduce-add onto a
    previous block's gradient) and lse, TS kernel against SS kernel bit for bit."""
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    B, D, h, w, K = 2, 512, 16, 32, 300
    x, t, y, wt = _case(B, D, h, w, K, seed=31 + s0)
    xd = x.to(dev()).to(torch.bfloat16)
    y4, w4 = _group(y.to(dev())), _group(wt.to(dev()))
    w4 = (w4 * (y4 >= 0)).contiguous()
    Kb = min(256, K - s0)
    tb, ttb = ops.text_to_bf16(t[s0:s0 + Kb].to(dev()))
    y_rel = (y4 - s0).contiguous()
    M = B * h * w
    fwd = 1 | ops.RC_INFONCE_KEEP_WEIGHT
    # round 1: a backward launch in round-1 form runs the TS / SS kernels; the forward-only launch runs the SS forward kernel
    r1 = [_launch_block(L, xd, tb, ttb, Kb, y_rel, w4, torch.empty(M, device=dev()), torch.empty_like(xd), fwd | extra)
          for extra in (TS, SS)]
    assert torch.equal(r1[0]["lse"].view(torch.int32), r1[1]["lse"].view(torch.int32))
    assert torch.equal(r1[0]["dx"].view(torch.int16), r1[1]["dx"].view(torch.int16))
    _assert_sums_equal(r1[0], r1[1], ("loss_sum", "w_sum", "dlogtau"))
    r0 = _launch_block(L, xd, tb, ttb, Kb, y_rel, w4, torch.empty(M, device=dev()), None, fwd)
    assert maxrel(r0["lse"], r1[0]["lse"]) < 1e-6
    assert abs(float(r0["loss_sum"]) - float(r1[0]["loss_sum"])) <= 1e-6 * abs(float(r1[0]["loss_sum"]))
    # round 2: lse given, weights kept, dX added to an existing gradient
    lse_in = r1[0]["lse"] + 0.25
    base = torch.randn(xd.shape, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).to(dev())
    acc_flags = fwd | ops.RC_INFONCE_LSE_GIVEN | ops.RC_INFONCE_ACCUMULATE_DX
    r2 = [_launch_block(L, xd, tb, ttb, Kb, y_rel, w4, lse_in.clone(), base.clone(), acc_flags | extra) for extra in (TS, SS)]
    assert torch.equal(r2[0]["dx"].view(torch.int16), r2[1]["dx"].view(torch.int16))
    assert torch.equal(r2[0]["lse"].view(torch.int32), lse_in.view(torch.int32))
    assert torch.equal(r2[1]["lse"].view(torch.int32), lse_in.view(torch.int32))
    _assert_sums_equal(r2[0], r2[1], ("loss_sum", "w_sum", "dlogtau"))
    assert not torch.equal(r2[0]["dx"], base)


def test_other_entry_points_keep_rejecting_rep4_kblocking():
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    x = torch.zeros(1, 512, 8, 16, device=dev(), dtype=torch.bfloat16)
    tb, ttb = ops.text_to_bf16(F.normalize(torch.randn(64, 512, device=dev()), dim=1))
    y4 = torch.zeros(128, 4, device=dev(), dtype=torch.int32)
    w4 = torch.ones(128, 4, device=dev())
    lse = torch.empty(128, device=dev())
    acc = torch.zeros(4, device=dev(), dtype=torch.float64)
    ws = torch.empty(1 << 20, device=dev(), dtype=torch.uint8)
    dt = torch.zeros(64, 512, device=dev())
    dx = torch.empty_like(x)
    st = torch.cuda.current_stream().cuda_stream
    # K-blocked flags with dText
    assert L.rc_infonce_bf16_rep4(x.data_ptr(), _lib.RC_BF16, 1, 512, 128, tb.data_ptr(), ttb.data_ptr(), 64, y4.data_ptr(),
                                  w4.data_ptr(), 10.0, lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr(),
                                  None, dx.data_ptr(), dt.data_ptr(), acc[2:].data_ptr(), ws.data_ptr(), 1 << 20,
                                  ops.RC_INFONCE_KEEP_WEIGHT, st) == -2
    assert b"no dText" in L.rc_last_error()
    kd = torch.tensor([64], device=dev(), dtype=torch.int32)
    lt = torch.zeros(1, device=dev())
    assert L.rc_infonce_bf16_dyn(x.data_ptr(), _lib.RC_BF16, 1, 512, 128, tb.data_ptr(), ttb.data_ptr(), 64, kd.data_ptr(),
                                 y4.data_ptr(), w4.data_ptr(), lt.data_ptr(), 4, lse.data_ptr(), acc[0:].data_ptr(),
                                 acc[1:].data_ptr(), None, None, None, None, ws.data_ptr(), 1 << 20, ops.RC_INFONCE_KEEP_WEIGHT,
                                 st) == -1
    torch.cuda.synchronize()


class _Model(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.log_temperature_text = torch.nn.Parameter(torch.log(torch.tensor(0.07)))
        self.log_temperature_image = torch.nn.Parameter(torch.log(torch.tensor(0.1)))


@pytest.mark.parametrize("D,C,kd,H", [(256, 400, 300, 64), (512, 700, 500, 128)])
def test_compute_loss_shared2x2_above_256_contrast_rows(D, C, kd, H):
    """The public training step at K > 256 contrast rows equals compute_loss on the decoder tail, without ever building the
    upsampled tensor (F.interpolate patched to raise); its peak memory stays below that tensor's size."""
    import rangeclip_b200 as R
    g = torch.Generator().manual_seed(D + C)
    e = torch.randn(2, D, H // 2, H // 2, generator=g).to(dev())
    seg = torch.randint(0, 9, (2, H // 4, H // 4), generator=g).repeat_interleave(4, 1).repeat_interleave(4, 2).to(dev())
    text = torch.randn(C, D, generator=g).to(dev())
    sets = {"medium": {}, "hard": {}}
    rand_idx = torch.randint(0, H * H, (2, int(0.7 * H * H)), generator=g).to(dev())
    kw = dict(W_image=0.0, W_smooth=0.0, k_distractors=kd, pct_medium=0.0, pct_hard=0.0, pct_rand=1.0)
    res = []
    peak = None
    for shared in (True, False):
        model = _Model().to(dev())
        x = e.clone().requires_grad_(True)
        np.random.seed(3); torch.manual_seed(3)
        with mock.patch("torch.randint", lambda *a, **k: rand_idx):
            if shared:
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                with mock.patch("torch.nn.functional.interpolate", side_effect=RuntimeError("upsampled")):
                    total, info = R.compute_loss_shared2x2(model, x, seg, text, sets, None, None, **kw)
                    total.backward()
                torch.cuda.synchronize()
                peak = torch.cuda.max_memory_allocated() - base
            else:
                up = F.normalize(F.interpolate(x, scale_factor=2, mode="nearest"), dim=1)
                total, info = R.compute_loss(model, up, seg, text, sets, None, None, **kw)
                total.backward()
        res.append((float(total), x.grad.float().cpu(), float(model.log_temperature_text.grad)))
    up_bytes = e.numel() * 4 * e.element_size()
    print(f"compute_loss_shared2x2 D={D} rows={H // 2}^2 K>256: peak {peak / 2**20:.2f} MiB above the inputs, "
          f"upsampled tensor {up_bytes / 2**20:.2f} MiB")
    assert peak < up_bytes, (peak, up_bytes)
    assert abs(res[0][0] - res[1][0]) <= LOSS_REL * abs(res[1][0])
    assert maxrel(res[0][1], res[1][1]) < BF16_MAXREL
    assert abs(res[0][2] - res[1][2]) <= BF16_MAXREL * abs(res[1][2])


def test_opcheck_infonce_rep4_above_256_candidates():
    import rangeclip_b200  # noqa: F401  (registers torch.ops.rangeclip.*)
    x, t, y, wt = _case(1, 512, 8, 16, 300, seed=9)
    xd = x.to(dev()).requires_grad_(True)
    log_tau = torch.tensor(math.log(0.07), device=dev(), requires_grad=True)
    args = (xd, t.to(dev()), log_tau, _group(y.to(dev())), _group(wt.to(dev())), True, False, "auto", 4, None, None)
    torch.library.opcheck(torch.ops.rangeclip.infonce.default, args,
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))
