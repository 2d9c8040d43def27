"""Row-level checks of the fused pixel-text InfoNCE: every row's lse and dX, every dText row, the loss sum and dlogtau of
each kernel form against the float64 per-row reference, within the worst-case bound of oracle/infonce_rows.py (built
from the kernels' rounding points; its derivation is that module's docstring).  The aggregate checks elsewhere in the
suite scale the dX error by the largest |dX| of the whole tensor and the lse error by the largest lse; a bug confined
to a few rows, or to rows with a small gradient, passes them.  Here a single row out of its bound fails.

Temperatures: 1, 0.07, the two sides of the kernels' switch from the fixed exp offset to the row maximum
(inv_tau 2.02 log2(e) < 100, tau = 0.029142), 0.02 and CLIP's clamp 0.01.  Forms: the TS backward kernel (default), the
SS kernel (RC_INFONCE_SS_KERNEL, forward-only launches), the single-CTA kernel (D = 128 / 384), the device-parameter
launch (_dyn, log tau and K read on the device) for one and four targets per row, the one-launch K-blocked form
(kblocks), the two-round K-blocked path for one and four targets per row, dText, an fp32 x through the pre-pass and the
fp32 CUDA-core kernel.  The inputs (oracle/infonce_rows.make_case) put targets on the column-half and K boundaries,
special rows in the partial last tile, confident and near-uniform rows, zero / large weights, ignored and duplicate
targets and rows whose norm F.normalize clamps.  The K-blocked overflow case (make_overflow_case) has lse - (largest
logit of the target's block) of ~2 / tau.

Run with -s to see the worst error-to-bound ratio of each case."""
import math

import pytest
import torch

from oracle import infonce_rows as O

pytestmark = pytest.mark.gpu

TAUS = [1.0, 0.07, 0.0292, 0.0291, 0.02, 0.01]
TS, SS = 0, 32


def dev():
    return torch.device("cuda:0")


def _rows(a, B, D, HW):
    """[B, D, HW] -> [B * HW, D] float64 on the host"""
    return a.detach().reshape(B, D, HW).permute(0, 2, 1).reshape(B * HW, D).double().cpu()


def _check_rows(name, err, bound):
    err, bound = err.double(), bound.double()
    assert bool(torch.isfinite(err).all()), f"{name}: non-finite rows {torch.nonzero(~torch.isfinite(err))[:8].flatten().tolist()}"
    ratio = err / bound
    worst = float(ratio.max())
    bad = torch.nonzero(ratio > 1).flatten()
    assert bad.numel() == 0, (f"{name}: {bad.numel()} rows out of bound, worst ratio {worst:.3g} at row {int(ratio.argmax())} "
                              f"(first rows {bad[:8].tolist()})")
    return worst


def _check_case(tag, r, ref, D, Kb, nb=1, lse_given=False, store_points=None, n_acc=64, check_dx=True):
    """dX per row, lse per row, loss sum and dlogtau against the bounds; prints the worst ratios."""
    out = {}
    B, Dx, HW = r["shape"]
    lse = r["lse"].double().cpu()
    out["lse"] = _check_rows(f"{tag} lse", (lse - ref["lse"]).abs(), O.lse_bound(ref, D, Kb, nb))
    loss_b, dlt_b = O.sums_bounds(ref, D, Kb, n_acc, nb, lse_given)
    e_loss = abs(float(r["loss_sum"]) - float(ref["loss_sum"]))
    assert math.isfinite(float(r["loss_sum"])) and e_loss <= loss_b, (tag, "loss_sum", e_loss, loss_b)
    out["loss"] = e_loss / loss_b
    if check_dx:
        dx = _rows(r["dx"].float(), B, Dx, HW)
        out["dx"] = _check_rows(f"{tag} dx", (dx - ref["dx"]).norm(dim=1),
                                O.dx_bound(ref, D, Kb, store_points=store_points, lse_given=lse_given, nb=nb))
        e_dlt = abs(float(r["dlogtau"]) - float(ref["dlogtau"]))
        assert math.isfinite(float(r["dlogtau"])) and e_dlt <= dlt_b, (tag, "dlogtau", e_dlt, dlt_b)
        out["dlogtau"] = e_dlt / dlt_b
    print(f"\n[rows] {tag}: worst error / bound " + ", ".join(f"{k} {v:.3f}" for k, v in out.items()))
    return out


def _launch(x, t, y, w, inv_tau, form, xdtype=torch.bfloat16):
    from rangeclip_b200 import ops
    B, D, HW = x.shape
    xd = x.to(dev()).to(xdtype)
    td, yd, wd = t.to(dev()), y.to(dev()), w.to(dev())
    rep = 4 if y.dim() == 2 else 1
    if form == "dyn":
        lt = torch.tensor(math.log(1.0 / inv_tau), dtype=torch.float32)
        r = ops.infonce_raw(xd, td, yd, wd, 0.0, True, False, "bf16", t_bf16=ops.text_to_bf16(td), rep=rep,
                            k_dev=torch.tensor([t.shape[0]], dtype=torch.int32, device=dev()), log_tau_dev=lt.to(dev()))
    elif form == "fwd":
        r = ops.infonce_raw(xd, td, yd, wd, inv_tau, False, False, "bf16", rep=rep)
    elif form == "dtext":
        r = ops.infonce_raw(xd, td, yd, wd, inv_tau, True, True, "bf16")
    elif form == "simt":
        r = ops.infonce_raw(xd, td, yd, wd, inv_tau, True, False, "fp32")
    elif form in ("kblocked", "kblocks"):
        r = ops.infonce_raw(xd, td, yd, wd, inv_tau, True, False, "auto", rep=rep)
        assert r["precision"] == "bf16-kblocked"
    else:
        r = ops.infonce_raw(xd, td, yd, wd, inv_tau, True, False, "bf16", rep=rep, flags=SS if form == "ss" else TS)
    torch.cuda.synchronize()
    r = dict(r)
    r["shape"] = (B, D, HW)
    return r


def _ref(x, t, y, w, inv_tau):
    B, D, HW = x.shape
    return O.reference(_rows(x, B, D, HW), t, y, w, inv_tau)


# (form, B, D, HW, K, R): small shapes; HW not a multiple of 128 gives a partial last tile, B * tiles odd an odd tile count
FORMS = [
    ("ts", 2, 256, 200, 200, 1),
    ("ts", 1, 512, 328, 256, 4),
    ("ss", 3, 256, 136, 100, 1),
    ("ss", 1, 256, 200, 256, 4),
    ("fwd", 1, 512, 328, 130, 1),
    ("fwd", 1, 256, 200, 70, 4),
    ("cta1", 2, 128, 72, 40, 1),
    ("cta1", 1, 384, 200, 256, 1),
    ("dyn", 2, 256, 200, 150, 1),
    ("dyn", 1, 512, 200, 256, 4),
    ("dtext", 1, 256, 328, 120, 1),
    ("f32x", 2, 512, 136, 200, 1),
]


def _form_id(f):
    return f"{f[0]}-B{f[1]}-D{f[2]}-HW{f[3]}-K{f[4]}-R{f[5]}"


@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("form", FORMS, ids=_form_id)
def test_rows_single_launch(form, tau):
    name, B, D, HW, K, R = form
    x, t, y, w = O.make_case(B, D, HW, K, R, seed=B * 1000 + D + HW + K + R)
    inv_tau = 1.0 / tau
    if name == "dyn":           # the kernel computes inv_tau = expf(-log tau) from the fp32 log tau
        inv_tau = math.exp(-float(torch.tensor(math.log(tau), dtype=torch.float32)))
    r = _launch(x, t, y, w, 1.0 / tau, name, torch.float32 if name == "f32x" else torch.bfloat16)
    ref = _ref(x, t, y, w, inv_tau)
    _check_case(f"{_form_id(form)} tau={tau}", r, ref, D, K, check_dx=name != "fwd")
    if name == "dtext":
        dt = r["dt"].double().cpu()
        worst = _check_rows(f"{_form_id(form)} tau={tau} dText", (dt - ref["dt"]).norm(dim=1), O.dt_bound(ref, D, K))
        print(f"[rows] {_form_id(form)} tau={tau}: dText worst error / bound {worst:.3f}")


KB_FORMS = [
    ("kblocked", 2, 256, 136, 300, 1),
    ("kblocked", 2, 512, 200, 600, 1),
    ("kblocked", 1, 256, 200, 300, 4),
    ("kblocked", 2, 512, 72, 600, 4),
    ("kblocks", 1, 256, 256, 300, 1),
    ("kblocks", 1, 512, 512, 600, 1),
]


def _kb_check(tag, r, ref, D, K, R, B, HW):
    nb = (K + 255) // 256
    in_kernel = not (R == 1 and B == 1 and HW % 256 == 0) and nb <= 4
    sp = O.store_points_kblocked(ref, in_kernel)
    _check_case(tag, r, ref, D, 256, nb=nb, lse_given=True, store_points=sp, n_acc=64 * nb)


@pytest.mark.parametrize("tau", TAUS)
@pytest.mark.parametrize("form", KB_FORMS, ids=_form_id)
def test_rows_kblocked(form, tau):
    name, B, D, HW, K, R = form
    x, t, y, w = O.make_case(B, D, HW, K, R, seed=B * 1000 + D + HW + K + R)
    r = _launch(x, t, y, w, 1.0 / tau, name)
    _kb_check(f"{_form_id(form)} tau={tau}", r, _ref(x, t, y, w, 1.0 / tau), D, K, R, B, HW)


@pytest.mark.parametrize("tau", [0.07, 0.0291, 0.01])
def test_rows_fp32_simt(tau):
    """The fp32 CUDA-core kernel: its 1e-5 relative contract per row (plus the fp32 logit error the softmax carries)."""
    B, D, HW, K, R = 2, 256, 72, 60, 1
    x, t, y, w = O.make_case(B, D, HW, K, R, seed=77)
    r = _launch(x, t, y, w, 1.0 / tau, "simt", torch.float32)
    ref = _ref(x, t, y, w, 1.0 / tau)
    dx = _rows(r["dx"], B, D, HW)
    err = (dx - ref["dx"]).norm(dim=1)
    worst = _check_rows(f"simt tau={tau} dx", err, O.dx_bound_f32(ref, D))
    lse = r["lse"].double().cpu()
    wl = _check_rows(f"simt tau={tau} lse", (lse - ref["lse"]).abs(), 1e-5 * (ref["lse"].abs() + 1))
    plain = float((err / (1e-5 * ref["dx"].norm(dim=1) + 1e-30)).max())
    print(f"\n[rows] simt tau={tau}: worst error / bound dx {worst:.3f}, lse {wl:.3f}; against 1e-5 |ref_r| alone {plain:.3f}")


@pytest.mark.parametrize("tau", [0.02, 0.01])
@pytest.mark.parametrize("R,B,HW", [(1, 2, 128), (4, 2, 128), (1, 1, 256)], ids=["R1", "R4", "R1-kblocks"])
def test_kblocked_lse_far_above_the_target_block(R, B, HW, tau):
    """Targets in a block whose largest logit lies ~2 / tau below the row's lse: finite dX that matches the reference."""
    D, K = 256, 300
    x, t, y, w = O.make_overflow_case(B, D, HW, K, R, seed=11 + R + B)
    ref = _ref(x, t, y, w, 1.0 / tau)
    gap = float((ref["lse"] - ref["z"][:, 256:].amax(1)).max())
    assert gap > 128 * math.log(2), gap
    r = _launch(x, t, y, w, 1.0 / tau, "kblocked" if B > 1 or R == 4 else "kblocks")
    dx = _rows(r["dx"].float(), B, D, HW)
    assert bool(torch.isfinite(dx).all()), f"non-finite dX in {int((~torch.isfinite(dx)).any(1).sum())} rows (lse - block max {gap:.1f})"
    print(f"\n[rows] overflow case R={R} B={B} tau={tau}: lse - block-1 max up to {gap:.1f} nats")
    _kb_check(f"overflow R={R} B={B} HW={HW} tau={tau}", r, ref, D, K, R, B, HW)
