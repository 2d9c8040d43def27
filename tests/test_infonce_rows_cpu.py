"""Calibration of the row-level InfoNCE bound (oracle/infonce_rows.py) without a GPU.

A torch emulation of one tensor-core launch at the kernels' rounding points (bf16 e, bf16 rsv, their bf16 product,
fp32 target entries, fp32 accumulation, bf16 dX) must stay within the bound on the inputs and temperatures of
tests/test_gpu_infonce_rows.py, with room to spare; the worst ratio is printed (-s) and asserted below 0.5.  Three
wrong results must each put at least one row out of bound -- the one-hot weight dropped for targets in the second
column half, one row's dX scaled (below), the target entry rounded before its subtraction -- and the test records which
of them the suite's aggregate checks (2e-2 max-relative dX, 2e-3 on lse and the mean loss) would let through.

A row scaled by 1.02 is NOT detectable by a worst-case bound: three bf16 roundings of up to 2^-8 each on every entry of
G already allow ~1.2 % of sum_k |G_k| |t_k|, which is at least |dX_r|, and with the safety factor of 2 and the store
rounding the bound is 3.8-5 % of |dX_r| on the rows of this grid.  The scaling variant therefore scales the row with the
tightest bound by 1.05.  The rounded target entry shows on rows of moderate confidence (p_y ~ 0.99 at tau = 0.07),
where |e_y - sum| rs is a few bf16 steps of rs; on extremely confident rows it is below the logit-error term."""
import pytest
import torch

from oracle import infonce_rows as O

TAUS = [1.0, 0.07, 0.0292, 0.0291, 0.02, 0.01]
# (B, D, HW, K, R): the single-launch shapes of the GPU grid
SHAPES = [(2, 256, 200, 200, 1), (1, 512, 328, 256, 4), (3, 256, 136, 100, 1), (1, 256, 200, 256, 4), (2, 128, 72, 40, 1),
          (1, 384, 200, 256, 1), (1, 256, 328, 120, 1)]


def _rows(x):
    B, D, HW = x.shape
    return x.permute(0, 2, 1).reshape(B * HW, D)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "B{}-D{}-HW{}-K{}-R{}".format(*s))
def test_emulated_kernel_is_well_inside_the_row_bound(shape):
    B, D, HW, K, R = shape
    x, t, y, w = O.make_case(B, D, HW, K, R, seed=B * 1000 + D + HW + K + R)
    xr = _rows(x)
    worst = {}
    for tau in TAUS:
        ref = O.reference(xr, t, y, w, 1.0 / tau)
        em = O.emulate_bf16(xr, t, y, w, 1.0 / tau)
        err = (em["dx"].double() - ref["dx"]).norm(dim=1)
        assert bool(torch.isfinite(err).all())
        rdx = float((err / O.dx_bound(ref, D, K)).max())
        rl = float(((em["lse"].double() - ref["lse"]).abs() / O.lse_bound(ref, D, K)).max())
        worst[tau] = (rdx, rl)
        assert rdx < 0.5 and rl < 0.5, (tau, rdx, rl)
    print("\n[rows-emulation] " + str(shape) + ": worst error / bound (dx, lse) per tau: "
          + ", ".join(f"{tau}: {a:.3f} / {b:.3f}" for tau, (a, b) in worst.items()))


@pytest.mark.parametrize("mutant,tau,slips_through", [("drop_w_hi", 0.07, False), ("scale_row", 0.02, True), ("round_y", 0.07, True)])
def test_wrong_results_break_the_row_bound(mutant, tau, slips_through):
    """Each wrong variant puts at least one row out of bound; the second and third pass the aggregate checks."""
    B, D, HW, K, R = 2, 256, 200, 200, 1
    x, t, y, w = O.make_case(B, D, HW, K, R, seed=B * 1000 + D + HW + K + R)
    xr = _rows(x)
    ref = O.reference(xr, t, y, w, 1.0 / tau)
    bound = O.dx_bound(ref, D, K)
    if mutant == "scale_row":
        em = O.emulate_bf16(xr, t, y, w, 1.0 / tau)
        rel = torch.where(ref["wrow"] > 0, bound / ref["dx"].norm(dim=1).clamp_min(1e-300), torch.full_like(bound, float("inf")))
        em["dx"][int(rel.argmin())] *= 1.05
    else:
        em = O.emulate_bf16(xr, t, y, w, 1.0 / tau, mutate=mutant)
    ratio = (em["dx"].double() - ref["dx"]).norm(dim=1) / bound
    n_bad = int((ratio > 1).sum())
    accepted = O.global_checks_accept(em["dx"], em["lse"], em["loss_sum"], em["wsum"], ref)
    print(f"\n[rows-mutant] {mutant}: {n_bad} rows out of bound (worst ratio {float(ratio.max()):.1f}); "
          f"aggregate checks {'accept' if accepted else 'reject'} it")
    assert n_bad >= 1
    assert accepted == slips_through
    # the correct emulation on the same input passes both
    ok = O.emulate_bf16(xr, t, y, w, 1.0 / tau)
    assert O.global_checks_accept(ok["dx"], ok["lse"], ok["loss_sum"], ok["wsum"], ref)
    assert bool(((ok["dx"].double() - ref["dx"]).norm(dim=1) <= O.dx_bound(ref, D, K)).all())
