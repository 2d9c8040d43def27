"""Row-level checker for the fused pixel-text InfoNCE: a float64 reference of every row's lse, loss term, softmax
gradient and dX, dText per text row, and a worst-case bound on each of them for the tensor-core kernels.

TEST INFRASTRUCTURE ONLY (tests/test_gpu_infonce_rows.py, tests/test_infonce_rows_cpu.py); nothing under
``rangeclip_b200/`` imports it.

Notation, row r (an embedding row; R = 1 target per row, or the four targets of a shared 2x2 block), candidate k:
  inv_n = 1 / max(|x_r|, 1e-12)            (F.normalize, eps 1e-12), xn = x_r inv_n, s = |xn| (1, or < 1 when clamped)
  z_k = inv_tau xn . t_k,  p = softmax(z),  lse = logsumexp(z)
  W_k = sum_j w_j [y_j = k]  (ignored targets y_j < 0 carry no weight),  wrow = sum_k W_k
  Gt_k = p_k - W_k / wrow                  (Gt = 0 on a row of zero weight)
  coef = gscale wrow / wsum,  rs = inv_n inv_tau coef
  dX_r = rs sum_k Gt_k t_k - inv_n coef (sum_k Gt_k z_k) xn     (no projection term when |x_r| < 1e-12: F.normalize is
                                                                  then x / eps, whose Jacobian is I / eps)
  loss term = wrow lse - sum_j w_j z_{y_j};  dText_k = sum_r rs Gt_rk x_r;  dlogtau = -sum_r coef sum_k Gt_k z_k.

The bound follows the kernels' rounding points (u = 2^-24 the fp32 unit roundoff, b = 2^-8 the bf16 one; tensor-core
products of bf16 operands are exact in fp32; one fp32 rounding -- 2^-23 to allow truncation -- per 16-deep MMA step):
  * logits: S = x . t_k accumulated in fp32 over D, |dS| <= (D/16 + 2) 2^-23 |x| |t_k|; row norm from an fp32 sum of
    squares, |d inv_n| / inv_n <= eps_n = (D + 8) u / 2 + 2 u; the exponent fma(S, zl, -ml) with zl = inv_n inv_tau
    log2(e) (two roundings) and one rounding of the result; ex2.approx.ftz (relative error < 2^-21).  Together a logit
    error eps_z (nats), the same for every column of the row.  A K-blocked round that is given the row's lse also
    carries the error of that lse.
  * the softmax: sum = sum_k e_k in fp32 (relative error eps_sum = (Kb + 8) u); an error eps_z on every logit moves
    p_k by at most 2 eps_z p_k.  Term C = rs (2 eps_z + eps_sum) sum_k p_k |t_k|.
  * the stored G: e -> bf16, rsv = rs / sum -> bf16, the non-target entries are the bf16 product of the two: three
    roundings, relative (1 + b)^3 - 1; the target entries are formed in fp32 (e_y - sum W_k / wrow) rsv and rounded once.
    The dX GEMM accumulates G t in fp32 ((Kb / 16 + 2) 2^-23).  Term A = alpha rs sum_k |Gt_k| |t_k| with
    alpha = (1 + b)^3 - 1 + (Kb / 16 + 2) 2^-23.
  * the target entries cancel (e_y - sum W_k / wrow) on confident rows, so their error does not scale with |Gt_k|:
    Term B = rs (eps_sum + 4 u) sum_{k targeted} (p_k + W_k / wrow) |t_k|.
  * the projection: cj = coef (sez zs / sum - tz zs / wrow) with sez = sum_k e_k S_k and tz = sum_j w_j S_{y_j} in
    fp32; |d cj| <= coef [(2 eps_z + 2 eps_sum + (K + 8) u) sum_k p_k |z_k| + 2 eps_z + 4 u (sum p |z| + sum W |z_y| /
    wrow)], and dx = acc - inv_n^2 cj x adds inv_n s (|d cj| + |cj| (2 eps_n + 3 u)).  Term P.
  * underflow: ex2.approx.ftz and the bf16 products flush below 2^-126.  Term F = (rs + 1) K 2^-120.
  * the dX stores: bf16, b |value| at every rounding point -- once for a single launch; K-blocked launches that add
    into the same bf16 tensor round every partial sum; more than four K blocks round each block's dX once and add them
    in fp32.  Term S = b (1 + 2^-6) sum over the rounding points of |the exact value there|.
  |dX_r - ref_r|_2 <= c (A + B + C + P + F) + S, c = 2 (a safety factor over the first-order terms above).
lse: (ml + log2 sum) ln 2 with ml fp32, __log2f (absolute error < 2^-21): |d lse| <= c (eps_z + eps_sum + 2^-21 +
6 u (|lse| + 1)) -- about 1e-4 nats at tau = 0.07 -- and the host logsumexp over K blocks adds (nb + 2) 2 u (|lse| + 1).
The loss sum, dlogtau and every dText row are bounded by the sums of these per-row terms over the rows that feed them.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

U = 2.0 ** -24          # fp32 unit roundoff
BF = 2.0 ** -8          # bf16 unit roundoff (8 significant bits)
SAFETY = 2.0


def targets_and_weights(y: torch.Tensor, w: torch.Tensor, K: int):
    """y, w [M] or [M, R] -> (y [M, R] long, w [M, R] float64 with ignored targets at weight 0, W [M, K] float64)."""
    y = y.reshape(y.shape[0], -1).long()
    w = w.reshape(y.shape).double() * (y >= 0)
    W = torch.zeros(y.shape[0], K, dtype=torch.float64)
    W.scatter_add_(1, y.clamp_min(0), w)
    return y, w, W


def reference(x: torch.Tensor, t: torch.Tensor, y: torch.Tensor, w: torch.Tensor, inv_tau: float, gscale: float = 1.0,
              block: int = 256) -> Dict[str, torch.Tensor]:
    """float64 per-row reference.  x [M, D] (the values the kernel reads), t [K, D], y / w [M] or [M, R].
    Returns dict with the per-row lse, loss (term per row), Gt [M, K], p, z, dx [M, D], dx_blocks [nb, M, D] (the part
    of dX from each block of `block` candidates, as a K-blocked launch computes it), dt [K, D], dlogtau, loss_sum, wsum,
    and what the bound needs (inv_n, s, rs, coef, cj, wrow, W)."""
    x = x.double()
    t = t.double()
    M, D = x.shape
    K = t.shape[0]
    yy, ww, W = targets_and_weights(y, w, K)
    nrm = x.norm(dim=1)
    clamped = nrm < 1e-12
    inv_n = 1.0 / nrm.clamp_min(1e-12)
    xn = x * inv_n[:, None]
    s = xn.norm(dim=1)
    z = (xn @ t.T) * inv_tau
    lse = torch.logsumexp(z, dim=1)
    p = torch.softmax(z, dim=1)
    wrow = W.sum(1)
    wsum = wrow.sum()
    has_w = wrow > 0
    Gt = torch.where(has_w[:, None], p - W / wrow.clamp_min(1e-300)[:, None], torch.zeros_like(p))
    coef = gscale * wrow / wsum if float(wsum) > 0 else torch.zeros_like(wrow)
    rs = inv_n * inv_tau * coef
    proj = torch.where(clamped, torch.zeros_like(inv_n), inv_n * coef)       # inv_n coef, 0 when the norm is clamped
    nb = (K + block - 1) // block
    dx_blocks = torch.zeros(nb, M, D, dtype=torch.float64)
    cj = torch.zeros(M, dtype=torch.float64)
    for b in range(nb):
        sl = slice(b * block, min(K, (b + 1) * block))
        cj_b = coef * (Gt[:, sl] * z[:, sl]).sum(1)
        cj += cj_b
        dx_blocks[b] = rs[:, None] * (Gt[:, sl] @ t[sl]) - (proj * (Gt[:, sl] * z[:, sl]).sum(1))[:, None] * xn
    dx = dx_blocks.sum(0)
    loss = wrow * lse - (ww * z.gather(1, yy.clamp_min(0))).sum(1)
    dt = (rs[:, None] * Gt).T @ x
    return dict(lse=lse, loss=loss, loss_sum=loss.sum(), wsum=wsum, Gt=Gt, p=p, z=z, dx=dx, dx_blocks=dx_blocks, dt=dt,
                dlogtau=-cj.sum(), inv_n=inv_n, s=s, rs=rs, coef=coef, cj=cj, wrow=wrow, W=W, y=yy, w=ww, t=t, x=x,
                inv_tau=torch.tensor(inv_tau, dtype=torch.float64), clamped=clamped)


def _logit_error(ref, D: int, Kb: int):
    """(eps_z [M] in nats, eps_sum) of the tensor-core kernels."""
    inv_tau = float(ref["inv_tau"])
    tmax = float(ref["t"].norm(dim=1).max())
    cmax = ref["z"].abs().amax(1) / inv_tau
    eps_n = (D + 8) * U / 2 + 2 * U
    eps_z = (inv_tau * ((D / 16 + 2) * 2.0 ** -23 * tmax + (eps_n + 3 * U) * cmax) + 2.0 ** -21
             + (3 * inv_tau * (cmax + 1) + 1) * U)
    return eps_z, (Kb + 8) * U, eps_n


def lse_bound(ref, D: int, Kb: int, nb: int = 1) -> torch.Tensor:
    """Per-row bound on |lse_kernel - lse| (nats); nb > 1: the lse of nb K blocks combined on the host."""
    eps_z, eps_sum, _ = _logit_error(ref, D, Kb)
    a = ref["lse"].abs() + 1
    b = SAFETY * (eps_z + eps_sum + 2.0 ** -21 + 6 * U * a)
    if nb > 1:
        b = b + (nb + 2) * 2 * U * a
    return b


def dx_bound(ref, D: int, Kb: int, store_points: Optional[torch.Tensor] = None, lse_given: bool = False,
             nb: int = 1) -> torch.Tensor:
    """Per-row bound on |dx_kernel - ref|_2 (module docstring).  Kb: candidate rows per launch (<= 256).
    store_points [M]: sum of |exact value| over the bf16 rounding points of the row's dX (default: |ref| once).
    lse_given: K-blocked rounds that take the row's lse from the first round."""
    eps_z, eps_sum, eps_n = _logit_error(ref, D, Kb)
    if lse_given:
        eps_z = eps_z + lse_bound(ref, D, Kb, nb) / SAFETY + 3 * U * (ref["lse"].abs() + 1)
    tn = ref["t"].norm(dim=1)
    rs, Gt, p, z = ref["rs"], ref["Gt"], ref["p"], ref["z"]
    alpha = (1 + BF) ** 3 - 1 + (Kb / 16 + 2) * 2.0 ** -23
    A = alpha * rs * (Gt.abs() * tn).sum(1)
    C = rs * (2 * eps_z + eps_sum) * (p * tn).sum(1)
    wrow = ref["wrow"].clamp_min(1e-300)
    Wn = ref["W"] / wrow[:, None]
    tgt = (ref["W"] > 0).double()
    B = rs * (eps_sum + 4 * U) * (tgt * (p + Wn) * tn).sum(1)
    K = p.shape[1]
    spz = (p * z.abs()).sum(1)
    swz = (Wn * z.abs()).sum(1)
    dcj = ref["coef"] * ((2 * eps_z + 2 * eps_sum + (K + 8 * nb) * U) * spz + 2 * eps_z + 4 * U * (spz + swz))
    P = ref["inv_n"] * ref["s"] * (dcj + ref["cj"].abs() * (2 * eps_n + 3 * U))
    F = (rs + 1) * K * 2.0 ** -120
    if store_points is None:
        store_points = ref["dx"].norm(dim=1)
    S = BF * (1 + 2.0 ** -6) * store_points
    return SAFETY * (A + B + C + P + F) + S


def store_points_kblocked(ref, in_kernel: bool) -> torch.Tensor:
    """sum over the bf16 rounding points of a K-blocked dX: in_kernel (<= 4 blocks added into one bf16 tensor): every
    partial sum; else every block's own dX (then added in fp32)."""
    blocks = ref["dx_blocks"]
    if in_kernel:
        return blocks.cumsum(0).norm(dim=2).sum(0)
    return blocks.norm(dim=2).sum(0)


def dcj_bound(ref, D: int, Kb: int, nb: int = 1, lse_given: bool = False) -> torch.Tensor:
    """Per-row bound on the error of cj (the row's share of -dlogtau)."""
    eps_z, eps_sum, eps_n = _logit_error(ref, D, Kb)
    if lse_given:
        eps_z = eps_z + lse_bound(ref, D, Kb, nb) / SAFETY + 3 * U * (ref["lse"].abs() + 1)
    p, z = ref["p"], ref["z"]
    K = p.shape[1]
    wrow = ref["wrow"].clamp_min(1e-300)
    spz = (p * z.abs()).sum(1)
    swz = (ref["W"] / wrow[:, None] * z.abs()).sum(1)
    return SAFETY * ref["coef"] * ((2 * eps_z + 2 * eps_sum + (K + 8 * nb) * U) * spz + 2 * eps_z + 4 * U * (spz + swz))


def sums_bounds(ref, D: int, Kb: int, n_acc: int, nb: int = 1, lse_given: bool = False):
    """(bound on |loss_sum_kernel - loss_sum|, bound on |dlogtau_kernel - dlogtau|): sums of the per-row bounds plus the
    fp32 running sums (n_acc = values a thread and its warp add before the float64 total)."""
    eps_z, _, _ = _logit_error(ref, D, Kb)
    dl = lse_bound(ref, D, Kb, nb)
    loss_b = (ref["wrow"] * dl * (nb if nb > 1 else 1) + ref["w"].sum(1) * SAFETY * eps_z).sum()
    loss_b = loss_b + (n_acc + 8) * U * (ref["wrow"] * ref["lse"].abs() + (ref["w"] * ref["z"].gather(1, ref["y"].clamp_min(0)).abs()).sum(1)).sum()
    dlt_b = dcj_bound(ref, D, Kb, nb, lse_given).sum() + (n_acc + 8) * U * ref["cj"].abs().sum()
    return float(loss_b), float(dlt_b)


def dt_bound(ref, D: int, Kb: int) -> torch.Tensor:
    """Per-text-row bound on |dText_kernel - ref|_2 (G stored in bf16 as for dX; the split-K GEMM over the M rows
    accumulates G^T x in fp32)."""
    eps_z, eps_sum, _ = _logit_error(ref, D, Kb)
    rs, Gt, p = ref["rs"][:, None], ref["Gt"], ref["p"]
    M = Gt.shape[0]
    xn = ref["x"].norm(dim=1)[:, None]
    wrow = ref["wrow"].clamp_min(1e-300)[:, None]
    tgt = (ref["W"] > 0).double()
    alpha = (1 + BF) ** 3 - 1
    dG = rs * (alpha * Gt.abs() + (2 * eps_z[:, None] + eps_sum) * p + tgt * (eps_sum + 4 * U) * (p + ref["W"] / wrow))
    acc = (M / 16 + 8) * 2.0 ** -23 * (rs * Gt.abs() * xn).sum(0)
    return SAFETY * ((dG * xn).sum(0) + acc) + 2.0 ** -20 * ref["dt"].norm(dim=1) + 1e-30


# ------------------------------------------------------------------------------------------------
# fp32 CUDA-core path (rc_infonce_f32): every step in fp32
# ------------------------------------------------------------------------------------------------
def dx_bound_f32(ref, D: int) -> torch.Tensor:
    """Per-row bound on the fp32 kernel's dX: 1e-5 of the row's gradient plus the fp32 logit error (dot products of D
    terms, the row norm, expf) carried through the softmax, and the projection term."""
    inv_tau = float(ref["inv_tau"])
    K = ref["p"].shape[1]
    cmax = ref["z"].abs().amax(1) / inv_tau
    eps_z = inv_tau * (D + 8) * U * (cmax + 1) + 4 * U * (ref["z"].abs().amax(1) + 1)
    tn = ref["t"].norm(dim=1)
    rs, Gt, p = ref["rs"], ref["Gt"], ref["p"]
    main = rs * ((2 * eps_z + (K + 8) * U) * (p * tn).sum(1) + (K + 8) * U * (Gt.abs() * tn).sum(1))
    spz = (p * ref["z"].abs()).sum(1)
    P = ref["inv_n"] * ref["s"] * ref["coef"] * (2 * eps_z + (K + 8) * U) * (spz + 2)
    return 1e-5 * ref["dx"].norm(dim=1) + SAFETY * (main + P) + 1e-30


def emulate_bf16(x: torch.Tensor, t: torch.Tensor, y: torch.Tensor, w: torch.Tensor, inv_tau: float, mutate: str = "",
                 gscale: float = 1.0) -> Dict[str, torch.Tensor]:
    """A torch restatement of one tensor-core launch (K <= 256) at the kernels' rounding points: S in fp32 from bf16
    operands, fp32 row norm, e = exp2(S zl - ml) rounded to bf16, fp32 sums, rsv rounded to bf16, non-target entries of G
    the bf16 product, target entries formed in fp32 and rounded once, the dX GEMM in fp32, the projection term, dX stored
    in bf16.  `mutate` builds the wrong variants the row-level bound must reject:
      'drop_w_hi'   the one-hot weight dropped on rows whose target lies in the second half of the columns;
      'round_y'     the target entry formed from the bf16-rounded e_y rsv and sum rsv W_k / wrow (cancels after rounding)."""
    bf = torch.bfloat16
    xb = x.to(bf).float()
    tb = t.to(bf).float()
    M, D = xb.shape
    K = tb.shape[0]
    Kp = (K + 63) // 64 * 64
    Kh = Kp // 2
    yy, ww, W = targets_and_weights(y, w, K)
    W32 = W.float()
    q = (xb * xb).sum(1)
    inv_n = 1.0 / torch.sqrt(q).clamp_min(1e-12)
    S = xb @ tb.T                                                     # fp32
    log2e = 1.4426950408889634
    zs = inv_n * inv_tau
    zl = zs * log2e
    use_bound = inv_tau * (2.02 * log2e) < 100.0
    ml = torch.full((M,), inv_tau * 1.01 * log2e) if use_bound else S.amax(1) * zl
    e = torch.exp2(torch.addcmul(-ml[:, None], S, zl[:, None]))
    e16 = e.to(bf).float()
    s = e.sum(1)
    sez = (e * S).sum(1)
    wrow = W32.sum(1)
    wsum = float(ww.sum())
    tz = (ww.float() * S.gather(1, yy.clamp_min(0))).sum(1)
    coefb = gscale / wsum if wsum > 0 else 0.0
    coef = coefb * wrow
    inv_sum = 1.0 / s
    rsv = inv_n * inv_tau * coef * inv_sum
    rsv16 = rsv.to(bf).float()
    G = (e16 * rsv16[:, None]).to(bf).float()
    frac = torch.where(wrow[:, None] > 0, W32 / wrow.clamp_min(1e-30)[:, None], torch.zeros_like(W32))
    tgt = W32 > 0
    gy = ((e - s[:, None] * frac) * rsv[:, None]).to(bf).float()
    if mutate == "drop_w_hi":
        hi = torch.arange(K)[None, :] >= Kh
        gy = torch.where(hi, (e * rsv[:, None]).to(bf).float(), gy)
    if mutate == "round_y":
        gy = (e * rsv[:, None]).to(bf).float() - (s[:, None] * rsv[:, None] * frac).to(bf).float()
    G = torch.where(tgt, gy, G)
    cj = coef * sez * zs * inv_sum - coefb * tz * zs
    dx = (G @ tb) - (inv_n * inv_n * cj)[:, None] * xb
    dx = dx.to(bf).float()
    lse = (ml + torch.log2(s)) / log2e
    loss = wrow * lse - tz * zs
    return dict(dx=dx, lse=lse, loss_sum=loss.double().sum(), dlogtau=-cj.double().sum(), wsum=wsum)


def global_checks_accept(dx, lse, loss_sum, wsum, ref) -> bool:
    """The suite's aggregate checks: max-relative dX < 2e-2 of the tensor's largest |dX|, lse within 2e-3 of the largest
    lse, the mean loss within 2e-3."""
    dxr = float((dx.double() - ref["dx"]).abs().max() / ref["dx"].abs().max().clamp_min(1e-30))
    lr = float((lse.double() - ref["lse"]).abs().max() / ref["lse"].abs().max().clamp_min(1e-30))
    ws = float(ref["wsum"])
    lossr = abs(float(loss_sum) / ws - float(ref["loss_sum"]) / ws) / max(abs(float(ref["loss_sum"]) / ws), 1e-30)
    return dxr < 2e-2 and lr < 2e-3 and lossr < 2e-3


# ------------------------------------------------------------------------------------------------
# inputs built to hit the kernels' known failure modes
# ------------------------------------------------------------------------------------------------
def make_case(B: int, D: int, HW: int, K: int, R: int, seed: int):
    """(x [B, D, HW] bf16-exact float32, t [K, D] normalised bf16-exact, y / w [B * HW] (R = 1) or [B * HW, 4]).
    Random rows (10 % ignored targets, weights 0..3) with special rows at the start of the first image and at the end of
    the last one (the partial last tile): targets at Kh - 1, Kh, K - 1 and in the 16-column step that straddles K
    (Kh = half of K rounded up to 64); confident rows (x along its target: p_y > 1 - 1e-6 at tau <= 0.02) in both
    column halves; a near-uniform row (x orthogonal to every candidate, when K < D); a row of weight 0 next to a row of
    weight 3; an ignored target with a weight; a row of norm 1e-20 (clamped by F.normalize's eps) and one of norm 1e-11
    (just above it).  R = 4: duplicate targets, targets spread over both halves, ignored targets among weighted ones."""
    g = torch.Generator().manual_seed(seed)
    bf = torch.bfloat16
    M = B * HW
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g, dtype=torch.float64), dim=1).to(bf).double()
    x = torch.randn(M, D, generator=g, dtype=torch.float64) * (0.5 + torch.rand(M, 1, generator=g, dtype=torch.float64))
    Kh = (K + 63) // 64 * 32
    kst = (K // 16) * 16 if K % 16 else K - 16            # first column of the step that straddles K (or the last step)
    kst = min(kst + (K - kst) // 2, K - 1)
    y = torch.randint(0, K, (M, R), generator=g, dtype=torch.int64)
    w = torch.randint(0, 4, (M, R), generator=g).double()
    y[torch.rand(M, R, generator=g) < 0.1] = -1
    if R == 4:                                             # mostly one label per block, as in a segmentation
        same = torch.rand(M, generator=g) < 0.6
        y[same] = y[same][:, :1].expand(-1, 4)
    # a third of the rows leans towards its (first) target by a random amount: every confidence from p_y ~ 1 / K to ~ 1,
    # where the target entry's cancellation (e_y - sum) matters most
    lean = (torch.rand(M, generator=g) < 0.35) & (y[:, 0] >= 0)
    a = 4.0 * torch.rand(M, 1, generator=g, dtype=torch.float64) * x.norm(dim=1, keepdim=True) / math.sqrt(D)
    x = torch.where(lean[:, None], x / math.sqrt(D) + a * t[y[:, 0].clamp_min(0)], x)

    def along(k, scale=2.0):
        return t[k] * scale + 0.01 * torch.randn(D, generator=g, dtype=torch.float64) / math.sqrt(D)

    specials = []                                          # (x row or None, targets, weights)
    ylist = [Kh - 1, Kh, K - 1, kst]
    for k in ylist:
        specials.append((None, [k] * R if R == 1 else [k, (k + 1) % K, k, -1], [2.0] * R))
    specials.append((along(K - 2), [K - 2] * R, [1.0] * R))                       # confident, second half
    specials.append((along(1), [1] * R, [3.0] * R))                                # confident, first half
    if K < D:
        q, _ = torch.linalg.qr(t.T)                       # [D, K] orthonormal basis of the candidates' span
        v = torch.randn(D, generator=g, dtype=torch.float64)
        v = v - q @ (q.T @ v)
        specials.append((v / v.norm() * 1.5, [3] * R, [1.0] * R))                  # near-uniform softmax
    specials.append((None, [5] * R, [0.0] * R))                                    # zero weight ...
    specials.append((None, [6] * R, [3.0] * R))                                    # ... next to weight 3
    specials.append((None, [-1] * R, [2.0] * R))                                   # ignored target with a weight
    v = torch.randn(D, generator=g, dtype=torch.float64)
    specials.append((v / v.norm() * 1e-20, [2] * R, [1.0] * R))                    # clamped norm
    specials.append((v / v.norm() * 1e-11, [K - 1] * R, [1.0] * R))                # just above the eps
    specials.append((along(0, 1.0), [0] * R, [1.0] * R))
    if R == 4:
        specials.append((None, [Kh - 1, Kh, K - 1, 0], [1.0, 2.0, 3.0, 1.0]))     # both halves
        specials.append((along(K - 1), [K - 1, 4, K - 1, K - 1], [1.0, 2.0, 1.0, 2.0]))   # duplicates, confident
        specials.append((None, [-1, Kh, -1, Kh - 1], [3.0, 1.0, 2.0, 1.0]))       # ignored among weighted
    n = len(specials)
    rows = list(range(n)) + list(range(M - n, M))
    for i, r in enumerate(rows):
        xr, yr, wr = specials[i % n]
        if xr is not None:
            x[r] = xr
        y[r] = torch.tensor(yr)
        w[r] = torch.tensor(wr)
    x = x.to(bf).double()
    x = x.view(B, HW, D).permute(0, 2, 1).contiguous()
    if R == 1:
        y, w = y[:, 0], w[:, 0]
    return x.float(), t.float(), y.int(), w.float()


def make_overflow_case(B: int, D: int, HW: int, K: int, R: int, seed: int):
    """K-blocked rows whose lse exceeds the largest logit of their target's block by ~2 / tau: candidate rows 256..K-1
    point away from x (cosine ~ -0.95), row 5 of block 0 along x, every target in block 1.  Below the tau switch a block
    offset by its own maximum would need exp(lse - max) ~ exp(195) at tau = 0.01 (exp(97) at tau = 0.02): beyond fp32."""
    g = torch.Generator().manual_seed(seed)
    bf = torch.bfloat16
    M = B * HW
    u = torch.nn.functional.normalize(torch.randn(D, generator=g, dtype=torch.float64), dim=0)
    t = torch.randn(K, D, generator=g, dtype=torch.float64)
    t[5] = u
    t[256:] = -u + 0.3 * torch.randn(K - 256, D, generator=g, dtype=torch.float64) / math.sqrt(D)
    t = torch.nn.functional.normalize(t, dim=1).to(bf).double()
    x = u + 0.05 * torch.randn(M, D, generator=g, dtype=torch.float64) / math.sqrt(D)
    plain = torch.rand(M, generator=g) < 0.25                      # a quarter of the rows ordinary
    x[plain] = torch.randn(int(plain.sum()), D, generator=g, dtype=torch.float64)
    x = x.to(bf).double()
    y = torch.randint(256, K, (M, R), generator=g, dtype=torch.int64)
    if R == 4:
        y[:, 2] = y[:, 0]                                          # duplicates
    w = torch.randint(1, 4, (M, R), generator=g).double()
    x = x.view(B, HW, D).permute(0, 2, 1).contiguous()
    if R == 1:
        y, w = y[:, 0], w[:, 0]
    return x.float(), t.float(), y.int(), w.float()
