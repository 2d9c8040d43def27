"""Inputs with exact logits, and the exact ranking, for the evaluation top-k kernels (K7: eval_topk_umma.cu, and the fp32
top-k of infonce_simt.cu).

TEST INFRASTRUCTURE ONLY (tests/test_gpu_exact_topk.py, tests/test_exact_topk_cpu.py); nothing under ``rangeclip_b200/``
imports it.

A top-k only compares.  Once every logit is exact, the whole output is fixed to the last id by the stated contract: rank
by logit, ties to the smaller text index, and -1 past a device row count.  The builders below make every logit exact in
any summation order, on the tensor cores as on the CUDA cores:

* every x and t entry is a / 8 with |a| <= 64 in the core channels (filler channels: |a| <= 256), so bf16 holds it and
  every product is a multiple of 2^-6;
* for every (pixel, text row) pair, sum_d |x_d t_d| stays below 2^14 units of 2^-6 (``SPAN_UNITS``), so every partial sum
  in any order is exact in fp32, with room left for the tensor cores' internal alignment;
* every pixel row has a power-of-two norm, and every non-zero text row the same power-of-two norm, by filler channels:
  ``X_FILL`` channels that are zero in every text row, and ``T_FILL`` channels that are zero in every pixel row.  The logits
  do not change; the normalisations of the fp32 kernel, of the bf16 pre-pass and of ``text_prepare`` multiply by exact
  powers of two, and ties stay ties.

Ties are built, not hoped for.  Pixel rows are constant on groups of four channels; a text row's group holds a random
split of the group's sum, so equal logits come from different bits.  Each pixel belongs to one of four classes, and each
class reads one selector group of the text rows, so four independent arrangements run in every launch:

* class 0, ``seams``: one unique winner, then a tie group at the columns where the scan changes code path -- the first
  32-column chunk (static insertion), a later chunk of the same thread, a column c and c + 128 (the two scan threads of a
  pixel), a later 256-row block, the partial last chunk, K - 1 and Kv - 1 -- then near-ties 2^-6 below;
* class 1, ``boundary``: k - 1 strictly ordered rows, then a tie group larger than the one rank left, then near-ties;
* class 2, ``partner``: k + 2 tied rows in the first chunk of the second scan thread (columns 128..) and as many with
  SMALLER indices in a later chunk of the first (columns 64..): the first thread's candidate filter then runs against the
  partner's k-th best equal to its own candidates (the next-lower-float bound), and the smaller indices must win;
* class 3: zero pixel rows; every logit is 0 and the answer is the first k indices in order.

``sign`` shifts the same arrangement: "neg" makes every logit negative (x >= 0, t <= 0), so the zero pad rows of the bf16
text copy, the zero fill past it and any unmasked column would beat every real row; "nonpos" (x <= 0, t >= 0) puts class
2's tie at exactly 0, with half of its rows all-zero (-0 against +0 logits, the partner bound 0).
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np

from oracle.exact_inputs import fits  # noqa: F401  (re-exported for the tests)

X_FILL = 8            # channels zero in every text row: make |x|^2 a power of 4
T_FILL = 8            # channels zero in every pixel row: make every non-zero |t|^2 the same power of 4
N_CLS = 4             # pixel classes = selector groups
GROUP = 4             # channels per group (pixel rows are constant on a group)
SPAN_UNITS = 2 ** 14  # bound on sum_d |x_d t_d| in units of 2^-6
L_TOP = 24            # level (group sum in eighths) of the planted rows; background levels are in [-4, 4]
MAX_NOISE = 32        # noise channels (random +-1/8 in background rows)
CORE_MIN = 2 * N_CLS * GROUP


# ----------------------------------------------------------------------------------------------------------------------
# building blocks
# ----------------------------------------------------------------------------------------------------------------------

def split_sum(rng: np.random.Generator, L: int, n: int = GROUP, cap: int = 64) -> np.ndarray:
    """n integers in [-cap, cap] summing to L, in a random split (equal sums, different contents)."""
    a = np.full(n, L // n, np.int64)
    a[: L % n] += 1
    for _ in range(2 * n):
        i, j = rng.choice(n, 2, replace=False)
        d = int(rng.integers(0, 6))
        if abs(a[i] + d) <= cap and abs(a[j] - d) <= cap:
            a[i] += d
            a[j] -= d
    assert a.sum() == L and np.abs(a).max() <= cap
    return a


def four_squares(r: int):
    """Four non-negative integers whose squares sum to r (Lagrange), smallest search first."""
    for a in range(math.isqrt(r), -1, -1):
        for b in range(min(a, math.isqrt(r - a * a)), -1, -1):
            for c in range(min(b, math.isqrt(r - a * a - b * b)), -1, -1):
                d2 = r - a * a - b * b - c * c
                d = math.isqrt(d2)
                if d * d == d2 and d <= c:
                    return [a, b, c, d]
    raise AssertionError(r)


def _pow4_at_least(S: int) -> int:
    t = 1
    while t < S:
        t *= 4
    return t


def filler(S: int, n: int, target: Optional[int] = None) -> np.ndarray:
    """n integers in [0, 256] with S + sum of squares = ``target`` (default: the smallest power of 4 >= max(S, 1)):
    greedy squares capped at 256^2, then a four-square decomposition of the rest."""
    if target is None:
        target = _pow4_at_least(S)
    r = target - S
    assert r >= 0
    f = []
    while r > 1024:
        a = min(256, math.isqrt(r))
        f.append(a)
        r -= a * a
    f += four_squares(r)
    assert len(f) <= n, (S, target, f)
    return np.array(f + [0] * (n - len(f)), np.int64)


# ----------------------------------------------------------------------------------------------------------------------
# the case builder
# ----------------------------------------------------------------------------------------------------------------------

def seam_columns(K: int, Kv: int):
    """The scan seams of a row count: first chunk, later chunk, c / c + 128, later block, partial last chunk, K-1, Kv-1."""
    cols = [3, 40, 131, 168, 259, 300, 389, 520, (Kv // 32) * 32 + 1, Kv - 2, Kv - 1, K - 1]
    return sorted({c for c in cols if 0 <= c < Kv})


def topk_case(D: int, K: int, B: int, HW: int, k: int, seed: int, Kv: Optional[int] = None, sign: str = "mixed",
              pads: str = "winner") -> Dict[str, object]:
    """x [B, D, HW] and t [K, D] float64 (exact in bf16), with the arrangement of the module docstring.

    ``Kv`` (default K): rows past it are device-count pads: 2x copies of class 0's winner (``pads="winner"``; they would
    win every class-0 pixel if scanned) or zero rows (``pads="zero"``).  Returns a dict with x, t, k, Kv, cls (pixel class
    [B*HW]), the planted row sets and the channel layout."""
    assert sign in ("mixed", "neg", "nonpos") and D - X_FILL - T_FILL >= CORE_MIN, (sign, D)
    Kv = K if Kv is None else Kv
    assert 1 <= Kv <= K
    rng = np.random.default_rng(seed)
    n = min(k, Kv)
    core = D - X_FILL - T_FILL
    g_sel = [list(range(GROUP * c, GROUP * c + GROUP)) for c in range(N_CLS)]
    g_off = [list(range(GROUP * (N_CLS + c), GROUP * (N_CLS + c) + GROUP)) for c in range(N_CLS)]
    noise_ch = list(range(CORE_MIN, CORE_MIN + min(MAX_NOISE, core - CORE_MIN)))
    xf_ch = list(range(core, core + X_FILL))
    tf_ch = list(range(core + X_FILL, D))

    # ---- planted (level, offset) per class; everything else background ----
    # class c reads selector group c (x = s / 8) and offset group c (x = 1 / 8): one offset unit is 2^-6 of logit
    lev = rng.integers(-4, 5, size=(K, N_CLS))
    off = rng.integers(-8, 9, size=(K, N_CLS))
    planted = np.zeros(K, bool)

    def plant(c, rows_off):
        for j, o in rows_off:
            lev[j, c], off[j, c] = L_TOP, o
            planted[j] = True

    # class 0: unique winner, the tie group at the seams, near-ties right after them
    seams = seam_columns(K, Kv)
    free = [j for j in range(Kv) if j not in seams]
    win0 = int(rng.choice(free)) if free else seams[0]
    tie0 = [j for j in seams if j != win0]
    near0 = sorted({j + 1 for j in seams if j + 1 < Kv and j + 1 not in seams and j + 1 != win0})
    plant(0, [(win0, 20)] + [(j, 19) for j in tie0] + [(j, 18) for j in near0])
    # class 1: n - 1 strictly ordered rows, then a tie group of n + 2 rows for the one rank left, then near-ties
    perm = rng.permutation(Kv)
    strict = [int(j) for j in perm[:n - 1]]
    tie1 = sorted(int(j) for j in perm[n - 1:2 * n + 1])
    near1 = sorted(int(j) for j in perm[2 * n + 1:2 * n + 3])
    plant(1, [(j, 20 - i) for i, j in enumerate(strict)] + [(j, 13) for j in tie1] + [(j, 12) for j in near1])
    # class 2: k + 2 tied rows at 128.. (first chunk of the second scan thread), k + 2 at 64.. (later chunk of the first)
    hi = [j for j in range(128, 130 + k) if j < Kv]
    lo = [j for j in range(64, 66 + k) if j < Kv]
    plant(2, [(j, 20) for j in hi + lo])
    plants = dict(win0=win0, tie0=tie0, near0=near0, strict1=strict, tie1=tie1, near1=near1, hi2=hi, lo2=lo)
    # ---- sign transforms: the order of (level, offset) within a class is kept ----
    zero_rows = np.zeros(K, bool)
    if sign == "neg":
        lev, off = lev - (L_TOP + 1), off - 21
    elif sign == "nonpos":
        lev, off = L_TOP - lev, 20 - off       # >= 0; class 2's tie -> exactly 0
        zero_rows[hi] = True                   # all-zero rows (what a -1 entry of a device-built list becomes)
    # ---- text rows ----
    t = np.zeros((K, D), np.float64)
    for j in range(K):
        if zero_rows[j]:
            continue
        for c in range(N_CLS):
            t[j, g_sel[c]] = split_sum(rng, int(lev[j, c])) / 8
            t[j, g_off[c]] = split_sum(rng, int(off[j, c])) / 8
        if not planted[j] and noise_ch:
            lo_n, hi_n = {"mixed": (-1, 1), "neg": (-1, 0), "nonpos": (0, 1)}[sign]
            t[j, noise_ch] = rng.integers(lo_n, hi_n + 1, size=len(noise_ch)) / 8
    if Kv < K:                          # device-count pads
        if pads == "winner":
            t[Kv:] = 2 * t[win0]
        else:
            t[Kv:] = 0
    # common power-of-two norm for the non-zero rows
    S = np.rint((t[:, :core] * 8) ** 2).astype(np.int64).sum(1)
    nz = S > 0
    if nz.any():
        target = _pow4_at_least(int(S[nz].max()))
        for j in np.nonzero(nz)[0]:
            t[j, tf_ch] = filler(int(S[j]), T_FILL, target) / 8
            if sign == "neg":
                t[j, tf_ch] = -t[j, tf_ch]
    # ---- pixel rows ----
    P = B * HW
    cls = rng.integers(0, N_CLS, size=P)
    cls[: N_CLS] = np.arange(N_CLS)
    x = np.zeros((P, D), np.float64)
    sgn = -1.0 if sign == "nonpos" else 1.0
    s = rng.integers(4, 9, size=P)
    for p in range(P):
        c = int(cls[p])
        if c == 3:
            continue
        x[p, g_sel[c]] = sgn * s[p] / 8
        x[p, g_off[c]] = sgn / 8
        if noise_ch:
            lo_n, hi_n = {"mixed": (-1, 1), "neg": (0, 1), "nonpos": (-1, 0)}[sign]
            x[p, noise_ch] = rng.integers(lo_n, hi_n + 1, size=len(noise_ch)) / 8
    if sign == "nonpos":               # -0 in the unused channels of odd pixels: -0 and +0 products both occur
        odd = (np.arange(P) % 2 == 1)[:, None]
        x = np.where((x == 0) & odd, -0.0, x)
    Sx = np.rint((x[:, :core] * 8) ** 2).astype(np.int64).sum(1)
    for p in range(P):
        x[p, xf_ch] = sgn * filler(int(Sx[p]), X_FILL) / 8
    x = x.reshape(B, HW, D).transpose(0, 2, 1).copy()
    return dict(x=x, t=t, k=k, K=K, Kv=Kv, B=B, HW=HW, D=D, cls=cls, sign=sign, zero_rows=np.nonzero(zero_rows)[0].tolist(),
                core=core, xf_ch=xf_ch, tf_ch=tf_ch, planted=np.nonzero(planted)[0].tolist(), **plants)


# ----------------------------------------------------------------------------------------------------------------------
# references
# ----------------------------------------------------------------------------------------------------------------------

def logits(x: np.ndarray, t: np.ndarray) -> np.ndarray:
    """[B, K, HW] float64 raw dot products (exact for the builders' inputs)."""
    return np.einsum("bdn,kd->bkn", x, t)


def rank_ids(lg: np.ndarray, k: int, Kv: Optional[int] = None, index_map=None) -> np.ndarray:
    """The contract of every top-k kernel: [B, k, HW] int64, rank j = the j-th best of rows [0, Kv) by logit, ties to the
    smaller index (a stable sort of -logit), mapped through ``index_map``; ranks >= Kv are -1."""
    B, K, HW = lg.shape
    Kv = K if Kv is None else Kv
    order = np.argsort(-lg[:, :Kv, :], axis=1, kind="stable")
    n = min(k, Kv)
    out = np.full((B, k, HW), -1, np.int64)
    ids = order[:, :n, :]
    out[:, :n, :] = ids if index_map is None else np.asarray(index_map, np.int64)[ids]
    return out


def normalized_logits(x: np.ndarray, t: np.ndarray) -> np.ndarray:
    """Cosine logits (exact when the norms are powers of two); zero rows stay zero."""
    nx = np.sqrt((x * x).sum(1, keepdims=True))
    nt = np.sqrt((t * t).sum(1, keepdims=True))
    return logits(x / np.maximum(nx, 1e-12), t / np.maximum(nt, 1e-12))


def upsample2(a: np.ndarray, h: int, w: int) -> np.ndarray:
    """[B, k, h*w] -> [B, k, 2h, 2w] nearest x2 (the four pixels of row (i, j) are (2i + a, 2j + b))."""
    B, k = a.shape[:2]
    return a.reshape(B, k, h, w).repeat(2, axis=2).repeat(2, axis=3)


def expected_hist(gt: np.ndarray, ids: np.ndarray, E: np.ndarray, cmap: np.ndarray):
    """The five per-batch class histograms [5, C] and three counters the fused kernels add, from the expected ids
    [N, k] (column 0 = top-1; -1 = no prediction at that rank).  Rows: count of gt class, of top-1 class, of gt class
    where they agree, of the 'oracle' prediction (the gt class if any rank hits it, else the raw top-1 id), of gt class
    where that agrees; counters: E[gt, top1], any_j E[gt, id_j], pixels counted."""
    gt = np.asarray(gt, np.int64).reshape(-1)
    ids = np.asarray(ids, np.int64).reshape(len(gt), -1)
    C = len(cmap)
    t1 = ids[:, 0]
    ok = (gt >= 0) & (gt < C) & (t1 >= 0) & (t1 < C)
    g, ids = gt[ok], ids[ok]
    t1 = ids[:, 0]
    valid = (ids >= 0) & (ids < C)
    safe = np.where(valid, ids, 0)
    ge, p1 = cmap[g], cmap[t1]
    any_eqk = (E[g[:, None], safe].astype(bool) & valid).any(1)
    hit = ((cmap[safe] == ge[:, None]) & valid).any(1)
    orc = np.where(hit, ge, t1)
    bc = lambda v: np.bincount(v, minlength=C).astype(np.int64)
    hist = np.stack([bc(ge), bc(p1), bc(ge[p1 == ge]), bc(orc), bc(ge[orc == ge])])
    counters = np.array([int(E[g, t1].astype(bool).sum()), int(any_eqk.sum()), int(ok.sum())], np.int64)
    return hist, counters


def fold_hist(hist: np.ndarray):
    """The four accumulators of validate.py:110-139 from one batch's histograms (as rc_eval_fold forms them): label ->
    (I1, U1, IK, UK) for the labels of unique(gt class U top-1 class)."""
    ge, p1, i1, orc, ik = hist
    return {int(L): (int(i1[L]), int(ge[L] + p1[L] - i1[L]), int(ik[L]), int(ge[L] + orc[L] - ik[L]))
            for L in np.nonzero(ge + p1 > 0)[0]}


def metric_problem(rng: np.random.Generator, C: int, n: int):
    """gt [n] in [0, C), an equivalence matrix with a non-transitive chain (validate.py's Q9 quirk) and its class map."""
    from oracle import rangeclip_oracle as O
    eq = {i: {i} for i in range(C)}
    chain = rng.permutation(C)[: max(2, C // 4)]
    for a, b in zip(chain[:-1], chain[1:]):
        eq[int(a)].add(int(b))
        eq[int(b)].add(int(a))
    E = O.build_equivalence_tensor(eq, C)
    cmap = O.build_equivalence_class_map(E)
    gt = rng.integers(0, C, size=n)
    return gt, E, cmap
