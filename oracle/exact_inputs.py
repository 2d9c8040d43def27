"""Inputs with exactly representable results, and float64 references, for the memory-bound kernels: masked pooling, the
smoothness (TV-L1) forward / backward and its fp32 sign codes, row normalisation and the sampling helpers.

TEST INFRASTRUCTURE ONLY (tests/test_gpu_exact_memory_bound.py, tests/test_exact_inputs_cpu.py); nothing under
``rangeclip_b200/`` imports it.

These kernels do integer-like work on floating-point data: sums of masked pixels, counts, signs of differences, row norms
that are powers of two.  The builders choose values on a coarse dyadic grid (k / 8, power-of-two scales and counts) so
that every partial result a kernel can form -- in any summation order -- is exact in fp32 (and, where the kernel stores
it so, in bf16).  A correct kernel then matches the float64 reference bit for bit at every element; a kernel that drops a
pixel, reads the wrong neighbour or mis-signs a difference cannot hide behind a tolerance.  ``fits`` states the premise;
tests/test_exact_inputs_cpu.py checks it for every builder without a GPU.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch

F32_ONE_OVER_EPS = np.float32(1.0) / np.float32(1e-12)      # 1 / max(|x|, 1e-12) of a zero row, as the kernels form it


def fits(v, dtype: torch.dtype) -> bool:
    """Whether every element of the float64 array ``v`` is exactly representable in ``dtype`` (fp32 or bf16)."""
    t = torch.as_tensor(np.ascontiguousarray(v, dtype=np.float64))
    return bool(torch.equal(t.to(dtype).double(), t))


def dyadic(rng: np.random.Generator, shape, m: int = 16, den: int = 8) -> np.ndarray:
    """float64 values k / den with k uniform in [-m, m] (exact in bf16 for m <= 256)."""
    return rng.integers(-m, m + 1, size=shape).astype(np.float64) / den


# ----------------------------------------------------------------------------------------------------------------------
# masked pooling
# ----------------------------------------------------------------------------------------------------------------------

def seg_runs(rng: np.random.Generator, n: int, C: int) -> np.ndarray:
    """Labels along a flattened image in runs whose lengths mix cuts inside an 8-pixel group (1..7), whole groups and
    long runs; labels drawn from [-2, C + 2), so negative labels and labels >= C occur."""
    out = np.empty(n, np.int64)
    p = 0
    while p < n:
        kind = int(rng.integers(0, 4))
        L = int([rng.integers(1, 8), 8 * rng.integers(1, 4), rng.integers(9, 64), rng.integers(64, 300)][kind])
        out[p:p + L] = rng.integers(-2, C + 2)
        p += L
    return out


def pool_segmentation(rng: np.random.Generator, B: int, H: int, W: int, C: int) -> np.ndarray:
    """int64 [B, H*W].  On top of ``seg_runs``: one label in two runs of the first warp's 256 pixels separated by another
    label; runs across the 256-pixel chunk boundary and the 512-pixel chunk-pair boundary; and, at W = 256 (a chunk is one
    image row), every other chunk pair made of two identical rows, so that pairs merge and pairs do not."""
    HW = H * W
    seg = np.stack([seg_runs(rng, HW, C) for _ in range(B)])
    for b in range(B):
        a, c = rng.choice(C, size=2, replace=False)
        n0 = min(HW, 256)
        seg[b, :n0] = a
        seg[b, 64:min(HW, 128)] = c
        for lo, hi in ((250, 262), (500, 530)):
            if hi <= HW:
                seg[b, lo:hi] = rng.integers(0, C)
        if W == 256:
            for pair in range(1, H // 2, 2):
                seg[b, (2 * pair + 1) * W:(2 * pair + 2) * W] = seg[b, 2 * pair * W:(2 * pair + 1) * W]
    return seg


def pool_lut(rng: np.random.Generator, B: int, C: int, n_slots: int, per_image: bool) -> np.ndarray:
    """int32 [B, C] (per image) or [C] (batch-wide): a slot in [0, n_slots - 1) or -1; slot n_slots - 1 is never mapped,
    so its count is 0 and its mean row is zero."""
    shape = (B, C) if per_image else (C,)
    lut = rng.integers(0, n_slots - 1, size=shape).astype(np.int32)
    lut[rng.random(shape) < 0.2] = -1
    return lut


def pool_slots(seg: np.ndarray, lut: np.ndarray, per_image: bool) -> np.ndarray:
    """Slot of every pixel, [B, HW] (-1: label outside [0, C) or mapped to -1)."""
    C = lut.shape[-1]
    valid = (seg >= 0) & (seg < C)
    lab = np.where(valid, seg, 0)
    slot = np.take_along_axis(lut, lab, axis=1) if per_image else lut[lab]
    return np.where(valid, slot, -1)


def pool_reference(x: np.ndarray, segs: Sequence[np.ndarray], lut: np.ndarray, per_image: bool, n_slots: int):
    """x float64 [B, D, HW]: (sums float64 [n_slots, D], counts int64 [n_slots], mean float32 [n_slots, D]); every label map
    adds into the same sums and counts, and the mean is the fp32 quotient of the fp32 sum and count (0 for count 0)."""
    B, D, HW = x.shape
    sums = np.zeros((n_slots, D))
    cnt = np.zeros(n_slots, np.int64)
    for seg in segs:
        slots = pool_slots(seg, lut, per_image)
        for b in range(B):
            m = slots[b] >= 0
            onehot = np.zeros((int(m.sum()), n_slots))
            onehot[np.arange(onehot.shape[0]), slots[b][m]] = 1.0
            sums += (x[b][:, m] @ onehot).T
            cnt += np.bincount(slots[b][m], minlength=n_slots)
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = np.where(cnt[:, None] > 0, sums.astype(np.float32) / cnt.astype(np.float32)[:, None], np.float32(0))
    return sums, cnt, mean.astype(np.float32)


def pool_backward_reference(g: np.ndarray, cnt: np.ndarray, segs: Sequence[np.ndarray], lut: np.ndarray, per_image: bool,
                            D: int) -> List[np.ndarray]:
    """dx after each label map, float64 [B, D, HW]: map i adds g[slot] / cnt[slot] at every pixel with a slot of non-zero
    count.  The last entry is the gradient; the earlier ones are what the kernel stores between passes."""
    out, acc = [], None
    for seg in segs:
        slots = pool_slots(seg, lut, per_image)
        B, HW = slots.shape
        safe = np.maximum(cnt, 1).astype(np.float64)
        rows = np.where((cnt > 0)[:, None], g / safe[:, None], 0.0)
        d = np.where((slots >= 0)[:, None, :], rows[np.maximum(slots, 0)].transpose(0, 2, 1), 0.0)
        acc = d if acc is None else acc + d
        out.append(acc.copy())
    return out


def pool_backward_inputs(rng: np.random.Generator, n_slots: int, D: int, n_maps: int):
    """(g float64 [n_slots, D], cnt int64 [n_slots]) with power-of-two counts, so that g / cnt and its sums over the label
    maps are exact: one map m / 8 with |m| <= 16 and counts up to 2^10; four maps (accumulated in the output dtype
    between passes, bf16 included) |m| <= 4 and counts up to 8 -- every partial sum a multiple of 2^-6 below 2."""
    if n_maps == 1:
        return dyadic(rng, (n_slots, D), 16), 2 ** rng.integers(0, 11, size=n_slots)
    return dyadic(rng, (n_slots, D), 4), 2 ** rng.integers(0, 4, size=n_slots)


# ----------------------------------------------------------------------------------------------------------------------
# smoothness (TV-L1)
# ----------------------------------------------------------------------------------------------------------------------

def tv_input(rng: np.random.Generator, B: int, D: int, H: int, W: int) -> np.ndarray:
    """float64 [B, D, H, W] of k / 8, |k| <= 16, with many exactly equal neighbours; plane p is by p % 4: runs along the
    rows with repeated rows, a nearest-x2 upsampled map, a constant plane, independent values."""
    x = np.empty((B * D, H, W))
    for p in range(B * D):
        kind = p % 4
        if kind == 0:
            plane = np.repeat(dyadic(rng, (H, 1)), W, axis=1)
            for h in range(H):
                cuts = np.sort(rng.integers(0, W, size=3))
                for c in cuts:
                    plane[h, c:] = dyadic(rng, ())
            dup = rng.random(H) < 0.3
            for h in range(1, H):
                if dup[h]:
                    plane[h] = plane[h - 1]
        elif kind == 1:
            lo = dyadic(rng, ((H + 1) // 2, (W + 1) // 2))
            plane = np.repeat(np.repeat(lo, 2, axis=0), 2, axis=1)[:H, :W]
        elif kind == 2:
            plane = np.full((H, W), dyadic(rng, ()))
        else:
            plane = dyadic(rng, (H, W))
        x[p] = plane
    return x.reshape(B, D, H, W)


def tv_sums_reference(x: np.ndarray) -> np.ndarray:
    """float64 [2]: sum |x[.., w] - x[.., w+1]|, sum |x[.., h, :] - x[.., h+1, :]| (0 for an empty slice)."""
    x = np.asarray(x, np.float64)
    return np.array([np.abs(np.diff(x, axis=-1)).sum(), np.abs(np.diff(x, axis=-2)).sum()])


def tv_grad_reference(x: np.ndarray, sh: float, sv: float, dx_in: Optional[np.ndarray] = None, ds: float = 1.0) -> np.ndarray:
    """Closed form of ds * dx_in + sh d(sum_h)/dx + sv d(sum_v)/dx with sign(0) = 0, float64 (oracle smoothness_grad
    with a scale pair and an accumulated gradient)."""
    x = np.asarray(x, np.float64)
    g = np.zeros_like(x)
    s = np.sign(x[..., :, :-1] - x[..., :, 1:]) * sh
    g[..., :, :-1] += s
    g[..., :, 1:] -= s
    s = np.sign(x[..., :-1, :] - x[..., 1:, :]) * sv
    g[..., :-1, :] += s
    g[..., 1:, :] -= s
    if dx_in is not None:
        g = g + ds * np.asarray(dx_in, np.float64)
    return g


def tv_codes_reference(x32: np.ndarray) -> np.ndarray:
    """int32 [B, D, H, W/8] sign words of an fp32 x (W % 8 == 0): pixel j of a group at bits 4j..4j+3, bits 4j..4j+1 =
    sgn(x[h][w] - x[h][w+1]) + 1, bits 4j+2..4j+3 = sgn(x[h][w] - x[h+1][w]) + 1, the sign taken on the fp32 values and
    1 (no difference) past the last column / row."""
    x = np.asarray(x32, np.float32).astype(np.float64)
    ch = np.ones(x.shape, np.int64)
    cv = np.ones(x.shape, np.int64)
    ch[..., :, :-1] = np.sign(x[..., :, :-1] - x[..., :, 1:]).astype(np.int64) + 1
    cv[..., :-1, :] = np.sign(x[..., :-1, :] - x[..., 1:, :]).astype(np.int64) + 1
    nib = (ch | (cv << 2)).reshape(x.shape[:-1] + (x.shape[-1] // 8, 8))
    words = (nib << (4 * np.arange(8))).sum(-1)
    return words.astype(np.uint32).view(np.int32)


def tv_sign_edge_input(B: int, D: int, H: int, W: int) -> np.ndarray:
    """float32 [B, D, H, W] for the fp32 sign codes: along every row, pairs of neighbours that are +0 / -0, equal after
    bf16 rounding but not in fp32 (1 and 1 + 2^-20), the smallest normal magnitude apart (2^-126 vs 0 and vs 2^-125), and
    near 1e30 (whose differences overflow when scaled but keep their sign); the rows above and below shift the pattern."""
    pattern = np.array([0.0, -0.0, 0.0, 1.0, 1.0 + 2.0 ** -20, 1.0, 2.0 ** -126, 0.0, 2.0 ** -125, 2.0 ** -126,
                        1e30, -1e30, 1e30, np.float32(1e30) * (1 + 2.0 ** -23), -2.0 ** -126, 0.0], np.float32)
    n = B * D * H * W
    idx = (np.arange(n) + 3 * (np.arange(n) // W // 2)) % pattern.size
    return pattern[idx].reshape(B, D, H, W)


# ----------------------------------------------------------------------------------------------------------------------
# row normalisation
# ----------------------------------------------------------------------------------------------------------------------

def exact_rows(rng: np.random.Generator, B: int, D: int, H: int, W: int, zero_frac: float = 0.0) -> np.ndarray:
    """float64 [B, D, H, W] whose every pixel's channel vector has norm 2^e exactly, e in [-6, 6]: 4^j entries of
    +-2^(e-j) (4^j <= D; D = 256 allows 256 entries of +-2^(e-4)) at random channels, zeros elsewhere; a ``zero_frac``
    share of the pixels are zero rows (the 1e-12 clamp)."""
    js = [j for j in range(5) if 4 ** j <= D]
    x = np.zeros((B, H, W, D))
    e = rng.integers(-6, 7, size=(B, H, W))
    zero = rng.random((B, H, W)) < zero_frac
    for b in range(B):
        for h in range(H):
            for w in range(W):
                if zero[b, h, w]:
                    continue
                j = int(rng.choice(js))
                ch = rng.choice(D, size=4 ** j, replace=False)
                x[b, h, w, ch] = rng.choice([-1.0, 1.0], size=ch.size) * 2.0 ** (int(e[b, h, w]) - j)
    return x.transpose(0, 3, 1, 2).copy()


def normalize_reference(x: np.ndarray):
    """(x_hat float64 [B, D, H, W], inv float64 [B, H*W]): x / max(|x|, 1e-12) per pixel and 1 / max(|x|, 1e-12); zero
    rows get the fp32 value of 1 / 1e-12 that the kernels form."""
    x = np.asarray(x, np.float64)
    B, D = x.shape[:2]
    nrm = np.sqrt((x * x).sum(1))
    inv = np.where(nrm > 0, 1.0 / np.maximum(nrm, 1e-12), np.float64(F32_ONE_OVER_EPS))
    return x * inv[:, None], inv.reshape(B, -1)


def normalize_backward_reference(xhat: np.ndarray, g: np.ndarray, inv: np.ndarray):
    """(dx, sum_d |x_hat g|) float64 for dx = (g - x_hat (x_hat . g)) inv per pixel; xhat, g [B, D, H, W], inv [B, H*W]."""
    xhat = np.asarray(xhat, np.float64)
    g = np.asarray(g, np.float64)
    inv = np.asarray(inv, np.float64).reshape((xhat.shape[0], 1) + xhat.shape[2:])
    dot = (xhat * g).sum(1, keepdims=True)
    return (g - xhat * dot) * inv, np.abs(xhat * g).sum(1, keepdims=True)


def tv_normalize_backward_reference(xhat: np.ndarray, inv: np.ndarray, sh: float, sv: float) -> np.ndarray:
    """The composition rc_tv_normalize_bwd fuses: the closed-form TV gradient of x_hat, then the normalisation backward."""
    return normalize_backward_reference(xhat, tv_grad_reference(xhat, sh, sv), inv)[0]


# ----------------------------------------------------------------------------------------------------------------------
# sampling helpers
# ----------------------------------------------------------------------------------------------------------------------

def sample_draws(rng: np.random.Generator, B: int, HW: int, n: int) -> np.ndarray:
    """int64 [B, n] pixel draws: uniform, plus a few hundred draws of one pixel per image and draws outside [0, HW)."""
    r = rng.integers(0, HW, size=(B, n))
    for b in range(B):
        hot = rng.choice(n, size=min(n, 300), replace=False)
        r[b, hot] = rng.integers(0, HW)
        bad = rng.choice(np.setdiff1d(np.arange(n), hot), size=min(n - hot.size, 5), replace=False)
        r[b, bad] = rng.choice([-1, -7, HW, HW + 3], size=bad.size)
    return r


def sample_label_counts_reference(seg: np.ndarray, rand_idx: Optional[np.ndarray], C: int) -> np.ndarray:
    """int64 [C]: labels of the drawn pixels in [0, C) (every pixel once when rand_idx is None), draws outside [0, HW)
    skipped."""
    B, HW = seg.shape
    if rand_idx is None:
        lab = seg.reshape(-1)
    else:
        ok = (rand_idx >= 0) & (rand_idx < HW)
        lab = np.concatenate([seg[b, rand_idx[b][ok[b]]] for b in range(B)])
    lab = lab[(lab >= 0) & (lab < C)]
    return np.bincount(lab, minlength=C)[:C]


def sample_weights_reference(seg: np.ndarray, rand_idx: Optional[np.ndarray], label_map: np.ndarray):
    """(w float64 [B, HW], y int64 [B, HW]): y = label_map[seg] for 0 < seg < C, else -1; w = multiplicity of the pixel
    among the draws (1 without draws), 0 wherever y < 0."""
    B, HW = seg.shape
    C = label_map.size
    ok = (seg > 0) & (seg < C)
    y = np.where(ok, label_map[np.where(ok, seg, 0)], -1)
    if rand_idx is None:
        w = np.ones((B, HW))
    else:
        w = np.stack([np.bincount(r[(r >= 0) & (r < HW)], minlength=HW)[:HW] for r in rand_idx]).astype(np.float64)
    return np.where(y >= 0, w, 0.0), y


def text_reference(text: np.ndarray, idx: Optional[np.ndarray]) -> np.ndarray:
    """float64 [K, D]: F.normalize(text[idx], dim=1); idx -1 -> a zero row, another index outside the table -> NaN."""
    text = np.asarray(text, np.float64)
    n, D = text.shape
    idx = np.arange(n) if idx is None else np.asarray(idx)
    out = np.full((idx.size, D), np.nan)
    for k, i in enumerate(idx):
        if i == -1:
            out[k] = 0.0
        elif 0 <= i < n:
            out[k] = text[i] / max(np.sqrt((text[i] ** 2).sum()), 1e-12)
    return out
