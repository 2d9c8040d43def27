"""The premise of tests/test_gpu_exact_memory_bound.py, checked without a GPU: on every case of that file, the float64
reference is exactly representable where the kernels store or accumulate it, so that a bit-for-bit comparison is fair.

A builder change that makes some result inexact (a finer grid, a larger magnitude, a count that is not a power of two)
fails here instead of as a one-ulp mismatch on the GPU.  The oracle is also checked against plain loops and PyTorch on
small inputs, so that a shared mistake between the oracle's vectorised form and the kernels cannot pass unseen."""
import numpy as np
import pytest
import torch

import test_gpu_exact_memory_bound as G
from oracle import exact_inputs as E
from oracle import rangeclip_oracle as O

F32, BF16 = torch.float32, torch.bfloat16
FP32_EXACT_INT = 2 ** 24


@pytest.mark.parametrize("case", G.POOL_FWD, ids=[c[0] for c in G.POOL_FWD])
def test_pool_forward_premise(case):
    """Every partial slot sum a kernel can form is exact in fp32: the sum of |x| over a slot stays below 2^24 grid steps."""
    name, B, D, H, W, dtype, per_image, n_maps, off, vec = case
    x64, segs, lut, n_slots = G.pool_case(B, D, H, W, per_image, n_maps, seed=len(name) * 100 + D + H + W)
    assert E.fits(x64, dtype)
    sums, cnt, mean = E.pool_reference(x64, segs, lut, per_image, n_slots)
    abs_sums = E.pool_reference(np.abs(x64), segs, lut, per_image, n_slots)[0]
    assert E.fits(sums, F32) and (abs_sums * 8 < FP32_EXACT_INT).all() and cnt.max() < FP32_EXACT_INT
    assert cnt[-1] == 0 and not mean[-1].any()
    if W == 256 and H >= 4:       # the structured map: chunk pairs that merge (rows 2, 3) and pairs that do not (rows 0, 1)
        s0 = E.pool_segmentation(np.random.default_rng(0), 1, H, W, 23)[0].reshape(H, W)
        assert np.array_equal(s0[2], s0[3]) and not np.array_equal(s0[0], s0[1])


@pytest.mark.parametrize("case", G.POOL_BWD, ids=[c[0] for c in G.POOL_BWD])
def test_pool_backward_premise(case):
    """dx after every label map (what the kernel stores between accumulating passes) is exact in the output dtype."""
    segs, lut, g64, cnt64, refs = G.pool_bwd_case(case)
    assert E.fits(g64, F32) and (np.log2(np.maximum(cnt64, 1)) % 1 == 0).all()
    for r in refs:
        assert E.fits(r, case[5])
    assert len(refs) == case[7]


def test_pool_reference_against_the_loop_oracle():
    rng = np.random.default_rng(1)
    B, D, H, W, C = 2, 5, 4, 24, 6
    x = E.dyadic(rng, (B, D, H * W))
    seg = rng.integers(0, C, size=(B, H * W))
    lut = np.tile(np.arange(C, dtype=np.int32), (B, 1))
    sums, cnt, mean = E.pool_reference(x, [seg], lut, True, C)
    items = [b for b in range(B) for _ in range(C)]
    labels = [c for _ in range(B) for c in range(C)]
    ref = O.area_pool_per_image(torch.from_numpy(x).view(B, D, H, W), torch.from_numpy(seg).view(B, H, W), items, labels)
    folded = np.zeros((C, D))         # the loop oracle gives per-(image, label) means: fold them into the slot sums
    for b in range(B):
        folded += ref.view(B, C, D)[b].numpy() * np.bincount(seg[b], minlength=C)[:, None]
    assert np.allclose(folded, sums, rtol=1e-14, atol=1e-14)
    assert np.array_equal(cnt, np.bincount(seg.reshape(-1), minlength=C))


@pytest.mark.parametrize("case,mode", [(p.values[0], p.values[1]) for p in G.TV_PARAMS])
def test_tv_premise(case, mode):
    """Partial sums of |differences| exact in fp32 (below 2^24 steps of 1/8); the gradient exact in the output dtype."""
    x64, dx_in64, ds64, in_dtype = G.tv_case(case, mode)
    dtype = case[5]
    assert E.fits(x64, BF16)
    sums = E.tv_sums_reference(x64)
    assert (sums * 8 < FP32_EXACT_INT).all()
    if dx_in64 is not None:
        assert E.fits(dx_in64, in_dtype)
    assert E.fits(E.tv_grad_reference(x64, G.SH, G.SV, dx_in64, ds64), dtype)


def test_tv_reference_against_oracle():
    """The generalised closed form reduces to oracle smoothness_grad, and the sums to the oracle's l1 means."""
    rng = np.random.default_rng(2)
    B, D, H, W = 2, 3, 5, 7
    x = E.tv_input(rng, B, D, H, W)
    dh, dv = B * D * H * (W - 1), B * D * (H - 1) * W
    assert np.allclose(E.tv_grad_reference(x, 1.0 / dh, 1.0 / dv), O.smoothness_grad(torch.from_numpy(x)).numpy(), rtol=0, atol=1e-15)
    s = E.tv_sums_reference(x)
    assert abs(s[0] / dh + s[1] / dv - float(O.smoothness(torch.from_numpy(x)))) < 1e-12
    assert (np.diff(x, axis=-1) == 0).mean() > 0.3           # many exactly equal neighbours


@pytest.mark.parametrize("case,mode", [(p.values[0], p.values[1]) for p in G.CODE_PARAMS])
def test_codes_premise(case, mode):
    x32, dx_in64, ds64 = G.codes_case(case, mode)
    assert E.fits(E.tv_grad_reference(x32, G.SH, G.SV, dx_in64, ds64), F32)
    if case[5] == "dyadic":
        assert (E.tv_sums_reference(x32) * 8 < FP32_EXACT_INT).all()


def test_codes_reference_layout():
    """Decoding the reference words gives back the signs; the edge input has differences that vanish in bf16 only, +0
    against -0, smallest-normal differences and differences that overflow when scaled."""
    x = E.tv_sign_edge_input(1, 1, 4, 16)
    words = E.tv_codes_reference(x).view(np.uint32)
    nib = (words[..., None] >> (4 * np.arange(8))) & 15
    ch = (nib & 3).reshape(x.shape) - 1
    cv = (nib >> 2).reshape(x.shape) - 1
    xd = x.astype(np.float64)
    assert np.array_equal(ch[..., :-1], np.sign(xd[..., :-1] - xd[..., 1:])) and (ch[..., -1] == 0).all()
    assert np.array_equal(cv[..., :-1, :], np.sign(xd[..., :-1, :] - xd[..., 1:, :])) and (cv[..., -1, :] == 0).all()
    xb = torch.from_numpy(x).to(BF16).float().numpy()
    assert ((xb[..., :-1] == xb[..., 1:]) & (x[..., :-1] != x[..., 1:])).any()
    assert (np.signbit(x[..., :-1]) != np.signbit(x[..., 1:]))[(x[..., :-1] == 0) & (x[..., 1:] == 0)].any()
    assert (np.abs(xd[..., :-1] - xd[..., 1:]) == 2.0 ** -126).any()
    assert (np.abs(xd) >= 1e30).any()


@pytest.mark.parametrize("B,D,H,W,dtype", G.NORM)
def test_normalize_premise(B, D, H, W, dtype):
    """Rows of norm 2^e: x exact in the input dtype, x_hat, inv and the backward exact in fp32 (the kernels' arithmetic;
    a bf16 dx is that exact value rounded once)."""
    x64, g64 = G.norm_case(B, D, H, W)
    assert E.fits(x64, dtype) and E.fits(g64, BF16)
    xhat, inv = E.normalize_reference(x64)
    assert E.fits(xhat, F32) and E.fits(inv, F32)
    nz = (x64 != 0).any(1)
    assert nz.any() and (~nz).any()
    assert np.array_equal(np.log2(inv.reshape(nz.shape)[nz]) % 1, np.zeros(nz.sum()))
    assert E.fits(E.normalize_backward_reference(xhat, g64, inv)[0], F32)
    # against PyTorch's F.normalize on the non-zero rows
    ref = torch.nn.functional.normalize(torch.from_numpy(x64), dim=1).numpy()
    assert np.array_equal(ref, xhat)


@pytest.mark.parametrize("B,D,H,W,dtype", G.TVN)
def test_tv_normalize_premise(B, D, H, W, dtype):
    x64 = E.exact_rows(np.random.default_rng(B * 10 + D + H + W), B, D, H, W)
    xhat, inv = E.normalize_reference(x64)
    assert E.fits(xhat, F32) and E.fits(inv, F32)
    assert E.fits(E.tv_normalize_backward_reference(xhat, inv, G.SH, G.SV), F32)


def test_normalize_backward_reference_against_autograd():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 9, 3, 8, generator=g, dtype=torch.float64, requires_grad=True)
    gin = torch.randn(2, 9, 3, 8, generator=g, dtype=torch.float64)
    torch.nn.functional.normalize(x, dim=1).backward(gin)
    xhat, inv = E.normalize_reference(x.detach().numpy())
    dx = E.normalize_backward_reference(xhat, gin.numpy(), inv)[0]
    assert np.allclose(dx, x.grad.numpy(), rtol=1e-12, atol=1e-14)


def test_sampling_references():
    rng = np.random.default_rng(4)
    B, HW, C = 2, 50, 7
    seg = rng.integers(-2, C + 2, size=(B, HW))
    r = E.sample_draws(rng, B, HW, 400)
    counts = E.sample_label_counts_reference(seg, r, C)
    loop = np.zeros(C, np.int64)
    for b in range(B):
        for p in r[b]:
            if 0 <= p < HW and 0 <= seg[b, p] < C:
                loop[seg[b, p]] += 1
    assert np.array_equal(counts, loop) and loop[0] > 0
    lm = rng.integers(-1, 5, size=C).astype(np.int32)
    w, y = E.sample_weights_reference(seg, r, lm)
    assert E.fits(w, F32) and max(np.bincount(r[b][r[b] >= 0]).max() for b in range(B)) >= 300
    for b in range(B):
        for p in range(HW):
            yy = lm[seg[b, p]] if 0 < seg[b, p] < C else -1
            assert y[b, p] == yy and w[b, p] == (np.sum(r[b] == p) if yy >= 0 else 0)


def test_text_reference():
    rng = np.random.default_rng(5)
    text = rng.standard_normal((6, 33))
    text[2] = 0
    ref = E.text_reference(text, np.array([0, 2, -1, 6, -2, 5]))
    assert np.allclose(ref[[0, 5]], torch.nn.functional.normalize(torch.from_numpy(text[[0, 5]]), dim=1).numpy(), rtol=1e-15)
    assert not ref[1].any() and not ref[2].any() and np.isnan(ref[3]).all() and np.isnan(ref[4]).all()
