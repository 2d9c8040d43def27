"""GPU checks of the shared-embedding (2x2 block) evaluation, SURVEY 8(f)-1: `rc_eval_topk_bf16_rep4` ranks the decoder's
half-resolution rows once and gives every pixel of a row's 2x2 block the same ids.  Against the upsampled launch
(`rc_eval_topk_hist_bf16` / `_dyn_bf16` on the nearest-x2 tensor) ids, histograms and counters are bit-identical: a logit does
not depend on where its row sits in a tile, and both launches break ties towards the smaller index.  Against the oracle
(decoder tail -> predict tail -> metric accumulation) the ids agree up to near-ties.  The public entry points
(`predict_and_accumulate(shared2x2=True)`) give the metrics of the stock tail."""
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import rangeclip_oracle as O

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def nearest_x2(x):
    return x.repeat_interleave(2, 2).repeat_interleave(2, 3).contiguous()


def _equivalences(C):
    """Non-transitive equivalences (a~b, b~c, a!~c) as in test_fused_topk_histograms_bit_exact."""
    eq = {i: {i} for i in range(C)}
    for a, b in [(3, 7), (7, 11), (11, 2), (20, 21), (21, 22), (5, 30), (0, 9), (31, 1)]:
        eq[a].add(b); eq[b].add(a)
    E = torch.tensor(O.build_equivalence_tensor(eq, C))
    return E.to(torch.uint8), torch.tensor(O.build_equivalence_class_map(E.numpy()))


def _case(B, D, h, w, K, seed, bad_gt):
    """Rows near the text row of their label; a full-resolution segmentation whose 3x3 label blocks cut through the 2x2
    blocks (mixed blocks); a vocabulary of 2K ids of which the even ones are candidates (gt ids outside the reduced set) and,
    with ``bad_gt``, gt ids outside [0, C)."""
    g = torch.Generator().manual_seed(seed)
    C = 2 * K
    H, W = 2 * h, 2 * w
    text = F.normalize(torch.randn(C, D, generator=g), dim=1)
    seg = torch.randint(0, C, (B, H // 3 + 2, W // 3 + 2), generator=g).repeat_interleave(3, 1).repeat_interleave(3, 2)
    seg = seg[:, 1:H + 1, 2:W + 2].contiguous()
    if bad_gt:
        seg[torch.rand(B, H, W, generator=g) < 0.03] = -1
        seg[torch.rand(B, H, W, generator=g) < 0.03] = C + 5
    x = text[seg[:, ::2, ::2].clamp(0, C - 1)].permute(0, 3, 1, 2) + 0.4 * torch.randn(B, D, h, w, generator=g)
    reduced = torch.arange(0, C, 2)
    return x, text, seg, reduced, C


@pytest.mark.parametrize("B,D,h,w,K,k,xdtype,bad_gt", [
    (1, 512, 8, 16, 1024, 5, torch.bfloat16, False),     # one tile of rows (single CTA); the upsampled launch: four tiles (pair)
    (3, 256, 12, 16, 1024, 5, torch.bfloat16, True),     # h*w = 192: a partial tile per image, six tiles
    (1, 512, 24, 16, 1024, 1, torch.float32, False),     # three tiles (an odd count), k = 1, fp32 rows
    (2, 64, 10, 20, 200, 5, torch.bfloat16, True),       # K <= 256 with k = 5: the single-CTA form; D = 64
    (2, 256, 16, 16, 300, 3, torch.float32, True),       # generic k (KT = 0)
    (2, 512, 32, 32, 1024, 5, torch.bfloat16, True),     # 16 tiles
])
def test_rep4_bit_exact_against_upsampled_launch(B, D, h, w, K, k, xdtype, bad_gt):
    from rangeclip_b200 import ops
    x, text, seg, reduced, C = _case(B, D, h, w, K, seed=B * 13 + D + K + h + k, bad_gt=bad_gt)
    E, cmap = _equivalences(C)
    xd = x.to(dev()).to(xdtype)
    sd, rd, Ed, cd = seg.to(dev()), reduced.to(dev()), E.to(dev()), cmap.to(dev())
    t_norm = text[reduced].to(dev())
    tb = ops.text_to_bf16(t_norm)[0]
    x_up = nearest_x2(xd)

    def hist0():
        return torch.zeros(5, C, device=dev(), dtype=torch.int64), torch.zeros(3, device=dev(), dtype=torch.int64)

    h_up, c_up = hist0()
    ids_up = ops.eval_topk_hist(x_up, t_norm, rd, k, sd, Ed, cd, h_up, c_up, t_bf16=tb)
    h4, c4 = hist0()
    ids4 = ops.eval_topk_rep4(xd, tb, rd, k, sd, Ed, cd, h4, c4)
    assert ids4.shape == (B, k, 2 * h, 2 * w)
    assert torch.equal(ids4, ids_up)
    assert torch.equal(h4, h_up) and torch.equal(c4, c_up)
    n_valid = int(((seg >= 0) & (seg < C)).sum())
    assert int(c4[2]) == n_valid
    if not bad_gt:
        assert n_valid == B * 4 * h * w
    # metrics only (out = NULL)
    h0, c0 = hist0()
    assert ops.eval_topk_rep4(xd, tb, rd, k, sd, Ed, cd, h0, c0, want_ids=False) is None
    assert torch.equal(h0, h_up) and torch.equal(c0, c_up)
    # ids only (hist = NULL)
    assert torch.equal(ops.eval_topk_rep4(xd, tb, rd, k), ops.eval_topk(x_up, t_norm, rd, k, "bf16", t_bf16=tb))


@pytest.mark.parametrize("k_valid,k", [(180, 5), (3, 5), (256, 1)])
def test_rep4_device_sized_candidates_bit_exact(k_valid, k):
    """k_dev with padded rows (index -1, zero text rows), including fewer valid rows than k (ids -1 there)."""
    from rangeclip_b200 import ops
    B, D, h, w, K = 2, 256, 16, 24, 256
    x, text, seg, reduced, C = _case(B, D, h, w, K // 2, seed=k_valid + k, bad_gt=True)
    E, cmap = _equivalences(C)
    xd, sd, Ed, cd = x.to(dev()).to(torch.bfloat16), seg.to(dev()), E.to(dev()), cmap.to(dev())
    idx = torch.full((K,), -1, dtype=torch.int64)
    idx[:k_valid] = torch.randperm(C, generator=torch.Generator().manual_seed(k_valid))[:k_valid].sort().values
    tb = torch.zeros(K, D, dtype=torch.bfloat16)
    tb[:k_valid] = text[idx[:k_valid]].to(torch.bfloat16)
    tb, idx = tb.to(dev()), idx.to(dev())
    kinfo = torch.tensor([k_valid, 0, 0, 0], dtype=torch.int32, device=dev())
    h_up = torch.zeros(5, C, device=dev(), dtype=torch.int64); c_up = torch.zeros(3, device=dev(), dtype=torch.int64)
    ids_up = ops.eval_topk_dyn(nearest_x2(xd), tb, kinfo, idx, k, sd, Ed, cd, h_up, c_up)
    h4, c4 = torch.zeros_like(h_up), torch.zeros_like(c_up)
    ids4 = ops.eval_topk_rep4(xd, tb, idx, k, sd, Ed, cd, h4, c4, k_dev=kinfo)
    assert torch.equal(ids4, ids_up) and torch.equal(h4, h_up) and torch.equal(c4, c_up)
    if k_valid < k:
        assert bool((ids4[:, k_valid:] == -1).all())


def _hadamard(n):
    Hm = np.array([[1.0]])
    while Hm.shape[0] < n:
        Hm = np.block([[Hm, Hm], [Hm, -Hm]])
    return torch.tensor(Hm, dtype=torch.float32)


def _separated_batch(B, h, w, C, gen):
    """Text rows = orthonormal Hadamard rows (entries +-1/sqrt(D): unit norm and bf16-exact, so normalising changes nothing);
    every row of the conv output = 1.0 t_l + 0.8 t_{l+1} + 0.6 t_{l+2} + 0.45 t_{l+3} + 0.3 t_{l+4} (l = its label), rounded to
    bf16: its top-5 logits are separated by far more than any rounding moves them.  Mixed 2x2 blocks in the segmentation."""
    lab = torch.randint(0, C, (B, h, w), generator=gen)
    text = _hadamard(C) / C ** 0.5
    wts = torch.tensor([1.0, 0.8, 0.6, 0.45, 0.3])
    rows = sum(wts[j] * text[(lab + j) % C] for j in range(5))
    conv = (2.0 * rows.permute(0, 3, 1, 2)).to(torch.bfloat16).float()
    seg = lab.repeat_interleave(2, 1).repeat_interleave(2, 2).clone()
    flip = torch.rand(seg.shape, generator=gen) < 0.1
    seg[flip] = torch.randint(0, C, (int(flip.sum()),), generator=gen)
    return conv, text, seg


def test_rep4_against_oracle():
    """oracle.decoder_tail -> predict_tail -> metrics_accumulate: ids equal up to near-ties of the oracle's logits; the
    accumulator's state equals the oracle's accumulation of the kernel's ids."""
    import rangeclip_b200 as R
    g = torch.Generator().manual_seed(3)
    B, D, h, w, C, k, n_neg = 2, 64, 8, 12, 64, 5, 20
    lab = torch.randint(0, C, (B, h, w), generator=g)
    text = torch.sign(torch.randn(C, D, generator=g)) / D ** 0.5          # unit rows, bf16-exact
    conv = (3.0 * text[lab].permute(0, 3, 1, 2) + torch.randn(B, D, h, w, generator=g)).to(torch.bfloat16).float()
    seg = torch.randint(0, C, (B, 2 * h // 4, 2 * w // 4), generator=g).repeat_interleave(4, 1).repeat_interleave(4, 2)
    seg = torch.roll(seg, (1, 3), (1, 2)).contiguous()
    E, cmap = _equivalences(C)
    random.seed(17)
    reduced = O.build_candidate_set(seg, C, n_neg)
    emb = O.decoder_tail(conv.double(), (2 * h, 2 * w))
    ref, logits, _ = O.predict_tail(emb, text.double(), reduced, k)
    acc = R.MetricAccumulator(E, cmap, device=dev())
    random.seed(17)
    ids, xn = R.predict_and_accumulate(conv.to(dev()), text.to(dev()), seg.to(dev()), acc, n_neg, k, shared2x2=True)
    assert xn.shape == (B, D, h, w) and torch.allclose(xn.cpu(), F.normalize(conv, dim=1), atol=1e-6)
    ids = ids.cpu().numpy()
    ref = ref.numpy()
    glob = {c: i for i, c in enumerate(reduced)}
    W2 = 2 * w
    for b, j, y, x_ in np.argwhere(ids != ref):
        la = float(logits[b, glob[int(ids[b, j, y, x_])], y * W2 + x_])
        lb = float(logits[b, glob[int(ref[b, j, y, x_])], y * W2 + x_])
        assert abs(la - lb) < 1e-5, (b, j, y, x_, la, lb)
    st = O.MetricState()
    O.metrics_accumulate(st, seg.numpy().reshape(-1), ids.transpose(0, 2, 3, 1).reshape(-1, k), E.numpy().astype(bool), cmap.numpy())
    fin = acc.finalize(seg.to(dev()))
    assert fin["correct_pixels_top1"] == st.correct_top1 and fin["correct_pixels_topk"] == st.correct_topk
    assert fin["total_pixels"] == st.total == B * 4 * h * w
    for name in ("intersection_top1", "union_top1", "intersection_topk", "union_topk"):
        assert fin[name] == dict(getattr(st, name)), name


def test_public_validation_step_matches_stock_tail():
    """predict_and_accumulate on the conv output (shared2x2=True) over three batches gives the finalised metrics of the stock
    tail (F.interpolate + F.normalize, then predict_and_accumulate); the device-builder form runs without a host sync."""
    import rangeclip_b200 as R
    g = torch.Generator().manual_seed(8)
    B, h, w, C, k = 2, 16, 24, 256, 5
    E, cmap = _equivalences(C)
    a_stock = R.MetricAccumulator(E, cmap, device=dev())
    a_shared = R.MetricAccumulator(E, cmap, device=dev())
    a_dev = R.MetricAccumulator(E, cmap, device=dev())
    seg = None
    for i in range(3):
        conv, text, seg = _separated_batch(B, h, w, C, g)
        conv, text, seg = conv.to(dev()), text.to(dev()), seg.to(dev())
        random.seed(100 + i)
        ids_s, _ = R.predict_and_accumulate(F.normalize(F.interpolate(conv, scale_factor=2, mode="nearest"), dim=1), text, seg,
                                            a_stock, C, k)
        random.seed(100 + i)
        ids_r, _ = R.predict_and_accumulate(conv, text, seg, a_shared, C, k, shared2x2=True)
        assert torch.equal(ids_r, ids_s)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            ids_d, _ = R.predict_and_accumulate(conv, text, seg, a_dev, C, k, candidate_builder="device", shared2x2=True)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert torch.equal(ids_d, ids_s)
        ids_p, xn = R.predict_from_embeddings(conv, text, seg, C, k, shared2x2=True)
        assert torch.equal(ids_p, ids_s) and xn.shape == conv.shape
    f_stock, f_shared, f_dev = a_stock.finalize(seg), a_shared.finalize(seg), a_dev.finalize(seg)
    assert f_shared == f_stock and f_dev == f_stock
    assert f_stock["total_pixels"] == 3 * B * 4 * h * w


def test_rep4_opcheck():
    from rangeclip_b200 import ops
    x, text, seg, reduced, C = _case(1, 128, 8, 16, 100, seed=5, bad_gt=True)
    E, cmap = _equivalences(C)
    tb = ops.text_to_bf16(text[reduced].to(dev()))[0]
    hist = torch.zeros(5, C, device=dev(), dtype=torch.int64)
    cnt = torch.zeros(3, device=dev(), dtype=torch.int64)
    args = (x.to(dev()).to(torch.bfloat16), tb, reduced.to(dev()), 5, seg.to(dev()), E.to(dev()), cmap.to(dev()), hist, cnt, None)
    torch.library.opcheck(torch.ops.rangeclip.eval_topk_rep4.default, args + (True,))
    torch.library.opcheck(torch.ops.rangeclip.eval_topk_rep4.default, args + (False,))
    torch.library.opcheck(torch.ops.rangeclip.eval_topk_rep4.default, args[:4] + (None,) * 6 + (True,))
