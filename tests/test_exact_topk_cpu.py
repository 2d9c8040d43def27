"""The premises of oracle/exact_topk.py, checked without a GPU: every operand is bf16-exact, every partial sum is exact in
fp32, the norms are powers of two, each case holds the ties it claims, and the reference ranking and histograms agree
with a plain loop, with ``oracle.predict_tail`` and with ``O.metrics_accumulate``."""
import numpy as np
import pytest
import torch

from oracle import exact_topk as X
from oracle import rangeclip_oracle as O

CASES = [  # D, K, B, HW, k, Kv, sign
    (64, 300, 2, 136, 5, None, "mixed"), (48, 33, 1, 40, 3, None, "mixed"), (256, 600, 1, 200, 8, 150, "mixed"),
    (512, 700, 1, 128, 1, None, "neg"), (640, 1100, 1, 64, 7, None, "nonpos"), (1024, 520, 1, 72, 2, 140, "mixed"),
    (960, 257, 2, 40, 4, None, "neg"), (100, 5, 1, 24, 5, None, "mixed"), (64, 1, 1, 8, 1, None, "nonpos"),
]


@pytest.fixture(scope="module", params=CASES, ids=lambda c: "-".join(map(str, c)))
def case(request):
    D, K, B, HW, k, Kv, sign = request.param
    return X.topk_case(D, K, B, HW, k, seed=D + K, Kv=Kv, sign=sign)


def test_operands_are_bf16_exact(case):
    assert X.fits(case["x"], torch.bfloat16) and X.fits(case["t"], torch.bfloat16)
    assert X.fits(case["x"] * 8, torch.float64) and np.all(np.abs(case["t"][:, :case["core"]] * 8) <= 128)


def test_partial_sums_are_exact(case):
    """Every product is a multiple of 2^-6 and sum_d |x_d t_d| < 2^14 units: every partial sum, in any order, is an
    integer number of units below 2^14, exact in fp32 (24 bits) with ten bits to spare."""
    x, t = case["x"], case["t"]
    prods = np.einsum("bdn,kd->bdkn", x[:, :, :8], t)          # a sample of pixels, all rows
    assert np.all(np.mod(prods * 64, 1) == 0)
    span = np.einsum("bdn,kd->bkn", np.abs(x), np.abs(t)) * 64
    assert span.max() < X.SPAN_UNITS
    lg = X.logits(x, t)
    assert np.all(np.mod(lg * 64, 1) == 0)
    assert np.array_equal(lg.astype(np.float32).astype(np.float64), lg)


def test_norms_are_powers_of_two(case):
    x, t = case["x"], case["t"]
    nx = (x * x).sum(1)
    assert np.all(np.log2(nx) % 2 == 0), "every |x|^2 is a power of 4"
    nt = (t * t).sum(1)
    nz = nt[nt > 0]
    assert len(np.unique(nz)) == 1 and np.log2(nz[0]) % 2 == 0, "every non-zero |t|^2 is the same power of 4"
    # the fillers leave the logits alone
    core = case["core"]
    assert np.all(t[:, case["xf_ch"]] == 0) and np.all(x[:, case["tf_ch"], :] == 0)
    assert np.array_equal(X.logits(x[:, :core], t[:, :core]), X.logits(x, t))
    # normalising both sides multiplies each logit by a power of two: ties stay ties, order stays order
    ln = X.normalized_logits(x, t)
    assert np.array_equal(X.rank_ids(ln, case["k"], case["Kv"]), X.rank_ids(X.logits(x, t), case["k"], case["Kv"]))


def _by_class(case, c):
    lg = X.logits(case["x"], case["t"])
    B, K, HW = lg.shape
    cls = case["cls"].reshape(B, HW)
    return lg.transpose(0, 2, 1)[cls == c]                    # [pixels of class c, K]


def test_the_claimed_ties(case):
    k, K, Kv, sign = case["k"], case["K"], case["Kv"], case["sign"]
    n = min(k, Kv)
    if sign != "nonpos":
        L0 = _by_class(case, 0)
        tie = case["tie0"]
        if tie:
            v = L0[:, tie]
            assert np.all(v == v[:, :1]), "class 0: the seam rows tie"
            assert np.all(L0[:, case["win0"]] > v[:, 0]), "class 0: one winner above them"
            rest = np.delete(L0[:, :Kv], [case["win0"]] + tie, axis=1)
            assert np.all(rest < v[:, :1]), "class 0: the tie group is second"
            for j in case["near0"]:
                assert np.all(L0[:, j] == v[:, 0] - 2.0 ** -6), "class 0: near-ties one unit below"
            seams = set(tie)
            if Kv > 300:
                assert {3, 40, 131, 168}.issubset(seams), "first chunk, later chunk, c and c + 128"
                assert any(j >= 256 for j in seams), "a later block"
            assert Kv - 1 in seams or case["win0"] == Kv - 1
            if Kv % 32:
                assert any(j >= Kv // 32 * 32 for j in seams | {case["win0"]}), "the partial last chunk"
        L1 = _by_class(case, 1)
        if Kv >= 2 * n + 1:
            v = L1[:, case["tie1"]]
            assert np.all(v == v[:, :1])
            ranks_left = n - len(case["strict1"])
            assert len(case["tie1"]) > ranks_left, "class 1: the tie group is larger than the ranks left at the boundary"
            assert np.all(L1[:, case["strict1"]] > v[:, :1])
    L2 = _by_class(case, 2)
    if case["hi2"] and case["lo2"]:
        v = L2[:, case["hi2"] + case["lo2"]]
        assert np.all(v == v[:, :1]), "class 2: the rows at 128.. and 64.. tie"
        assert max(case["lo2"]) < min(case["hi2"]) and min(case["hi2"]) == 128 and len(case["lo2"]) > n
        if sign == "nonpos":
            assert np.all(v == 0), "class 2: the partner bound is exactly 0"
            assert case["zero_rows"] and np.all(case["t"][case["zero_rows"]] == 0)
            assert np.any(case["t"][case["lo2"]] != 0), "zero rows tie with non-zero rows at 0"
    L3 = _by_class(case, 3)
    assert np.all(L3 == 0)
    if sign == "neg":
        assert np.all(X.logits(case["x"], case["t"])[:, :Kv][_by_class_mask(case)] < 0), "every logit of a non-zero pixel < 0"
    # equal sums from different bits: some tied pair of rows differs in its contents
    rows = case["tie0"] if sign != "nonpos" else case["lo2"]
    if len(rows) >= 2:
        assert any(not np.array_equal(case["t"][rows[0]], case["t"][j]) for j in rows[1:])


def _by_class_mask(case):
    B, _, HW = case["x"].shape
    m = (case["cls"].reshape(B, HW) != 3)
    return np.broadcast_to(m[:, None, :], (B, case["Kv"], HW))


def test_rank_ids_against_a_plain_loop(case):
    lg = X.logits(case["x"], case["t"])
    k, Kv = case["k"], case["Kv"]
    got = X.rank_ids(lg, k, Kv)
    B, _, HW = lg.shape
    for b in range(B):
        for p in range(0, HW, 7):
            bv, bi = [], []
            for j in range(Kv):                                  # strict '>': the earlier index keeps its place
                v = lg[b, j, p]
                pos = next((q for q in range(len(bv)) if v > bv[q]), len(bv))
                bv.insert(pos, v)
                bi.insert(pos, j)
            want = (bi + [-1] * k)[:k]
            assert got[b, :, p].tolist() == want


def test_rank_ids_against_predict_tail(case):
    """oracle.predict_tail (torch.topk: tie order unspecified) agrees rank by rank on the values."""
    if case["Kv"] != case["K"]:
        pytest.skip("predict_tail has no device row count")
    x = torch.as_tensor(case["x"])
    B, D, HW = x.shape
    idx = list(range(case["K"]))
    k = case["k"]
    tail, lgn, _ = O.predict_tail(x.view(B, D, HW, 1), torch.as_tensor(case["t"]), idx, k)
    ours = X.rank_ids(X.logits(case["x"], case["t"]), k)
    lg = X.normalized_logits(case["x"], case["t"])
    v_tail = np.take_along_axis(lg, tail.view(B, k, HW).numpy(), 1)
    v_ours = np.take_along_axis(lg, ours, 1)
    assert np.array_equal(v_tail, v_ours)


def test_expected_hist_against_metrics_accumulate():
    rng = np.random.default_rng(0)
    for C, k, n in [(17, 1, 500), (64, 5, 2000), (300, 3, 1000)]:
        gt, E, cmap = X.metric_problem(rng, C, n)
        ids = rng.integers(0, C, size=(n, k))
        ids[: n // 3, 0] = gt[: n // 3]
        hist, cnt = X.expected_hist(gt, ids, E, cmap)
        st = O.MetricState()
        O.metrics_accumulate(st, gt, ids, E, cmap)
        fold = X.fold_hist(hist)
        assert sorted(fold) == sorted(st.union_top1)
        for L, v in fold.items():
            assert v == (st.intersection_top1[L], st.union_top1[L], st.intersection_topk[L], st.union_topk[L])
        assert cnt.tolist() == [st.correct_top1, st.correct_topk, st.total]
        # ranks holding -1 (past a device row count) count as no prediction: the same as a reference with fewer ranks
        if k > 1:
            pad = ids.copy()
            pad[:, 1:] = -1
            h2, c2 = X.expected_hist(gt, pad, E, cmap)
            h1, c1 = X.expected_hist(gt, ids[:, :1], E, cmap)
            assert np.array_equal(h2, h1) and np.array_equal(c2, c1)


def test_expected_ids_on_case_feed_metrics():
    """The expected ids of a case (class 3 pixels: the first k rows) through both metric statements."""
    c = X.topk_case(256, 300, 2, 64, 5, seed=4)
    ids = X.rank_ids(X.logits(c["x"], c["t"]), 5)
    flat = ids.transpose(0, 2, 1).reshape(-1, 5)
    cls = c["cls"]
    assert np.all(flat[cls == 3] == np.arange(5))
    gt, E, cmap = X.metric_problem(np.random.default_rng(1), 300, len(flat))
    hist, cnt = X.expected_hist(gt, flat, E, cmap)
    st = O.MetricState()
    O.metrics_accumulate(st, gt, flat, E, cmap)
    assert cnt.tolist() == [st.correct_top1, st.correct_topk, st.total]


def test_filler_and_four_squares():
    for S in [0, 1, 2, 3, 7, 63, 64, 65, 1000, 4095, 4097, 50000, 200000]:
        f = X.filler(S, 8)
        tot = S + int((f * f).sum())
        assert tot & (tot - 1) == 0 and (tot.bit_length() - 1) % 2 == 0 and tot >= max(S, 1)
        assert f.max() <= 256
    for r in range(0, 2000):
        a = X.four_squares(r)
        assert sum(v * v for v in a) == r
