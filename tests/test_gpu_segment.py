"""Open-vocabulary scores on the B200: ``rangeclip_b200.segment_from_embeddings`` / ``ops.eval_topk_scores`` (the scores form of
the tensor-core top-k, rc_eval_topk_scores_bf16 / _rep4).

* the ids equal ``ops.eval_topk``'s bit for bit (same ranking, same ties), on every kernel form: resident and streamed X,
  single CTA and CTA pair, k = 1, 5 and run-time k, bf16 and fp32 x;
* on the exact inputs of oracle/exact_topk.py every id and every cosine is exact; zero pixel rows get cosine 0 and
  probability 1/K; the ``neg`` variant would expose a zero pad row counted in the log-sum-exp;
* cosines and probabilities against float64 computed on the bf16-rounded operands, at tau 0.1, 0.07 and 0.01;
* shared 2x2 equals the full-resolution call on the nearest-x2 upsampled rows bit for bit;
* no host synchronisation, CUDA-graph replay equals the eager call, opcheck, and one full-size batch.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import exact_topk as X

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32


def dev():
    return torch.device("cuda:0")


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.key.replace(" ", "") for e in prof.key_averages()]


def _problem(B, D, H, W, K, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(B, D, H, W, generator=g) + 0.3 * torch.randn(1, D, 1, 1, generator=g)).to(dtype)
    t = F.normalize(torch.randn(K, D, generator=g), dim=1)
    return x.to(dev()), t.to(dev())


def _scores(x, t_norm, k, log_tau, shared2x2=False):
    from rangeclip_b200 import ops
    tb = ops.text_to_bf16(t_norm)[0]
    imap = torch.arange(t_norm.shape[0], device=dev())
    lt = torch.tensor([log_tau], device=dev(), dtype=F32)
    return ops.eval_topk_scores(x, tb, imap, k, lt, shared2x2), tb


def _reference(x, tb, K, tau, ids):
    """float64 cosine and probability of the ranked rows, computed on the bf16-rounded operands the tensor cores see (an fp32
    x is rounded by the pre-pass, which takes the norm of the rounded row)."""
    B, D = x.shape[:2]
    xb = x.to(BF16).double().reshape(B, D, -1)
    inv = 1.0 / xb.norm(dim=1, keepdim=True).clamp_min(1e-12)                   # [B, 1, HW]
    cos_all = torch.einsum("bdn,kd->bkn", xb, tb[:K].double()) * inv             # [B, K, HW]
    lse = torch.logsumexp(cos_all / tau, dim=1, keepdim=True)
    cos = torch.gather(cos_all, 1, ids.reshape(B, ids.shape[1], -1))
    return cos, torch.exp(cos / tau - lse)


def _check_bounds(cos, prob, cos_ref, prob_ref, what):
    B, k = cos.shape[:2]
    c, p = cos.double().reshape(B, k, -1), prob.double().reshape(B, k, -1)
    err_c = float((c - cos_ref).abs().max())
    assert err_c <= 1e-5, (what, "cosine", err_c)
    excess = (p - prob_ref).abs() - (2e-3 * prob_ref + 1e-7)
    assert float(excess.max()) <= 0, (what, "prob", float(excess.max()))


# ----------------------------------------------------------------------------------------------------------------------
# 1 + 3. ids equal eval_topk's; cosines and probabilities against float64 (tau 0.07), every kernel form
# ----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("D", [64, 512, 768, 1024])
@pytest.mark.parametrize("tiles", ["one", "many"])
def test_ids_equal_eval_topk_and_scores_match_fp64(dtype, D, tiles):
    from rangeclip_b200 import ops
    B, H, W = (1, 8, 16) if tiles == "one" else (2, 24, 40)
    seen = []
    for i, (K, k) in enumerate([(1, 1), (7, 8), (300, 5), (1000, 1), (1000, 8), (4097, 5), (300, 3)]):
        x, t = _problem(B, D, H, W, K, dtype, seed=1000 * D + i)
        ((ids, cos, prob), tb), names = _kernels(lambda: _scores(x, t, k, float(np.log(0.07))))
        seen += names
        ref = ops.eval_topk(x, t, torch.arange(K, device=dev()), k, "bf16", t_bf16=tb)
        assert torch.equal(ids, ref), (D, K, k, tiles)
        assert ids.shape == cos.shape == prob.shape and cos.dtype == prob.dtype == F32
        _check_bounds(cos, prob, *_reference(x, tb, K, 0.07, ids), (D, K, k, tiles))
    name = "eval_topk_scores_umma_xs_kernel<" if D > 512 else "eval_topk_scores_umma_kernel<"
    pair = ",true,2," if tiles == "many" else ",false,2,"
    assert any(name in n and pair in n for n in seen), [n for n in seen if "eval_topk" in n]


# ----------------------------------------------------------------------------------------------------------------------
# 2. exact inputs: every id, every cosine; zero rows -> cosine 0, probability 1/K
# ----------------------------------------------------------------------------------------------------------------------

# D, K, B, HW, k, sign
_EXACT = [
    (64, 300, 1, 128, 5, "neg"),           # single CTA, resident X
    (512, 1100, 2, 512, 5, "mixed"),       # CTA pair, five text blocks
    (256, 513, 3, 128, 7, "nonpos"),       # pair, run-time k, a phantom tile
    (768, 600, 2, 256, 5, "neg"),          # streamed X, pair
    (1024, 300, 1, 128, 3, "mixed"),       # streamed X, single CTA
    (576, 257, 1, 128, 1, "nonpos"),       # streamed X wrapping the 8-slot ring inside a block, arg-max
]


@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("case", _EXACT, ids=[f"D{c[0]}-K{c[1]}-k{c[4]}-{c[5]}" for c in _EXACT])
def test_exact_inputs(case, dtype):
    from rangeclip_b200 import ops
    D, K, B, HW, k, sign = case
    c = X.topk_case(D, K, B, HW, k, seed=D + K, sign=sign)
    c["x"][0, :, 1] = 0.0                  # one pixel row of norm 0: every cosine 0 (F.normalize's eps), uniform softmax
    c["cls"][1] = 3
    x = torch.tensor(c["x"], dtype=F32).to(dtype).reshape(B, D, HW // 8, 8).to(dev())
    _, tb, _ = ops.text_prepare(torch.tensor(c["t"], dtype=F32, device=dev()), None, want_f32=False, want_bf16=True)
    lt = torch.tensor([float(np.log(0.07))], device=dev())
    ids, cos, prob = ops.eval_topk_scores(x, tb, torch.arange(K, device=dev()), k, lt)
    want = X.rank_ids(X.logits(c["x"], c["t"]), k)
    assert torch.equal(ids.cpu().reshape(B, k, HW), torch.tensor(want))
    ncos = X.normalized_logits(c["x"], c["t"])
    cos_want = np.take_along_axis(ncos, want, axis=1)
    assert torch.equal(cos.cpu().reshape(B, k, HW).double(), torch.tensor(cos_want)), "cosines are exact on these inputs"
    zero = torch.tensor(c["cls"] == 3).reshape(B, HW)
    pz = prob.cpu().reshape(B, k, HW).permute(0, 2, 1)[zero]
    assert torch.equal(pz, torch.full_like(pz, np.float32(1.0 / K))), "zero rows: probability 1/K"
    assert torch.equal(ids.cpu().reshape(B, k, HW).permute(0, 2, 1)[zero], torch.arange(k).expand(int(zero.sum()), k))
    _check_bounds(cos, prob, *_reference(x, tb, K, 0.07, ids), case)


# ----------------------------------------------------------------------------------------------------------------------
# 3 + 4. probabilities across temperatures; a small vocabulary sums to one
# ----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tau", [0.1, 0.07, 0.01])
@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
def test_probabilities_against_fp64(tau, dtype):
    for (B, D, H, W, K, k) in [(2, 512, 32, 32, 1000, 5), (1, 256, 8, 16, 300, 8)]:
        x, t = _problem(B, D, H, W, K, dtype, seed=int(tau * 1000) + K)
        (ids, cos, prob), tb = _scores(x, t, k, float(np.log(tau)))
        _check_bounds(cos, prob, *_reference(x, tb, K, tau, ids), (tau, K))


@pytest.mark.parametrize("K", [1, 3, 8])
def test_probabilities_sum_to_one(K):
    x, t = _problem(2, 512, 16, 24, K, BF16, seed=K)
    for tau in (0.1, 0.01):
        (ids, cos, prob), _ = _scores(x, t, K, float(np.log(tau)))
        assert float((prob.double().sum(1) - 1).abs().max()) <= 1e-5, (K, tau)
        assert torch.equal(ids.sort(1).values, torch.arange(K, device=dev()).view(1, K, 1, 1).expand_as(ids))


# ----------------------------------------------------------------------------------------------------------------------
# 5. shared 2x2: the half-resolution launch equals the full-resolution one on the upsampled rows, bit for bit
# ----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [BF16, F32], ids=["bf16", "f32"])
@pytest.mark.parametrize("D,K,k,h,w", [(512, 1000, 5, 16, 20), (64, 40, 1, 4, 8), (768, 300, 3, 12, 12)])
def test_shared2x2_equals_upsampled(dtype, D, K, k, h, w):
    import rangeclip_b200 as R
    x, t = _problem(2, D, h, w, K, dtype, seed=D + k)
    lt = torch.tensor(float(np.log(0.05)), device=dev())
    half = R.segment_from_embeddings(x, t, lt, top_k=k, shared2x2=True)
    full = R.segment_from_embeddings(F.interpolate(x, scale_factor=2, mode="nearest"), t, lt, top_k=k)
    for a, b, name in zip(half, full, ("ids", "cosine", "prob")):
        assert a.shape == b.shape == (2, k, 2 * h, 2 * w), name
        assert torch.equal(a, b), name


# ----------------------------------------------------------------------------------------------------------------------
# 6 + 7. the public call: candidates, no host synchronisation, CUDA graphs, opcheck
# ----------------------------------------------------------------------------------------------------------------------

def test_candidates_map_to_the_vocabulary():
    import rangeclip_b200 as R
    x, t = _problem(2, 512, 16, 16, 700, BF16, seed=7)
    cand = torch.randperm(700, generator=torch.Generator().manual_seed(3))[:250].to(dev())
    lt = torch.tensor(float(np.log(0.07)), device=dev())
    ids, cos, prob = R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
    ids_s, cos_s, prob_s = R.segment_from_embeddings(x, t[cand], lt, top_k=5)
    assert torch.equal(ids, cand[ids_s]) and torch.equal(cos, cos_s) and torch.equal(prob, prob_s)
    ids_f, cos_f, prob_f = R.segment_from_embeddings(x, t, float(np.log(0.07)), top_k=5, candidates=cand)
    assert torch.equal(ids, ids_f) and torch.equal(cos, cos_f) and torch.equal(prob, prob_f)
    with pytest.raises(RuntimeError):
        R.segment_from_embeddings(x, t, lt, top_k=9)
    with pytest.raises(RuntimeError):
        R.segment_from_embeddings(x[:, :100], t[:, :100], lt)


def test_no_host_sync_and_cuda_graph_replay():
    import rangeclip_b200 as R
    x, t = _problem(2, 512, 32, 32, 1000, BF16, seed=11)
    x2 = x[:, :, ::2, ::2].contiguous()
    cand = torch.arange(0, 1000, 3, device=dev())
    lt = torch.nn.Parameter(torch.tensor(float(np.log(0.07)), device=dev()))
    eager = R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
    eager2 = R.segment_from_embeddings(x2, t, lt, top_k=5, shared2x2=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
        R.segment_from_embeddings(x2, t, lt, top_k=5, shared2x2=True)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
        out2 = R.segment_from_embeddings(x2, t, lt, top_k=5, shared2x2=True)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out + out2, eager + eager2):
        assert torch.equal(a, b)
    with torch.no_grad():                        # the temperature is read on the device at every replay
        lt.fill_(float(np.log(0.02)))
    g.replay()
    want = R.segment_from_embeddings(x, t, lt, top_k=5, candidates=cand)
    assert torch.equal(out[2], want[2]) and not torch.equal(out[2], eager[2])


def test_opcheck():
    import rangeclip_b200  # noqa: F401
    from rangeclip_b200 import ops
    x, t = _problem(2, 256, 8, 16, 100, BF16, seed=5)
    tb = ops.text_to_bf16(t)[0]
    lt = torch.tensor([float(np.log(0.07))], device=dev())
    for args in ((x, tb, torch.arange(100, device=dev()), 5, lt, False), (x, tb, torch.arange(100, device=dev()), 3, lt, True)):
        torch.library.opcheck(torch.ops.rangeclip.eval_topk_scores.default, args,
                              test_utils=("test_schema", "test_faketensor", "test_autograd_registration"))


# ----------------------------------------------------------------------------------------------------------------------
# 8. one full-size batch: B = 64, 256 x 256, D = 512, K = 1024, top-5
# ----------------------------------------------------------------------------------------------------------------------

def test_full_size_batch():
    from rangeclip_b200 import ops
    B, D, H, W, K, k, tau = 64, 512, 256, 256, 1024, 5, 0.07
    g = torch.Generator(device=dev()).manual_seed(0)
    x = torch.randn(B, D, H, W, device=dev(), dtype=BF16, generator=g)
    t = F.normalize(torch.randn(K, D, device=dev(), generator=g), dim=1)
    (ids, cos, prob), tb = _scores(x, t, k, float(np.log(tau)))
    assert torch.equal(ids, ops.eval_topk(x, t, torch.arange(K, device=dev()), k, "bf16", t_bf16=tb))
    sel = torch.randint(0, H * W, (4096,), device=dev(), generator=g)
    xs = x.reshape(B, D, H * W)[:, :, sel]
    pick = lambda a: a.reshape(B, k, H * W)[:, :, sel]
    cos_ref, prob_ref = _reference(xs, tb, K, tau, pick(ids))
    _check_bounds(pick(cos), pick(prob), cos_ref, prob_ref, "full size")
