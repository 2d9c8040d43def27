"""Exact-arithmetic tests of the evaluation top-k kernels: every id at every rank, ties included, on every kernel form.

The inputs come from oracle/exact_topk.py: dyadic entries, a bounded partial-sum span and power-of-two norms, so every
logit is exact in any summation order, on the tensor cores as on the CUDA cores.  The contract -- rank by logit, ties to
the smaller text index, -1 past a device row count -- then fixes every output id, and each one is compared with the
stable float64 ranking by ``torch.equal``.  The fused histograms and counters are compared, also by ``torch.equal``, with
the histograms of the EXPECTED ids (``exact_topk.expected_hist``), and their fold with ``O.metrics_accumulate``; never
with ``rc_eval_hist`` on the returned ids, which shares ``pixel_metric`` with the kernel and cannot see a ranking error.
Each case asserts, by name from ``torch.profiler``, the kernel it is meant to reach.

Dispatch table (host conditions -> kernel -> the test that reaches it)

eval_topk_bf16_impl (eval_topk_umma.cu): pair = n_tiles >= 2 && (n_blocks >= 2 || k == 1); streamed X = D > 512;
KT = k for k in {1, 5}, else 0 (run-time k); R = 4 only through rc_eval_topk_bf16_rep4.  Every form runs with bf16 x
and with fp32 x (the rownorm pre-pass), ids only and with the fused metrics, inside canary words (test_topk_form).
  eval_topk_umma_kernel<1,false,2,1>      D <= 512, one tile                        test_topk_form[res-r1-k1-single]
  eval_topk_umma_kernel<5,false,2,1>      D <= 512, one text block                  test_topk_form[res-r1-k5-single]
  eval_topk_umma_kernel<0,false,2,1>      D <= 512, one tile, k = 3                 test_topk_form[res-r1-k3-single]
  eval_topk_umma_kernel<1,true,2,1>       D <= 512, 3 tiles (phantom), one block    test_topk_form[res-r1-k1-pair]
  eval_topk_umma_kernel<5,true,2,1>       D <= 512, 4 tiles, 5 blocks               test_topk_form[res-r1-k5-pair]
  eval_topk_umma_kernel<0,true,2,1>       D <= 512, 3 tiles, k = 7                  test_topk_form[res-r1-k7-pair]
  eval_topk_umma_kernel<1,false,2,4>      rep4, one tile                            test_topk_form[res-r4-k1-single]
  eval_topk_umma_kernel<5,false,2,4>      rep4, one tile                            test_topk_form[res-r4-k5-single]
  eval_topk_umma_kernel<0,false,2,4>      rep4, one block, k = 2                    test_topk_form[res-r4-k2-single]
  eval_topk_umma_kernel<1,true,2,4>       rep4, 3 tiles                             test_topk_form[res-r4-k1-pair]
  eval_topk_umma_kernel<5,true,2,4>       rep4, 4 tiles                             test_topk_form[res-r4-k5-pair]
  eval_topk_umma_kernel<0,true,2,4>       rep4, 3 tiles, k = 4                      test_topk_form[res-r4-k4-pair]
  eval_topk_umma_xs_kernel<...>           the same twelve at 512 < D <= 1024        test_topk_form[xs-*]
    (D = 576, 640, 960 wrap the 8-slot X ring inside a text block; 768 and 1024 at a block boundary)
  KT = 0 for k = 2, 3, 4, 6, 7, 8, resident and streamed                            test_topk_generic_k
  K = 1, K = k, K % 32 != 0, K = 257, K = 1024, 1100; HW % 128 != 0                test_topk_shapes
  device row count Kv in {1, < k, < K, = K}, pads that would win                    test_topk_dyn
rc_eval_topk_f32 (infonce_simt.cu): dispatch_dpt on D, the wide form above 512      test_topk_f32
  eval_topk_f32_kernel<8>                 D <= 64 (D = 48)
  eval_topk_f32_kernel<16>                64 < D <= 128 (D = 100)
  eval_topk_f32_kernel<32>                128 < D <= 256 (D = 200, 256)
  eval_topk_f32_kernel<64>                256 < D <= 512 (D = 300, 512)
  eval_topk_f32_wide_kernel               512 < D <= 1024 (D = 640, 1024)
Public calls: predict_from_embeddings (auto / bf16 / fp32, shared2x2, reference / device candidates), and
MetricAccumulator.update_from_embeddings / update_from_device_candidates with finalize()     test_predict_*, test_accumulator_*
"""
import random
import zlib

import numpy as np
import pytest
import torch

from oracle import exact_topk as X
from oracle import rangeclip_oracle as O

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32
CANARY = -0x5A5A5A5A5A5A5A5B
PAD = 2                     # canary words on each side of out (16 bytes: the rep4 stores stay aligned)


def dev():
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.key.replace(" ", "") for e in prof.key_averages()]


def _ran(names, want):
    assert any(want in n for n in names), (want, names)


def _umma_name(streamed, kt, pair, R):
    return f"eval_topk_umma{'_xs' if streamed else ''}_kernel<{kt},{'true' if pair else 'false'},2,{R}>"


def _equal(got: torch.Tensor, want: np.ndarray, what: str):
    w = torch.as_tensor(np.ascontiguousarray(want))
    g = got.detach().cpu()
    if not torch.equal(g, w):
        bad = (g != w).nonzero()
        raise AssertionError(f"{what}: {bad.shape[0]} of {w.numel()} differ, first at {bad[:4].tolist()}: "
                             f"{g[tuple(bad[0])].item()} vs {w[tuple(bad[0])].item()}")


def _metrics(C, n, seed):
    gt, E, cmap = X.metric_problem(np.random.default_rng(seed), C, n)
    return gt, E, cmap


def _check_metrics(hist, counters, gt, ids_flat, E, cmap, what):
    """hist / counters equal the histograms of the expected ids, and their fold equals O.metrics_accumulate."""
    eh, ec = X.expected_hist(gt, ids_flat, E, cmap)
    _equal(hist, eh, what + " hist")
    _equal(counters, ec, what + " counters")
    st = O.MetricState()
    O.metrics_accumulate(st, gt, ids_flat, E, cmap)
    fold = X.fold_hist(hist.cpu().numpy())
    assert sorted(fold) == sorted(st.union_top1), what
    for L, (i1, u1, ik, uk) in fold.items():
        assert (i1, u1, ik, uk) == (st.intersection_top1[L], st.union_top1[L], st.intersection_topk[L], st.union_topk[L]), (what, L)
    assert counters.tolist() == [st.correct_top1, st.correct_topk, st.total], what


def _flat_ids(ids, n):
    """[B, k, ...] -> [N, n]: the ranks a reference with k = min(top_k, candidates) would have."""
    B, k = ids.shape[:2]
    return np.ascontiguousarray(ids.reshape(B, k, -1).transpose(0, 2, 1).reshape(-1, k)[:, :n])


# ----------------------------------------------------------------------------------------------------------------------
# 1. every tensor-core form through the C ABI, inside canary words
# ----------------------------------------------------------------------------------------------------------------------

# id, D, B, HW or (h, w), K, k, sign, pair
_SHAPES = [
    ("r1-k1-single", 1, 120, 300, 1, "mixed", False),
    ("r1-k5-single", 2, 128, 256, 5, "neg", False),
    ("r1-k3-single", 1, 64, 700, 3, "nonpos", False),
    ("r1-k1-pair", 1, 376, 100, 1, "neg", True),
    ("r1-k5-pair", 2, 200, 1100, 5, "mixed", True),
    ("r1-k7-pair", 3, 128, 513, 7, "nonpos", True),
    ("r4-k1-single", 1, (5, 8), 257, 1, "neg", False),
    ("r4-k5-single", 1, (8, 16), 600, 5, "mixed", False),
    ("r4-k2-single", 2, (8, 8), 200, 2, "nonpos", False),
    ("r4-k1-pair", 1, (24, 11), 64, 1, "mixed", True),
    ("r4-k5-pair", 2, (9, 24), 520, 5, "nonpos", True),
    ("r4-k4-pair", 1, (16, 17), 300, 4, "neg", True),
]
_RES_D = [64, 256, 512]
_XS_D = [576, 640, 960, 768, 1024]
FORMS = ([("res-" + s[0], _RES_D[i % 3]) + s[1:] for i, s in enumerate(_SHAPES)]
         + [("xs-" + s[0], _XS_D[i % 5]) + s[1:] for i, s in enumerate(_SHAPES)])


def _form_pair(B, HW, K, k):
    n_tiles = B * -(-HW // 128)
    return n_tiles >= 2 and (-(-K // 256) >= 2 or k == 1)


def _raw_topk(x, tb, K, index_map, k, out_shape, R, w=0, hist=None, gt=None, E=None, cmap=None, counters=None):
    """rc_eval_topk_bf16 / _hist_bf16 / _bf16_rep4 on x as given, into an out buffer framed by canary words."""
    from rangeclip_b200 import _lib
    from rangeclip_b200.ops import _dt
    L = _lib.lib()
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    n_out = int(np.prod(out_shape))
    buf = torch.full((n_out + 2 * PAD,), CANARY, device=dev(), dtype=torch.int64)
    out = buf[PAD:PAD + n_out]
    ws, ws_bytes = None, 0
    if x.dtype == F32:
        ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, _dt(x)))
        ws = torch.empty(ws_bytes, device=dev(), dtype=torch.uint8)
    p = lambda t: t.data_ptr() if t is not None else None
    C = 0 if cmap is None else cmap.numel()
    if R == 4:
        _lib.check(L.rc_eval_topk_bf16_rep4(p(x), _dt(x), B, D, HW // w, w, p(tb), K, None, p(index_map), k, p(out), p(gt), p(E),
                                            p(cmap), C, p(hist), p(counters), p(ws), ws_bytes, _stream()), "rc_eval_topk_bf16_rep4")
    elif hist is not None:
        _lib.check(L.rc_eval_topk_hist_bf16(p(x), _dt(x), B, D, HW, p(tb), K, p(index_map), k, p(out), p(gt), p(E), p(cmap), C,
                                            p(hist), p(counters), p(ws), ws_bytes, _stream()), "rc_eval_topk_hist_bf16")
    else:
        _lib.check(L.rc_eval_topk_bf16(p(x), _dt(x), B, D, HW, p(tb), K, p(index_map), k, p(out), p(ws), ws_bytes, _stream()),
                   "rc_eval_topk_bf16")
    return buf


def _unframe(buf, shape, what):
    b = buf.cpu()
    assert (b[:PAD] == CANARY).all() and (b[-PAD:] == CANARY).all(), f"{what}: a canary word outside out was overwritten"
    return b[PAD:-PAD].view(shape)


@pytest.mark.parametrize("name,D,B,HW,K,k,sign,pair", FORMS, ids=[f[0] for f in FORMS])
def test_topk_form(name, D, B, HW, K, k, sign, pair):
    from rangeclip_b200 import ops
    R = 4 if isinstance(HW, tuple) else 1
    h, w = HW if R == 4 else (0, 0)
    rows = h * w if R == 4 else HW
    assert _form_pair(B, rows, K, k) == pair
    case = X.topk_case(D, K, B, rows, k, seed=zlib.crc32(name.encode()) % 1000, sign=sign)
    C = K + 3
    index_map = torch.as_tensor(np.random.default_rng(1).permutation(C)[:K]).to(dev())
    want = X.rank_ids(X.logits(case["x"], case["t"]), k, index_map=index_map.cpu().numpy())        # [B, k, rows]
    if R == 4:
        want = X.upsample2(want, h, w)
        x_shape, out_shape = (B, D, h, w), (B, k, 2 * h, 2 * w)
    else:
        x_shape, out_shape = (B, D, rows), (B, k, rows)
    tb = ops.text_to_bf16(torch.as_tensor(case["t"]).float().to(dev()))[0]
    xb = torch.as_tensor(case["x"]).reshape(x_shape).to(BF16).to(dev())
    kname = _umma_name(D > 512, k if k in (1, 5) else 0, pair, R)
    buf, names = _kernels(lambda: _raw_topk(xb, tb, K, index_map, k, out_shape, R, w=w))
    _ran(names, kname)
    ids_b = _unframe(buf, out_shape, f"{name} bf16 x")
    _equal(ids_b, want, f"{name} bf16 x")
    # fp32 x with the fused metrics: the same ids, and the histograms of the expected ids
    gt, E, cmap = _metrics(C, int(np.prod(out_shape)) // k, seed=7)
    gt_d = torch.as_tensor(gt.reshape((B,) + out_shape[2:])).to(dev())
    E_d, cmap_d = torch.as_tensor(E.astype(np.uint8)).to(dev()), torch.as_tensor(cmap).to(dev())
    hist = torch.zeros(5, C, dtype=torch.int64, device=dev())
    cnt = torch.zeros(3, dtype=torch.int64, device=dev())
    xf = torch.as_tensor(case["x"]).reshape(x_shape).float().to(dev())
    buf, names = _kernels(lambda: _raw_topk(xf, tb, K, index_map, k, out_shape, R, w=w, hist=hist, gt=gt_d, E=E_d, cmap=cmap_d,
                                            counters=cnt))
    _ran(names, kname)
    ids_f = _unframe(buf, out_shape, f"{name} fp32 x")
    assert torch.equal(ids_f, ids_b), f"{name}: fp32-x ids differ from the bf16-x launch"
    _check_metrics(hist, cnt, gt, _flat_ids(want, k), E, cmap, name)


# ----------------------------------------------------------------------------------------------------------------------
# 2. the entry points: ops.eval_topk (bf16 / fp32), eval_topk_hist, eval_topk_dyn, eval_topk_rep4
# ----------------------------------------------------------------------------------------------------------------------

def _prep(case, xdtype=BF16, shape=None):
    B, D, HW = case["x"].shape
    x = torch.as_tensor(case["x"]).reshape(shape or (B, D, HW)).to(xdtype).to(dev())
    t = torch.as_tensor(case["t"]).float().to(dev())
    return x, t


@pytest.mark.parametrize("k", [2, 3, 4, 6, 7, 8])
@pytest.mark.parametrize("D", [256, 640])
def test_topk_generic_k(D, k):
    from rangeclip_b200 import ops
    B, HW, K = 2, 136, 777
    case = X.topk_case(D, K, B, HW, k, seed=100 + k, sign=("mixed", "neg", "nonpos")[k % 3])
    x, t = _prep(case)
    out, names = _kernels(lambda: ops.eval_topk(x, t, torch.arange(K, device=dev()), k, "bf16"))
    _ran(names, _umma_name(D > 512, 0, True, 1))
    _equal(out, X.rank_ids(X.logits(case["x"], case["t"]), k), f"D={D} k={k}")


SHAPES = [  # D, B, HW, K, k
    (64, 1, 8, 1, 1), (256, 2, 24, 5, 5), (512, 1, 40, 8, 8), (576, 1, 136, 31, 3), (640, 2, 128, 32, 4),
    (960, 1, 264, 33, 5), (256, 3, 72, 257, 6), (768, 1, 200, 1024, 5), (1024, 2, 96, 1100, 8), (64, 1, 1000, 160, 5),
    (512, 1, 128, 150, 2), (256, 1, 384, 129, 1),
]


@pytest.mark.parametrize("D,B,HW,K,k", SHAPES)
@pytest.mark.parametrize("sign", ["mixed", "neg"])
def test_topk_shapes(D, B, HW, K, k, sign):
    from rangeclip_b200 import ops
    case = X.topk_case(D, K, B, HW, k, seed=K + HW, sign=sign)
    x, t = _prep(case)
    out = ops.eval_topk(x, t, torch.arange(K, device=dev()), k, "bf16")
    _equal(out, X.rank_ids(X.logits(case["x"], case["t"]), k), f"{(D, B, HW, K, k, sign)}")


F32_CASES = [(48, "eval_topk_f32_kernel<8>"), (100, "eval_topk_f32_kernel<16>"), (200, "eval_topk_f32_kernel<32>"),
             (256, "eval_topk_f32_kernel<32>"), (300, "eval_topk_f32_kernel<64>"), (512, "eval_topk_f32_kernel<64>"),
             (640, "eval_topk_f32_wide_kernel"), (1024, "eval_topk_f32_wide_kernel")]


@pytest.mark.parametrize("D,kname", F32_CASES)
@pytest.mark.parametrize("k", [1, 5, 8])
def test_topk_f32(D, kname, k):
    """The fp32 kernels normalise x: the builders' power-of-two norms keep every logit exact."""
    from rangeclip_b200 import ops
    B, HW, K = 2, 45, 300
    case = X.topk_case(D, K, B, HW, k, seed=D + k, sign=("mixed", "neg", "nonpos")[(D // 4 + k) % 3])
    x, t = _prep(case, F32)
    out, names = _kernels(lambda: ops.eval_topk(x, t, torch.arange(K, device=dev()), k, "fp32"))
    _ran(names, kname)
    _equal(out, X.rank_ids(X.logits(case["x"], case["t"]), k), f"fp32 D={D} k={k}")


@pytest.mark.parametrize("want_ids", [True, False])
@pytest.mark.parametrize("D,xdtype", [(512, BF16), (768, F32)])
def test_topk_hist_entry(D, xdtype, want_ids):
    from rangeclip_b200 import ops
    B, H, W, K, k = 2, 8, 17, 600, 5
    case = X.topk_case(D, K, B, H * W, k, seed=3, sign="mixed")
    x, t = _prep(case, xdtype, (B, D, H, W))
    C = K
    gt, E, cmap = _metrics(C, B * H * W, 11)
    hist = torch.zeros(5, C, dtype=torch.int64, device=dev())
    cnt = torch.zeros(3, dtype=torch.int64, device=dev())
    out = ops.eval_topk_hist(x, t, torch.arange(K, device=dev()), k, torch.as_tensor(gt).view(B, H, W).to(dev()),
                             torch.as_tensor(E.astype(np.uint8)).to(dev()), torch.as_tensor(cmap).to(dev()), hist, cnt,
                             want_ids=want_ids)
    want = X.rank_ids(X.logits(case["x"], case["t"]), k)
    if want_ids:
        _equal(out, want.reshape(B, k, H, W), "eval_topk_hist ids")
    else:
        assert out is None
    _check_metrics(hist, cnt, gt, _flat_ids(want, k), E, cmap, "eval_topk_hist")


DYN = [  # D, B, HW, K, Kv, k, pads
    (256, 2, 128, 300, 1, 5, "winner"), (640, 1, 136, 300, 3, 5, "winner"), (256, 1, 256, 600, 150, 5, "winner"),
    (576, 2, 64, 520, 140, 8, "winner"), (512, 1, 384, 700, 700, 1, "winner"), (1024, 1, 128, 513, 300, 4, "zero"),
    (64, 3, 40, 64, 2, 3, "zero"), (960, 1, 256, 257, 257, 5, "zero"),
]


@pytest.mark.parametrize("D,B,HW,K,Kv,k,pads", DYN)
def test_topk_dyn(D, B, HW, K, Kv, k, pads):
    """A device row count: rows past Kv would win (2x copies of a winner, or zero rows against negative logits) and must
    never be scanned; ranks >= Kv are -1, and the fused metrics are those of the Kv-candidate reference."""
    from rangeclip_b200 import ops
    case = X.topk_case(D, K, B, HW, k, seed=Kv, Kv=Kv, pads=pads, sign="mixed" if pads == "winner" else "neg")
    x, t = _prep(case)
    tb = ops.text_to_bf16(t)[0]
    idx = torch.arange(K, device=dev())
    kd = torch.tensor([Kv, 0, 0, 0], dtype=torch.int32, device=dev())
    want = X.rank_ids(X.logits(case["x"], case["t"]), k, Kv)
    out = ops.eval_topk_dyn(x, tb, kd, idx, k)
    _equal(out, want, f"dyn Kv={Kv}")
    C = K
    gt, E, cmap = _metrics(C, B * HW, Kv)
    hist = torch.zeros(5, C, dtype=torch.int64, device=dev())
    cnt = torch.zeros(3, dtype=torch.int64, device=dev())
    out2 = ops.eval_topk_dyn(x.float(), tb, kd, idx, k, torch.as_tensor(gt).to(dev()), torch.as_tensor(E.astype(np.uint8)).to(dev()),
                             torch.as_tensor(cmap).to(dev()), hist, cnt)
    assert torch.equal(out2, out)
    _check_metrics(hist, cnt, gt, _flat_ids(want, min(k, Kv)), E, cmap, f"dyn Kv={Kv}")


@pytest.mark.parametrize("D,B,h,w,K,Kv,k", [(256, 1, 5, 8, 400, 150, 5), (768, 2, 8, 9, 300, 2, 3), (512, 1, 16, 9, 64, 64, 1)])
def test_topk_rep4_entry(D, B, h, w, K, Kv, k):
    from rangeclip_b200 import ops
    case = X.topk_case(D, K, B, h * w, k, seed=h * w, Kv=Kv)
    x, t = _prep(case, BF16, (B, D, h, w))
    tb = ops.text_to_bf16(t)[0]
    kd = torch.tensor([Kv], dtype=torch.int32, device=dev())
    want = X.upsample2(X.rank_ids(X.logits(case["x"], case["t"]), k, Kv), h, w)
    C = K
    gt, E, cmap = _metrics(C, B * 4 * h * w, 5)
    hist = torch.zeros(5, C, dtype=torch.int64, device=dev())
    cnt = torch.zeros(3, dtype=torch.int64, device=dev())
    out = ops.eval_topk_rep4(x, tb, torch.arange(K, device=dev()), k, torch.as_tensor(gt).view(B, 2 * h, 2 * w).to(dev()),
                             torch.as_tensor(E.astype(np.uint8)).to(dev()), torch.as_tensor(cmap).to(dev()), hist, cnt, k_dev=kd)
    _equal(out, want, "rep4")
    _check_metrics(hist, cnt, gt, _flat_ids(want, min(k, Kv)), E, cmap, "rep4")


# ----------------------------------------------------------------------------------------------------------------------
# 3. public calls on exact inputs
# ----------------------------------------------------------------------------------------------------------------------

def _public_problem(D, B, H, W, total, seed, shared2x2):
    case = X.topk_case(D, total, B, (H // 2) * (W // 2) if shared2x2 else H * W, 5, seed=seed)
    emb_shape = (B, D, H // 2, W // 2) if shared2x2 else (B, D, H, W)
    emb = torch.as_tensor(case["x"]).reshape(emb_shape).float().to(dev())
    text = torch.as_tensor(case["t"]).float().to(dev())
    seg = torch.as_tensor(np.random.default_rng(seed).integers(0, total, size=(B, H, W))).to(dev())
    return case, emb, text, seg


def _candidates(seed, builder_device, seg, text, num_negatives):
    """The candidate set a call made after ``random.seed(seed)`` used: (rows, Kv)."""
    from rangeclip_b200 import evaluation as EV
    random.seed(seed)
    if builder_device:
        reduced, _, kinfo = EV.build_reduced_candidates_device(seg, text, num_negatives)
        Kv = int(kinfo[0])
        return reduced.cpu().numpy()[:Kv], Kv
    red = EV.build_reduced_candidates(seg, text.shape[0], num_negatives)
    return np.asarray(red, np.int64), len(red)


def _expected_public(case, rows, top_k, shared2x2, H, W):
    x = case["x"]
    lg = X.normalized_logits(x, case["t"][rows])
    want = X.rank_ids(lg, top_k, len(rows), index_map=rows)
    return X.upsample2(want, H // 2, W // 2) if shared2x2 else want.reshape(want.shape[0], top_k, H, W)


@pytest.mark.parametrize("builder", ["reference", "device"])
@pytest.mark.parametrize("precision,shared2x2", [("auto", False), ("bf16", False), ("fp32", False), ("auto", True), ("bf16", True)])
def test_predict_exact(precision, shared2x2, builder):
    from rangeclip_b200 import evaluation as EV
    D, B, H, W, total, neg, top_k = 640 if precision == "auto" else 256, 2, 16, 16, 300, 120, 5
    case, emb, text, seg = _public_problem(D, B, H, W, total, seed=21, shared2x2=shared2x2)
    random.seed(5)
    (ids, _), names = _kernels(lambda: EV.predict_from_embeddings(emb, text, seg, neg, top_k, precision=precision,
                                                                  candidate_builder=builder, shared2x2=shared2x2))
    device = builder == "device" and (shared2x2 or precision != "fp32")
    rows, _ = _candidates(5, device, seg, text, neg)
    _equal(ids, _expected_public(case, rows, top_k, shared2x2, H, W), f"predict {precision} {shared2x2} {builder}")
    if precision == "fp32":
        _ran(names, "eval_topk_f32_kernel<32>")
    else:
        _ran(names, "eval_topk_umma" + ("_xs" if D > 512 else "") + "_kernel<5,true,2," + ("4>" if shared2x2 else "1>"))


@pytest.mark.parametrize("device_candidates", [False, True])
@pytest.mark.parametrize("shared2x2", [False, True])
def test_accumulator_exact(device_candidates, shared2x2):
    """Two batches through the fused kernels; finalize() equals the oracle's metrics on the expected ids, bit for bit."""
    from rangeclip_b200 import MetricAccumulator, ops
    from rangeclip_b200 import evaluation as EV
    D, B, H, W, total, neg, top_k = 512, 2, 16, 24, 200, 60, 5
    rng = np.random.default_rng(9)
    _, E, cmap = X.metric_problem(rng, total, 1)
    acc = MetricAccumulator(torch.as_tensor(E), torch.as_tensor(cmap), device=dev())
    st = O.MetricState()
    for bi in range(2):
        case, emb, text, seg = _public_problem(D, B, H, W, total, seed=30 + bi, shared2x2=shared2x2)
        random.seed(40 + bi)
        if device_candidates:
            reduced, tb, kinfo = EV.build_reduced_candidates_device(seg, text, neg)
            ids = acc.update_from_device_candidates(emb, tb, kinfo, reduced, seg, top_k, shared2x2=shared2x2)
        else:
            red = EV.build_reduced_candidates(seg, total, neg)
            idx = torch.tensor(red, device=dev())
            t_norm, _, _ = ops.text_prepare(text, idx, want_f32=True)
            ids = acc.update_from_embeddings(emb, t_norm, idx, seg, min(top_k, len(red)), shared2x2=shared2x2)
        rows, Kv = _candidates(40 + bi, device_candidates, seg, text, neg)
        want = _expected_public(case, rows, top_k, shared2x2, H, W)
        _equal(ids, want, f"accumulator batch {bi}")
        O.metrics_accumulate(st, seg.cpu().numpy().reshape(-1), _flat_ids(want, min(top_k, Kv)), E, cmap)
    fin = acc.finalize(seg)
    ofin = O.metrics_finalize(st, seg.cpu().numpy(), cmap)
    for nm in ["intersection_top1", "union_top1", "intersection_topk", "union_topk"]:
        assert list(fin[nm].items()) == list(getattr(st, nm).items()), nm
    assert (fin["correct_pixels_top1"], fin["correct_pixels_topk"], fin["total_pixels"]) == (st.correct_top1, st.correct_topk, st.total)
    for key in ["mIoU_t1", "mIoU_tk", "pixel_accuracy_t1", "pixel_accuracy_tk"]:
        assert fin[key] == ofin[key], key
