"""CPU checks of the open-vocabulary scores entry points (rc_eval_topk_scores_bf16 / _rep4, ops.eval_topk_scores,
rangeclip_b200.segment_from_embeddings): malformed arguments are refused before any launch, CPU tensors are refused, and
the fake-tensor rule of rangeclip::eval_topk_scores gives the outputs' shapes and dtypes."""
import ctypes

import pytest
import torch

BUF = (ctypes.c_uint8 * 4096)()
P = (ctypes.addressof(BUF) + 255) // 256 * 256        # a 256-byte aligned host address: the checks never dereference it


def _lib():
    from rangeclip_b200 import _lib
    return _lib, _lib.lib()


def _full(L, lib, *, x=P, B=1, D=64, HW=128, t=P, K=16, imap=P, k=1, lt=P, ids=P, cos=P, prob=P):
    return lib.rc_eval_topk_scores_bf16(x, L.RC_BF16, B, D, HW, t, K, imap, k, lt, ids, cos, prob, None, 0, None)


def _rep4(L, lib, *, x=P, B=1, D=64, h=4, w=4, t=P, K=16, imap=P, k=1, lt=P, ids=P, cos=P, prob=P):
    return lib.rc_eval_topk_scores_bf16_rep4(x, L.RC_BF16, B, D, h, w, t, K, imap, k, lt, ids, cos, prob, None, 0, None)


@pytest.mark.parametrize("call", [_full, _rep4])
@pytest.mark.parametrize("missing", ["x", "t", "imap", "lt", "ids", "cos", "prob"])
def test_scores_entry_points_refuse_null_pointers(call, missing):
    L, lib = _lib()
    assert call(L, lib, **{missing: None}) == -1
    assert b"null pointer" in lib.rc_last_error()


@pytest.mark.parametrize("call", [_full, _rep4])
def test_scores_entry_points_refuse_shapes_outside_the_kernel(call):
    L, lib = _lib()
    assert call(L, lib, k=9) == -1                                     # k <= 8
    assert b"bad shape" in lib.rc_last_error()
    assert call(L, lib, k=0) == -1
    assert call(L, lib, K=4, k=5) == -1                                # k <= K
    assert call(L, lib, D=96) == -2                                    # D % 64
    assert b"multiple of 64" in lib.rc_last_error()
    assert call(L, lib, D=1088) == -2                                  # D <= 1024
    if call is _full:
        assert call(L, lib, HW=100) == -2                              # HW % 8
    else:
        assert call(L, lib, h=5, w=5) == -2                            # h * w % 8
        assert call(L, lib, h=0) == -1
    assert b"multiple of 8" in lib.rc_last_error() or b"bad shape" in lib.rc_last_error()


def test_rep4_scores_refuse_misaligned_outputs():
    """The half-resolution form writes every id as one 16-byte store and every score pair as one 8-byte store."""
    L, lib = _lib()
    assert _rep4(L, lib, ids=P + 8) == -1
    assert b"16-byte aligned" in lib.rc_last_error()
    assert _rep4(L, lib, cos=P + 4) == -1
    assert b"8-byte aligned" in lib.rc_last_error()
    assert _rep4(L, lib, prob=P + 4) == -1
    assert b"8-byte aligned" in lib.rc_last_error()


def test_scores_python_layer_refuses_cpu_tensors_and_bad_shared2x2_input():
    import rangeclip_b200 as R
    from rangeclip_b200 import ops
    x, t = torch.zeros(1, 64, 4, 4), torch.randn(10, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        R.segment_from_embeddings(x, t, 0.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.eval_topk_scores(x, torch.zeros(64, 64, dtype=torch.bfloat16), torch.arange(10), 1, torch.zeros(()))
    with pytest.raises(RuntimeError, match="output_conv"):
        R.segment_from_embeddings(torch.zeros(1, 64, 16), t, 0.0, shared2x2=True)
    assert "segment_from_embeddings" in R.__all__


@pytest.mark.parametrize("shared2x2", [False, True])
@pytest.mark.parametrize("K,k", [(100, 5), (3, 5), (1000, 1)])
def test_scores_fake_rule_on_meta_tensors(shared2x2, K, k):
    import rangeclip_b200  # noqa: F401  (registers the operators)
    x = torch.empty(2, 512, 12, 20, device="meta", dtype=torch.bfloat16)
    tb = torch.empty((K + 63) // 64 * 64, 512, device="meta", dtype=torch.bfloat16)
    imap = torch.empty(K, device="meta", dtype=torch.int64)
    ids, cos, prob = torch.ops.rangeclip.eval_topk_scores(x, tb, imap, k, torch.empty(1, device="meta"), shared2x2)
    shape = (2, min(k, K)) + ((24, 40) if shared2x2 else (12, 20))
    assert tuple(ids.shape) == tuple(cos.shape) == tuple(prob.shape) == shape
    assert (ids.dtype, cos.dtype, prob.dtype) == (torch.int64, torch.float32, torch.float32)
