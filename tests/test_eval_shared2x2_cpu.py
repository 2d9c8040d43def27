"""CPU-side checks of the shared-embedding (2x2 block) evaluation entry points: rc_eval_topk_bf16_rep4 rejects malformed
arguments before any launch, and the Python layers refuse CPU tensors and a segmentation that is not twice the
resolution of the rows instead of falling back."""
import pytest
import torch


def _rep4(L, x=None, h=4, w=4, t=None, index_map=None, out=None, gt=None, hist=None, counters=None, k=1):
    from rangeclip_b200 import _lib
    return L.rc_eval_topk_bf16_rep4(x, _lib.RC_BF16, 1, 512, h, w, t, 4, None, index_map, k, out, gt, None, None, 4, hist, counters,
                                    None, 0, None)


def test_rep4_entry_point_validates_arguments():
    import ctypes
    from rangeclip_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_uint8 * 4096)()
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16      # 16-byte aligned, never dereferenced
    assert _rep4(L) == -1
    assert b"null pointer" in L.rc_last_error()
    assert _rep4(L, x=p, t=p, index_map=p) == -1                     # neither out nor hist
    assert b"null pointer" in L.rc_last_error()
    assert _rep4(L, x=p, t=p, index_map=p, out=p, h=0) == -1
    assert b"bad shape" in L.rc_last_error()
    assert _rep4(L, x=p, t=p, index_map=p, hist=p, counters=p) == -1      # metrics without gt / E / cmap
    assert _rep4(L, x=p, t=p, index_map=p, out=p, h=3, w=3) == -2          # h * w = 9 is not a multiple of 8
    assert b"multiple of 8" in L.rc_last_error()
    assert _rep4(L, x=p, t=p, index_map=p, out=p, k=9) == -1               # k > 8
    assert _rep4(L, x=p, t=p, index_map=p, out=p + 8) == -1                # ids are written 16 bytes at a time
    assert b"16-byte aligned" in L.rc_last_error()
    assert L.rc_eval_topk_bf16_rep4(p, _lib.RC_BF16, 1, 100, 4, 4, p, 4, None, p, 1, p, None, None, None, 4, None, None, None, 0,
                                    None) == -2                             # D not a multiple of 64


def test_rep4_ops_refuse_cpu_tensors_and_wrong_segmentation():
    from rangeclip_b200 import ops
    x = torch.zeros(1, 64, 2, 4)
    tb = torch.zeros(64, 64, dtype=torch.bfloat16)
    idx = torch.arange(3)
    with pytest.raises(RuntimeError):                                      # CPU tensors
        ops.eval_topk_rep4(x, tb, idx, 1)
    with pytest.raises(RuntimeError):
        ops.eval_topk_rep4(x, tb, idx, 1, torch.zeros(1, 4, 8, dtype=torch.long), torch.eye(3, dtype=torch.uint8), torch.arange(3),
                           torch.zeros(5, 3, dtype=torch.long), torch.zeros(3, dtype=torch.long))


def test_predict_shared2x2_refuses_cpu_tensors_wrong_segmentation_and_fp32():
    import rangeclip_b200 as R
    conv = torch.zeros(1, 64, 2, 4)
    text = torch.randn(5, 64)
    with pytest.raises(RuntimeError):                                      # CPU tensors
        R.predict_from_embeddings(conv, text, torch.zeros(1, 4, 8, dtype=torch.long), 2, 1, shared2x2=True)
    with pytest.raises(RuntimeError):                                      # segmentation at the rows' own resolution
        R.predict_from_embeddings(conv, text, torch.zeros(1, 2, 4, dtype=torch.long), 2, 1, shared2x2=True)
    with pytest.raises(ValueError):                                        # no CUDA-core form
        R.predict_from_embeddings(conv, text, torch.zeros(1, 4, 8, dtype=torch.long), 2, 1, precision="fp32", shared2x2=True)
    acc = R.MetricAccumulator(torch.eye(5, dtype=torch.uint8), torch.arange(5))
    with pytest.raises(RuntimeError):
        R.predict_and_accumulate(conv, text, torch.zeros(1, 4, 8, dtype=torch.long), acc, 2, 1, shared2x2=True)
    with pytest.raises(RuntimeError):
        R.predict_and_accumulate(conv, text, torch.zeros(1, 3, 8, dtype=torch.long), acc, 2, 1, shared2x2=True)
