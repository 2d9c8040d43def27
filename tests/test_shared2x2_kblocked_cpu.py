"""CPU-side checks of the K-blocked four-target loss (more than 256 contrast rows on the shared 2x2 embeddings): which kernel
family rangeclip::infonce plans for (its fake-tensor dX dtype depends on it; None = no kernel takes the call), and the entry points that keep rejecting the
K-blocked flags for four targets per row."""
import pytest
import torch


def _x(D, h=16, w=16, B=2, dtype=torch.bfloat16):
    return torch.empty(B, D, h, w, device="meta", dtype=dtype)


@pytest.mark.parametrize("D", [256, 512])
@pytest.mark.parametrize("K", [257, 300, 1100])
@pytest.mark.parametrize("precision", ["auto", "bf16"])
def test_rep4_above_256_candidates_plans_the_kblocked_rounds(D, K, precision):
    from rangeclip_b200 import ops
    assert ops._infonce_plan(_x(D), K, False, precision, 4) == "kblocked"
    assert ops._infonce_plan(_x(D, dtype=torch.float32), K, False, precision, 4) == "kblocked"


@pytest.mark.parametrize("D,K,need_dt,precision,h,w,route", [
    (128, 300, False, "auto", 16, 16, None),     # no CTA-pair kernel for D = 128
    (512, 300, False, "fp32", 16, 16, None),     # fp32 parity mode
    (512, 300, True, "auto", 16, 16, None),      # dText
    (512, 256, False, "auto", 16, 16, "bf16"),   # one launch covers every candidate
    (512, 300, False, "auto", 3, 3, None),       # rows % 8 != 0
])
def test_rep4_plan_outside_the_kblocked_shapes(D, K, need_dt, precision, h, w, route):
    """Outside the K-blocked shapes a four-target call takes one tensor-core launch, or no kernel takes it (None)."""
    from rangeclip_b200 import ops
    assert ops._infonce_plan(_x(D, h, w), K, need_dt, precision, 4) == route


def test_rep1_plan():
    from rangeclip_b200 import ops
    assert ops._infonce_plan(_x(512), 300, False, "auto", 1) == "kblocked"
    assert ops._infonce_plan(_x(512), 300, False, "bf16", 1) is None          # one launch takes at most 256 candidates
    assert ops._infonce_plan(_x(128), 300, False, "auto", 1) == "fp32"


def test_fake_dx_dtype_follows_the_plan():
    """The kblocked rounds return dX in x's dtype, the single four-target launch in bf16."""
    from rangeclip_b200 import ops
    log_tau = torch.zeros((), device="meta")
    for K, x_dtype, want in ((300, torch.float32, torch.float32), (200, torch.float32, torch.bfloat16)):
        x = _x(512, dtype=x_dtype)
        t = torch.empty(K, 512, device="meta")
        y = torch.empty(2 * 256, 4, device="meta", dtype=torch.int32)
        w = torch.empty(2 * 256, 4, device="meta")
        out = torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, False, "auto", 4, None, None, None)
        assert out[1].dtype == want and tuple(out[1].shape) == tuple(x.shape)


def test_dyn_entry_point_rejects_kblocked_flags_for_four_targets():
    import ctypes
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    buf = (ctypes.c_uint8 * 4096)()
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16      # 16-byte aligned, never dereferenced
    for fl in (ops.RC_INFONCE_KEEP_WEIGHT, ops.RC_INFONCE_LSE_GIVEN, ops.RC_INFONCE_ACCUMULATE_DX):
        st = L.rc_infonce_bf16_dyn(p, _lib.RC_BF16, 1, 512, 256, p, p, 256, p, p, p, p, 4, p, p, p, p, None, None, None, p,
                                   4096, fl, None)
        assert st == -1
        assert b"K-blocked flags" in L.rc_last_error()


def test_kblocked_path_refuses_cpu_tensors():
    from rangeclip_b200 import ops
    x = torch.zeros(1, 512, 4, 4)
    t = torch.zeros(300, 512)
    y = torch.zeros(16, 4, dtype=torch.int32)
    with pytest.raises(RuntimeError):
        ops.infonce_kblocked_raw(x, t, y, y.float(), 10.0, True, rep=4)
    with pytest.raises(RuntimeError):
        ops.infonce_raw(x, t, y, y.float(), 10.0, True, False, "auto", rep=4)
