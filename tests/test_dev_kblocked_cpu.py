"""CPU-side checks of the sync-free K-blocked InfoNCE (the device contrast builder above 256 rows): the routes the plan gives
the explicit ``dev_blocks`` opt-in, the fake-tensor dX dtype that follows them, and the argument checks of
rc_infonce_bf16_dyn_kblock that run before any device is touched."""
import ctypes

import pytest
import torch


def _x(D, h=16, w=16, B=2, dtype=torch.bfloat16):
    return torch.empty(B, D, h, w, device="meta", dtype=dtype)


# D, (h, w), capacity K, need_dt, precision, rep -> route with dev_blocks=True
DEV_BLOCK_ROUTES = [
    (512, (16, 16), 257, False, "bf16", 1, "kblocked"),
    (512, (16, 16), 512, False, "bf16", 1, "kblocked"),
    (256, (16, 16), 1024, False, "bf16", 1, "kblocked"),
    (512, (16, 16), 1024, False, "auto", 4, "kblocked"),
    (256, (16, 16), 300, False, "bf16", 4, "kblocked"),
    (512, (16, 16), 256, False, "bf16", 1, "bf16"),          # one launch (rc_infonce_bf16_dyn), as without the opt-in
    (512, (16, 16), 256, False, "bf16", 4, "bf16"),
    (512, (16, 16), 2, False, "bf16", 1, "bf16"),
    (512, (16, 16), 1025, False, "bf16", 1, None),           # four blocks at most
    (128, (16, 16), 512, False, "bf16", 1, None),            # no CTA-pair kernel
    (128, (16, 16), 256, False, "bf16", 1, None),
    (512, (16, 16), 512, True, "bf16", 1, None),             # dText
    (512, (16, 16), 256, True, "bf16", 1, None),
    (512, (16, 16), 512, False, "fp32", 1, None),            # fp32 parity mode
    (512, (3, 3), 512, False, "bf16", 1, None),              # rows % 8 != 0
]


@pytest.mark.parametrize("D,hw,K,need_dt,precision,rep,route", DEV_BLOCK_ROUTES)
def test_dev_blocks_route_table(D, hw, K, need_dt, precision, rep, route):
    from rangeclip_b200 import ops
    for dtype in (torch.bfloat16, torch.float32):
        assert ops._infonce_plan(_x(D, *hw, dtype=dtype), K, need_dt, precision, rep, True, True, dev_blocks=True) == route


@pytest.mark.parametrize("K", [257, 512, 1024])
def test_without_the_opt_in_device_parameters_above_256_still_have_no_route(K):
    from rangeclip_b200 import ops
    assert ops._infonce_plan(_x(512), K, False, "bf16", 1, True, True) is None
    assert ops._infonce_plan(_x(512), K, False, "kblocked", 1, True, True) is None


def _args(D, K, dtype, rep=1, hw=(16, 16)):
    x = _x(D, *hw, dtype=dtype)
    rows = 2 * hw[0] * hw[1]
    yw = (rows, 4) if rep == 4 else (rows,)
    return (x, torch.empty(K, D, device="meta"), torch.zeros((), device="meta"), torch.empty(yw, device="meta", dtype=torch.int32),
            torch.empty(yw, device="meta"))


@pytest.mark.parametrize("K,x_dtype,rep,dx_dtype", [
    (512, torch.float32, 1, torch.float32),       # K-blocked rounds: x's dtype
    (512, torch.bfloat16, 1, torch.bfloat16),
    (1024, torch.float32, 4, torch.float32),
    (256, torch.float32, 1, torch.bfloat16),      # one launch: dX stays bf16 until the backward
    (256, torch.float32, 4, torch.bfloat16),
])
def test_fake_dx_dtype_follows_the_dev_blocks_route(K, x_dtype, rep, dx_dtype):
    x, t, log_tau, y, w = _args(512, K, x_dtype, rep)
    k_dev = torch.empty(4, device="meta", dtype=torch.int32)
    out = torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, False, "bf16", rep, None, None, k_dev, True)
    assert out[1].dtype == dx_dtype and tuple(out[1].shape) == tuple(x.shape)
    if rep == 1:
        out = torch.ops.rangeclip.pixel_losses(x, t, log_tau, y, w, True, False, "bf16", None, None, k_dev, True)
        assert out[2].dtype == dx_dtype and tuple(out[2].shape) == tuple(x.shape)


def test_fakes_raise_above_the_capacity():
    x, t, log_tau, y, w = _args(512, 1100, torch.bfloat16)
    k_dev = torch.empty(4, device="meta", dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no kernel covers"):
        torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, False, "bf16", 1, None, None, k_dev, True)
    with pytest.raises(RuntimeError, match="no kernel covers"):
        torch.ops.rangeclip.pixel_losses(x, t, log_tau, y, w, True, False, "bf16", None, None, k_dev, True)


def _buf():
    buf = (ctypes.c_uint8 * 4096)()
    return buf, ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16      # 16-byte aligned, never dereferenced


def _call(L, p, *, D=512, K=256, k_dev=True, log_tau=True, k0=256, rep=1, dx=True, dlogtau=True, flags=None):
    from rangeclip_b200 import _lib, ops
    if flags is None:
        flags = ops.RC_INFONCE_KEEP_WEIGHT | ops.RC_INFONCE_LSE_GIVEN | ops.RC_INFONCE_ACCUMULATE_DX
    return L.rc_infonce_bf16_dyn_kblock(p, _lib.RC_BF16, 1, D, 256, p, p, K, p if k_dev else None, k0, p, p,
                                        p if log_tau else None, rep, p, p, p, p, None, p if dx else None,
                                        p if dlogtau else None, p, 4096, flags, None)


@pytest.mark.parametrize("kw,status,msg", [
    (dict(D=128), -2, b"D=128 must be 256 or 512"),
    (dict(D=384), -2, b"D=384 must be 256 or 512"),
    (dict(k_dev=False), -1, b"k_dev and log_tau_dev are required"),
    (dict(log_tau=False), -1, b"k_dev and log_tau_dev are required"),
    (dict(k0=-1), -1, b"k0=-1 must be >= 0"),
    (dict(K=257), -2, b"K=257 outside [1,256]"),
    (dict(K=0), -2, b"K=0 outside [1,256]"),
    (dict(rep=2), -1, b"rep must be 1 or 4"),
    (dict(dx=False, flags=0), -1, b"dlogtau needs dx"),       # a gradient of tau without dX
])
def test_dyn_kblock_entry_point_rejects(kw, status, msg):
    from rangeclip_b200 import _lib
    L = _lib.lib()
    buf, p = _buf()
    assert _call(L, p, **kw) == status
    assert msg in L.rc_last_error()


def test_dyn_entry_point_still_rejects_the_kblocked_flags():
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    buf, p = _buf()
    for rep in (1, 4):
        for fl in (ops.RC_INFONCE_KEEP_WEIGHT, ops.RC_INFONCE_LSE_GIVEN, ops.RC_INFONCE_ACCUMULATE_DX):
            st = L.rc_infonce_bf16_dyn(p, _lib.RC_BF16, 1, 512, 256, p, p, 256, p, p, p, p, rep, p, p, p, p, None, None, None, p,
                                       4096, fl, None)
            assert st == -1 and b"K-blocked flags" in L.rc_last_error()


def test_kblocked_raw_device_parameters_go_together_and_refuse_cpu_tensors():
    from rangeclip_b200 import ops
    x = torch.zeros(1, 512, 4, 4)
    t = torch.zeros(300, 512)
    y = torch.zeros(16, dtype=torch.int32)
    with pytest.raises(RuntimeError):
        ops.infonce_kblocked_raw(x, t, y, y.float(), 0.0, True, k_dev=torch.zeros(4, dtype=torch.int32))
    with pytest.raises(RuntimeError):
        ops.infonce_raw(x, t, y, y.float(), 0.0, True, False, "bf16", dev_blocks=True)
