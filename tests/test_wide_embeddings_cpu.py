"""Embeddings wider than 512 channels without a GPU: the InfoNCE route table at D = 768 / 1024 (CLIP ViT-L/14, ViT-H/14) and
at widths only the fp32 kernel takes (640) or none (1280), the fake-tensor rules that follow it, and the C entry points'
refusal of widths no kernel covers (before any launch)."""
import ctypes

import pytest
import torch


def _x(D, h=16, w=16, B=2, dtype=torch.bfloat16):
    return torch.empty(B, D, h, w, device="meta", dtype=dtype)


# D, K, need_dx, need_dt, precision, rep, device parameters -> route
ROUTES = [(D,) + r for D in (768, 1024) for r in [
    (256, True, False, "auto", 1, False, "bf16"),
    (1, True, False, "auto", 1, False, "bf16"),
    (256, False, False, "bf16", 1, False, "bf16"),           # forward only
    (257, True, False, "auto", 1, False, "kblocked"),
    (700, True, False, "auto", 1, False, "kblocked"),
    (257, True, False, "bf16", 1, False, None),
    (256, True, False, "kblocked", 1, False, "kblocked"),
    (256, True, False, "fp32", 1, False, "fp32"),
    (256, True, False, "auto", 4, False, "bf16"),           # four targets
    (700, True, False, "auto", 4, False, "kblocked"),
    (700, True, False, "bf16", 4, False, "kblocked"),
    (256, True, False, "bf16", 1, True, "bf16"),            # K and log tau in device memory
    (256, True, False, "auto", 4, True, "bf16"),
    (257, True, False, "auto", 1, True, None),
    (256, True, True, "auto", 1, False, "fp32"),            # dText stays on the tensor cores at 256 / 512 only
    (256, True, True, "bf16", 1, False, None),
    (256, True, True, "auto", 4, False, None),
    (256, True, True, "bf16", 1, True, None),
]] + [
    (640, 256, True, False, "auto", 1, False, "fp32"),      # no tensor-core kernel at 640 / 896: the fp32 kernel
    (896, 700, True, True, "auto", 1, False, "fp32"),
    (640, 256, True, False, "bf16", 1, False, None),
    (640, 300, True, False, "kblocked", 1, False, None),
    (640, 256, True, False, "auto", 4, False, None),
    (1280, 256, True, False, "auto", 1, False, None),       # wider than any kernel
    (1280, 256, True, False, "fp32", 1, False, None),
    (1280, 700, True, False, "auto", 1, False, None),
    (1280, 256, True, False, "auto", 4, False, None),
    (1280, 256, True, False, "bf16", 1, True, None),
    (1088, 256, True, False, "auto", 1, False, None),
]


@pytest.mark.parametrize("D,K,need_dx,need_dt,precision,rep,dev_params,route", ROUTES)
def test_route_table_wide(D, K, need_dx, need_dt, precision, rep, dev_params, route):
    from rangeclip_b200 import ops
    for dtype in (torch.bfloat16, torch.float32):
        assert ops._infonce_plan(_x(D, dtype=dtype), K, need_dt, precision, rep, need_dx, dev_params) == route


@pytest.mark.parametrize("D", [768, 1024])
@pytest.mark.parametrize("rep", [1, 4])
def test_device_blocks_up_to_1024_rows(D, rep):
    from rangeclip_b200 import ops
    x = _x(D)
    for K, route in ((1, "bf16"), (256, "bf16"), (257, "kblocked"), (700, "kblocked"), (1024, "kblocked"), (1025, None)):
        assert ops._infonce_plan(x, K, False, "bf16", rep, True, True, True) == route
    assert ops._infonce_plan(x, 300, True, "bf16", rep, True, True, True) is None            # no dText there
    assert ops._infonce_plan(_x(640), 256, False, "bf16", rep, True, True, True) is None


def test_other_checks_follow_the_plan():
    from rangeclip_b200 import evaluation, losses, ops
    for D in (768, 1024):
        assert ops.kblocked_supported(D, 256) and ops.topk_bf16_supported(D, 256)
        assert losses.device_builder_supported(_x(D), 1, 600, 1024, False, "auto")
        assert losses.device_builder_supported(_x(D), 4, 600, 256, False, "auto")
        assert not losses.device_builder_supported(_x(D), 1, 600, 256, True, "auto")        # trainable text: dText
    for D in (640, 1280):
        assert not ops.kblocked_supported(D, 256)
        assert not losses.device_builder_supported(_x(D), 1, 600, 256, False, "auto")
    assert ops.topk_bf16_supported(640, 256) and ops.topk_bf16_supported(960, 256)
    assert not ops.topk_bf16_supported(1088, 256) and not ops.topk_bf16_supported(1280, 256)
    assert not evaluation.device_candidates_supported(_x(1280), 100)                        # a meta tensor is not on CUDA either
    # the area-image loss: "auto" takes the K blocks from n = 512 at the new widths (frozen image embeddings, n % 8 == 0)
    for D in (768, 1024):
        x = torch.empty(1, D, 1024, 1, device="meta")
        assert ops._infonce_plan(x, 1024, False, "kblocked", 1) == "kblocked"
        assert ops._infonce_plan(torch.empty(1, D, 64, 1, device="meta"), 64, False, "fp32", 1) == "fp32"      # n = 64


def _args(D, K, dtype, hw=(16, 16), rep=1):
    x = _x(D, *hw, dtype=dtype)
    rows = 2 * hw[0] * hw[1]
    yw = (rows, 4) if rep == 4 else (rows,)
    return (x, torch.empty(K, D, device="meta"), torch.zeros((), device="meta"), torch.empty(yw, device="meta", dtype=torch.int32),
            torch.empty(yw, device="meta"))


@pytest.mark.parametrize("D,K,x_dtype,precision,rep,dx_dtype", [
    (768, 256, torch.float32, "auto", 1, torch.bfloat16),     # one tensor-core launch: dX stays bf16 until the backward
    (1024, 256, torch.bfloat16, "auto", 1, torch.bfloat16),
    (1024, 256, torch.float32, "fp32", 1, torch.float32),     # the CUDA-core kernel: x's dtype
    (768, 700, torch.float32, "auto", 1, torch.float32),      # the K blocks: x's dtype
    (1024, 300, torch.float32, "auto", 4, torch.float32),
    (768, 200, torch.float32, "auto", 4, torch.bfloat16),
    (640, 256, torch.float32, "auto", 1, torch.float32),      # the fp32 kernel
])
def test_fake_dx_dtype_follows_the_route_wide(D, K, x_dtype, precision, rep, dx_dtype):
    x, t, log_tau, y, w = _args(D, K, x_dtype, rep=rep)
    out = torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, False, precision, rep, None, None, None)
    assert out[1].dtype == dx_dtype and tuple(out[1].shape) == tuple(x.shape)


@pytest.mark.parametrize("D,K,need_dt,precision,rep", [
    (1280, 256, False, "auto", 1),
    (1280, 256, False, "fp32", 1),
    (1280, 700, False, "auto", 1),
    (640, 256, False, "bf16", 1),
    (768, 256, True, "bf16", 1),
])
def test_fakes_raise_where_no_kernel_takes_the_call_wide(D, K, need_dt, precision, rep):
    x, t, log_tau, y, w = _args(D, K, torch.bfloat16, rep=rep)
    with pytest.raises(RuntimeError, match="no kernel covers"):
        torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, need_dt, precision, rep, None, None, None)
    with pytest.raises(RuntimeError, match="no kernel covers"):
        torch.ops.rangeclip.pixel_losses(x, t, log_tau, y, w, True, need_dt, precision, None, None, None)


def _buf():
    buf = (ctypes.c_uint8 * 4096)()
    return buf, ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 16      # 16-byte aligned, never dereferenced


@pytest.mark.parametrize("D", [896, 1280, 640, 1088])
def test_tensor_core_entry_points_reject_uncovered_widths(D):
    """RC_ERR_UNSUPPORTED (-2) from the argument checks, before any launch (no device is touched here)"""
    from rangeclip_b200 import _lib
    L = _lib.lib()
    buf, p = _buf()
    B, HW, K = 1, 256, 256
    calls = {
        "rc_infonce_bf16": lambda: L.rc_infonce_bf16(p, _lib.RC_BF16, B, D, HW, p, p, K, p, p, 10.0, p, p, p, p, None, p, None, p,
                                                      p, 4096, 0, None),
        "rc_infonce_bf16_rep4": lambda: L.rc_infonce_bf16_rep4(p, _lib.RC_BF16, B, D, HW, p, p, K, p, p, 10.0, p, p, p, p, None, p,
                                                                None, p, p, 4096, 0, None),
        "rc_infonce_bf16_dyn": lambda: L.rc_infonce_bf16_dyn(p, _lib.RC_BF16, B, D, HW, p, p, K, p, p, p, p, 1, p, p, p, p, None, p,
                                                              p, p, 4096, 0, None),
        "rc_infonce_bf16_dyn_kblock": lambda: L.rc_infonce_bf16_dyn_kblock(p, _lib.RC_BF16, B, D, HW, p, p, K, p, 0, p, p, p, 1, p,
                                                                            p, p, p, None, p, p, p, 4096, 2, None),
        "rc_infonce_bf16_kblocks": lambda: L.rc_infonce_bf16_kblocks(p, _lib.RC_BF16, D, HW, p, p, 300, 2, p, p, 10.0, p, p, p, p,
                                                                      None, None, None, p, 4096, 0, None),
    }
    if D > 1024:
        calls["rc_eval_topk_bf16"] = lambda: L.rc_eval_topk_bf16(p, _lib.RC_BF16, B, D, HW, p, K, p, 5, p, None, 0, None)
    for name, call in calls.items():
        assert call() == -2, (name, L.rc_last_error())
        assert f"D={D}".encode() in L.rc_last_error(), (name, L.rc_last_error())


def test_fp32_entry_points_reject_wider_than_1024():
    from rangeclip_b200 import _lib
    L = _lib.lib()
    buf, p = _buf()
    assert L.rc_infonce_f32(p, 1, 1280, 64, 1280 * 64, p, 8, p, p, 10.0, p, p, p, None, None, None, None, None, None) == -2
    assert b"D=1280" in L.rc_last_error()
    assert L.rc_eval_topk_f32(p, 1, 1280, 64, 1280 * 64, p, 8, p, 5, p, None) == -2
    assert b"D=1280" in L.rc_last_error()
