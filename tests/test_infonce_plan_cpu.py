"""The InfoNCE route table (``ops._infonce_plan``) on meta tensors, and the fake-tensor rules of rangeclip::infonce and
rangeclip::pixel_losses that derive their outputs from it: 'fp32' = CUDA-core kernel, 'bf16' = one tensor-core launch,
'kblocked' = tensor cores over blocks of 256 candidate rows, None = no kernel takes the call (the op raises)."""
import pytest
import torch


def _x(D, h=16, w=16, B=2, dtype=torch.bfloat16):
    return torch.empty(B, D, h, w, device="meta", dtype=dtype)


# D, (h, w), K, need_dx, need_dt, precision, rep, device parameters -> route
ROUTES = [
    # one target per row
    (512, (16, 16), 256, True, False, "auto", 1, False, "bf16"),
    (128, (16, 16), 256, True, False, "auto", 1, False, "bf16"),
    (512, (16, 16), 257, True, False, "auto", 1, False, "kblocked"),
    (128, (16, 16), 257, True, False, "auto", 1, False, "fp32"),          # no CTA-pair kernel for D = 128
    (512, (16, 16), 257, True, False, "bf16", 1, False, None),            # one launch takes at most 256 candidates
    (512, (16, 16), 257, True, False, "fp32", 1, False, "fp32"),
    (256, (16, 16), 256, True, False, "kblocked", 1, False, "kblocked"),
    (128, (16, 16), 256, True, False, "kblocked", 1, False, None),
    # dText
    (512, (16, 16), 256, True, True, "auto", 1, False, "bf16"),
    (128, (16, 16), 256, True, True, "auto", 1, False, "fp32"),
    (128, (16, 16), 256, True, True, "bf16", 1, False, None),
    (512, (16, 16), 256, False, True, "bf16", 1, False, None),            # tensor-core dText comes from the dX pass
    (512, (16, 16), 256, False, True, "auto", 1, False, "fp32"),
    (512, (16, 16), 257, True, True, "auto", 1, False, "fp32"),           # the K blocks take no dText
    (512, (16, 16), 257, True, True, "kblocked", 1, False, None),
    # K and log(tau) in device memory
    (512, (16, 16), 256, True, False, "bf16", 1, True, "bf16"),
    (512, (16, 16), 256, True, False, "auto", 1, True, "bf16"),
    (128, (16, 16), 256, True, False, "bf16", 1, True, None),
    (512, (16, 16), 256, True, True, "bf16", 1, True, None),
    (512, (16, 16), 257, True, False, "auto", 1, True, None),
    (512, (16, 16), 256, True, False, "fp32", 1, True, None),
    (512, (16, 16), 256, True, False, "kblocked", 1, True, None),
    # rows % 8 != 0
    (512, (3, 3), 256, True, False, "auto", 1, False, "fp32"),
    (512, (3, 3), 256, True, False, "bf16", 1, False, None),
    (512, (3, 3), 257, True, False, "kblocked", 1, False, None),
    # four targets per row (shared 2x2 embeddings)
    (256, (16, 16), 256, True, False, "auto", 4, False, "bf16"),
    (256, (16, 16), 257, True, False, "auto", 4, False, "kblocked"),
    (512, (16, 16), 257, True, False, "bf16", 4, False, "kblocked"),
    (512, (16, 16), 256, True, False, "kblocked", 4, False, "kblocked"),
    (128, (16, 16), 256, True, False, "auto", 4, False, None),
    (512, (16, 16), 256, True, False, "fp32", 4, False, None),
    (512, (16, 16), 256, True, True, "auto", 4, False, "bf16"),
    (512, (16, 16), 257, True, True, "auto", 4, False, None),
    (512, (16, 16), 256, True, False, "bf16", 4, True, "bf16"),
    (512, (16, 16), 257, True, False, "bf16", 4, True, None),
    (512, (3, 3), 256, True, False, "auto", 4, False, None),
    # neither a kernel family nor a row form
    (512, (16, 16), 256, True, False, "tf32", 1, False, None),
    (512, (16, 16), 256, True, False, "auto", 2, False, None),
]


@pytest.mark.parametrize("D,hw,K,need_dx,need_dt,precision,rep,dev_params,route", ROUTES)
def test_route_table(D, hw, K, need_dx, need_dt, precision, rep, dev_params, route):
    from rangeclip_b200 import ops
    for dtype in (torch.bfloat16, torch.float32):
        assert ops._infonce_plan(_x(D, *hw, dtype=dtype), K, need_dt, precision, rep, need_dx, dev_params) == route


def _args(D, K, dtype, hw=(16, 16), rep=1):
    x = _x(D, *hw, dtype=dtype)
    rows = 2 * hw[0] * hw[1]
    yw = (rows, 4) if rep == 4 else (rows,)
    return (x, torch.empty(K, D, device="meta"), torch.zeros((), device="meta"), torch.empty(yw, device="meta", dtype=torch.int32),
            torch.empty(yw, device="meta"))


@pytest.mark.parametrize("D,K,x_dtype,precision,rep,dx_dtype", [
    (512, 256, torch.float32, "auto", 1, torch.bfloat16),     # one tensor-core launch: dX stays bf16 until the backward
    (512, 256, torch.bfloat16, "auto", 1, torch.bfloat16),
    (512, 256, torch.bfloat16, "fp32", 1, torch.bfloat16),    # the CUDA-core kernel: x's dtype
    (512, 256, torch.float32, "fp32", 1, torch.float32),
    (512, 257, torch.float32, "auto", 1, torch.float32),      # the K blocks: x's dtype
    (512, 200, torch.float32, "kblocked", 1, torch.float32),
    (512, 300, torch.float32, "auto", 4, torch.float32),
    (512, 200, torch.float32, "auto", 4, torch.bfloat16),
])
def test_infonce_fake_dx_dtype_follows_the_route(D, K, x_dtype, precision, rep, dx_dtype):
    x, t, log_tau, y, w = _args(D, K, x_dtype, rep=rep)
    out = torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, False, precision, rep, None, None, None)
    assert out[1].dtype == dx_dtype and tuple(out[1].shape) == tuple(x.shape)
    assert out[2].numel() == 0


@pytest.mark.parametrize("D,K,x_dtype,precision,hw,need_grad,codes", [
    (512, 256, torch.float32, "auto", (16, 16), True, (2, 512, 16, 2)),   # fp32 pre-pass: smoothness signs, 4 bits per element
    (512, 256, torch.float32, "auto", (16, 16), False, (0,)),            # no backward, no signs
    (512, 256, torch.bfloat16, "auto", (16, 16), True, (0,)),            # bf16 x: no pre-pass
    (512, 256, torch.float32, "fp32", (16, 16), True, (0,)),             # CUDA-core kernel
    (512, 256, torch.float32, "auto", (16, 12), True, (0,)),             # W % 8 != 0
    (512, 257, torch.float32, "auto", (16, 16), True, (0,)),             # K blocks
])
def test_pixel_losses_fake_sign_codes_follow_the_route(D, K, x_dtype, precision, hw, need_grad, codes):
    from rangeclip_b200 import ops
    x, t, log_tau, y, w = _args(D, K, x_dtype, hw)
    out = torch.ops.rangeclip.pixel_losses(x, t, log_tau, y, w, need_grad, False, precision, None, None, None)
    assert tuple(out[5].shape) == codes and out[5].dtype == torch.int32
    route = ops._infonce_plan(x, K, False, precision, 1, need_grad)
    if need_grad:
        assert out[2].dtype == (torch.bfloat16 if route == "bf16" else x_dtype) and tuple(out[2].shape) == tuple(x.shape)


@pytest.mark.parametrize("D,K,need_dt,precision,rep,dev", [
    (128, 256, False, "kblocked", 1, False),
    (512, 257, False, "bf16", 1, False),
    (512, 256, True, "bf16", 1, True),         # device parameters with a trainable t_norm: no kernel returns dText there
    (512, 256, False, "fp32", 4, False),
])
def test_fakes_raise_where_no_kernel_takes_the_call(D, K, need_dt, precision, rep, dev):
    x, t, log_tau, y, w = _args(D, K, torch.bfloat16, rep=rep)
    k_dev = torch.empty(4, device="meta", dtype=torch.int32) if dev else None
    with pytest.raises(RuntimeError, match="no kernel covers"):
        torch.ops.rangeclip.infonce(x, t, log_tau, y, w, True, need_dt, precision, rep, None, None, k_dev)
    if rep == 1:
        with pytest.raises(RuntimeError, match="no kernel covers"):
            torch.ops.rangeclip.pixel_losses(x, t, log_tau, y, w, True, need_dt, precision, None, None, k_dev)
