"""Exact-arithmetic tests of the memory-bound kernels of the training step: masked pooling, smoothness (TV-L1) forward and
backward with the fp32 sign codes, row normalisation, and the sampling / scaling / text helpers.

The inputs come from oracle/exact_inputs.py: values on a dyadic grid, power-of-two scales and counts, rows of
power-of-two norm.  Every result these kernels form is then exact whatever order they sum in, so each output is compared
with the float64 reference by ``torch.equal`` at every element.  The only bounds are the textbook forward-error bounds of
the random-row normalisation tests and of pooling backward with arbitrary counts, checked per element.  Each case also
asserts, by name from ``torch.profiler``, the kernel it is meant to reach, so that a dispatch change cannot quietly
move it onto another path.  Unaligned bases come from calling the C ABI on a view at an element offset of 1 (the Python
wrappers make every tensor contiguous, which never yields one).

Dispatch table (host conditions -> kernel -> the test that reaches it)

rc_pool_fwd (pool.cu); vec = HW % 8 == 0 and x 16-byte aligned
  vec, f32                          pool_fwd_kernel<float>                 test_pool_forward[vec-f32-*]
  vec, bf16                         pool_fwd_kernel<__nv_bfloat16>         test_pool_forward[vec-bf16-*]
    merged / unmerged chunk pairs (W = 256, identical row pairs), odd chunk count (H odd at W = 256), partial last chunk
    (HW % 256 != 0), mixed lanes, D % 64 != 0: all inside the two kernels above, in vec-*-structured / vec-*-partial
  HW % 8 != 0, f32 / bf16           pool_fwd_generic_kernel<float / bf16>  test_pool_forward[generic-*-hw]
  unaligned x, f32 / bf16           pool_fwd_generic_kernel<float / bf16>  test_pool_forward[generic-*-unaligned]
  every call (mean = sum / count)   pool_finish_kernel                     test_pool_forward[*]
rc_pool_bwd (pool.cu); vec_ok = HW % 8 == 0 and dx 16-byte aligned; one kernel per dtype, three branches
  uniform lane, vec_ok, D % 4 == 0, g aligned: 16-byte gather of g       test_pool_backward_exact[gather-*]
  mixed lane or D % 4 != 0 or unaligned g, vec_ok: scalar gather          test_pool_backward_exact[scalar-*]
  not vec_ok (HW % 8 != 0: the tail p0 + 8 > HW; unaligned dx): per element test_pool_backward_exact[tail-*, dxoff-*]
  pool_bwd_kernel<float> / <__nv_bfloat16>, accumulate over four maps    test_pool_backward_exact[*-4maps]
rc_tv_fwd (tv.cu); vec = W % 8 == 0 and x 16-byte aligned; TH = tv_tile_rows(...) < 1 -> element-wise kernel
  vec, f32                          tv_fwd_vec_kernel<float>               test_tv_forward_backward[f32-vec-*]
  vec, bf16 (66 KB opt-in tiles)    tv_fwd_bf16_walk_kernel                test_tv_forward_backward[bf16-vec-*]
  not vec, f32 / bf16               tv_fwd_kernel<float / bf16>            test_tv_forward_backward[*-scalar-*, *-unaligned]
  TH < 1, f32 / bf16                tv_fwd_direct_kernel<float / bf16>     test_tv_forward_backward[*-direct]
  (tv_load_rows' 16-byte branch is unreachable from tv_fwd_kernel: it runs only when the host found x unaligned or
  W % 8 != 0, the same condition the kernel re-tests)
rc_tv_bwd / rc_tv_bwd_from (tv.cu); vec additionally needs dx and dx_in 16-byte aligned
  vec, bf16 x (dx_in bf16 or none)  tv_bwd_bf16x2_kernel                   test_tv_forward_backward[bf16-vec-*]
  vec, f32 x, dx_in f32 / none      tv_bwd_vec_kernel<float, float>        test_tv_forward_backward[f32-vec-*]
  vec, f32 x, dx_in bf16            tv_bwd_vec_kernel<float, bf16>         test_tv_forward_backward[f32-vec-*-bf16in]
  not vec                           tv_bwd_kernel<float, float / bf16>, <bf16, bf16>   [*-scalar-*], [*-unaligned]
  x aligned, dx_in unaligned        tv_bwd_kernel<float, float> with 16-byte row loads test_tv_backward_unaligned_dx_in
  TH < 1                            tv_bwd_direct_kernel<float, float / bf16>, <bf16, bf16>   [*-direct]
  in-place accumulate (rc_tv_bwd)   tv_bwd_vec_kernel<float, float>        test_tv_backward_in_place
  bf16 x with f32 dx_in             rejected (RC_ERR_UNSUPPORTED)          test_tv_backward_rejects_f32_dx_in_under_bf16_x
rc_infonce_prepass_tv (infonce.cu) -> rc_tv_bwd_codes (tv.cu); fp32 x, W % 8 == 0
  with codes / without              rownorm_tv_kernel<4, true / false>     test_tv_sign_codes[*], test_prepass_tv_without_codes
  dx_in f32 or none / bf16          tv_bwd_codes_kernel<float / bf16>      test_tv_sign_codes[*]
    W / 8 divides 32 (several rows per warp, W = 8), W / 8 = 25 (idle lanes), W / 8 = 33 (a lane walks two groups),
    H % 4 != 0 (short strips): test_tv_sign_codes[w8-*, w200-*, w264-*]
rc_normalize_rows_fwd / _bwd, rc_tv_normalize_bwd (rows.cu); HW % 8 == 0 and 32-byte aligned pointers are required
  (no fallback: anything else raises)
  f32 / bf16 x                      normalize_rows_fwd_kernel<float / bf16>      test_normalize_exact, test_normalize_bound
  f32 / bf16 dx                     normalize_rows_bwd_kernel<float / bf16>      test_normalize_exact, test_normalize_bound
  f32 / bf16 dx                     tv_normalize_bwd_kernel<float / bf16>        test_tv_normalize_backward_exact
infonce_simt.cu helpers
  sample_label_count_kernel (C <= 12000; C = 12001 raises)        test_sample_label_counts, test_sample_label_counts_limit
  rand_idx: sample_count_kernel + sample_map_kernel; none: map only   test_sample_weights
  weight_sum_kernel (with / without the y mask)                     test_weight_sum
  scale_to_kernel<TI, TO>, four pairs, vector body / unaligned tail test_scale_to
  text_prepare_kernel                                               test_text_prepare
"""
import numpy as np
import pytest
import torch

from oracle import exact_inputs as E

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32


def dev():
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _kernels(fn):
    """(fn(), names of the CUDA kernels it launched, spaces removed)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.key.replace(" ", "") for e in prof.key_averages()]


def _ran(names, *want, absent=()):
    for w in want:
        assert any(w.replace(" ", "") in n for n in names), (w, names)
    for w in absent:
        assert not any(w.replace(" ", "") in n for n in names), (w, names)


def _offset_copy(t: torch.Tensor, offset: int) -> torch.Tensor:
    """A contiguous copy of ``t`` whose storage starts ``offset`` elements into a larger buffer (unaligned for offset 1)."""
    buf = torch.zeros(t.numel() + offset + 8, device=t.device, dtype=t.dtype)
    v = buf[offset:offset + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def _t(a, dtype=F32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(dtype).to(dev())


def _equal(got: torch.Tensor, ref, what=""):
    """Bit-identical to the float64 reference rounded to got's dtype (the builders make that rounding exact)."""
    r = torch.as_tensor(np.ascontiguousarray(ref, dtype=np.float64)).to(got.dtype)
    g = got.detach().cpu()
    if not torch.equal(g, r):
        bad = (g.double() != r.double()).nonzero()
        raise AssertionError(f"{what}: {bad.shape[0]} elements differ, first at {bad[:4].tolist()}: "
                             f"{g[tuple(bad[0])].item()} vs {r[tuple(bad[0])].item()}")


def _ulp(v: np.ndarray, dtype) -> np.ndarray:
    """The spacing of ``dtype`` at |v| (normal range)."""
    bits = 8 if dtype == BF16 else 24
    a = np.maximum(np.abs(v), np.finfo(np.float32).tiny)
    return 2.0 ** (np.floor(np.log2(a)) - (bits - 1))


# ----------------------------------------------------------------------------------------------------------------------
# 1. masked pooling
# ----------------------------------------------------------------------------------------------------------------------

def _pool_fwd_raw(x, segs, lut, per_image, n_slots):
    """rc_pool_fwd once per label map on x as given (any base offset), then rc_pool_finish: (sums, counts, means)."""
    from rangeclip_b200 import _lib
    from rangeclip_b200.ops import _dt
    L = _lib.lib()
    B, D = x.shape[0], x.shape[1]
    HW = x[0, 0].numel()
    C = lut.shape[-1]
    s = torch.zeros(n_slots, D, device=dev())
    c = torch.zeros(n_slots, device=dev(), dtype=torch.int32)
    for sg in segs:
        _lib.check(L.rc_pool_fwd(x.data_ptr(), _dt(x), B, D, HW, sg.data_ptr(), lut.data_ptr(), C if per_image else 0, C, n_slots,
                                 s.data_ptr(), c.data_ptr(), _stream()), "rc_pool_fwd")
    sums = s.clone()
    _lib.check(L.rc_pool_finish(s.data_ptr(), c.data_ptr(), n_slots, D, _stream()), "rc_pool_finish")
    return sums, c, s


POOL_FWD = [  # id, B, D, H, W, dtype, per_image lut, label maps, x offset, vector kernel
    ("vec-f32-structured", 2, 65, 6, 256, F32, True, 1, 0, True),
    ("vec-bf16-structured", 2, 130, 7, 256, BF16, False, 1, 0, True),
    ("vec-f32-partial", 3, 1, 13, 40, F32, True, 1, 0, True),
    ("vec-bf16-partial", 1, 200, 5, 104, BF16, True, 1, 0, True),
    ("vec-bf16-4maps", 2, 64, 8, 256, BF16, True, 4, 0, True),
    ("vec-f32-4maps", 2, 130, 4, 64, F32, False, 4, 0, True),
    ("generic-f32-hw", 2, 65, 5, 13, F32, True, 1, 0, False),
    ("generic-bf16-hw", 2, 130, 3, 11, BF16, False, 1, 0, False),
    ("generic-bf16-hw-4maps", 2, 3, 7, 9, BF16, True, 4, 0, False),
    ("generic-f32-unaligned", 2, 65, 6, 256, F32, True, 1, 1, False),
    ("generic-bf16-unaligned", 1, 130, 3, 64, BF16, False, 1, 1, False),
]


def pool_case(B, D, H, W, per_image, n_maps, seed):
    """(x float64 [B, D, HW] of k / 8, label maps, lut, n_slots)."""
    rng = np.random.default_rng(seed)
    C, n_slots = 23, 9
    x = E.dyadic(rng, (B, D, H * W))
    segs = [E.pool_segmentation(rng, B, H, W, C) for _ in range(n_maps)]
    lut = E.pool_lut(rng, B, C, n_slots, per_image)
    return x, segs, lut, n_slots


@pytest.mark.parametrize("case", POOL_FWD, ids=[c[0] for c in POOL_FWD])
def test_pool_forward(case):
    """Slot sums and counts bit-identical to fp64, means equal to the fp32 quotient, an absent slot a zero row."""
    name, B, D, H, W, dtype, per_image, n_maps, off, vec = case
    x64, segs, lut, n_slots = pool_case(B, D, H, W, per_image, n_maps, seed=len(name) * 100 + D + H + W)
    ref_sums, ref_cnt, ref_mean = E.pool_reference(x64, segs, lut, per_image, n_slots)
    assert ref_cnt[-1] == 0
    x = _offset_copy(_t(x64, dtype).view(B, D, H, W), off)
    sg = [_t(s, torch.int64) for s in segs]
    (sums, cnt, mean), names = _kernels(lambda: _pool_fwd_raw(x, sg, _t(lut, torch.int32), per_image, n_slots))
    tn = "float" if dtype == F32 else "__nv_bfloat16"
    want, other = (f"pool_fwd_kernel<{tn}>", f"pool_fwd_generic_kernel<{tn}>")[::1 if vec else -1]
    _ran(names, want, "pool_finish_kernel", absent=(other,))
    assert torch.equal(cnt.cpu(), torch.as_tensor(ref_cnt, dtype=torch.int32))
    _equal(sums, ref_sums, "sums")
    assert torch.equal(mean.cpu(), torch.from_numpy(ref_mean))


def test_masked_pool_op_and_autograd():
    """The registered operator on a bf16 tensor (means stored in bf16) and its autograd backward with the real, arbitrary
    counts: every element within 2 bf16 ulp of g / c in fp64."""
    from rangeclip_b200 import ops
    rng = np.random.default_rng(5)
    B, D, H, W = 2, 68, 6, 256
    x64, segs, lut, n_slots = pool_case(B, D, H, W, True, 1, seed=7)
    _, ref_cnt, ref_mean = E.pool_reference(x64, segs, lut, True, n_slots)
    x = _t(x64, BF16).view(B, D, H, W).requires_grad_(True)
    mean = ops.masked_pool(x, _t(segs[0], torch.int64).view(B, H, W), _t(lut, torch.int32), True, n_slots)
    assert torch.equal(mean.detach().cpu(), torch.from_numpy(ref_mean).to(BF16))
    g = E.dyadic(rng, (n_slots, D))
    mean.backward(_t(g, BF16))
    ref = E.pool_backward_reference(g, ref_cnt, segs, lut, True, D)[-1].reshape(B, D, H, W)
    err = np.abs(x.grad.double().cpu().numpy() - ref)
    assert (err <= 2 * _ulp(ref, BF16)).all(), err.max()


POOL_BWD = [  # id, B, D, H, W, dtype, per_image, maps, dx offset, g offset
    ("gather-f32", 2, 64, 6, 256, F32, True, 1, 0, 0),
    ("gather-bf16", 2, 128, 4, 64, BF16, False, 1, 0, 0),
    ("scalar-f32-d65", 2, 65, 6, 256, F32, True, 1, 0, 0),
    ("scalar-bf16-d130", 1, 130, 5, 104, BF16, True, 1, 0, 0),
    ("scalar-f32-goff", 2, 64, 3, 64, F32, True, 1, 0, 1),
    ("tail-f32-hw65", 2, 65, 5, 13, F32, True, 1, 0, 0),
    ("tail-bf16-hw33", 2, 8, 3, 11, BF16, False, 1, 0, 0),
    ("dxoff-f32", 1, 64, 4, 64, F32, True, 1, 1, 0),
    ("dxoff-bf16", 2, 65, 3, 64, BF16, True, 1, 1, 0),
    ("gather-bf16-4maps", 2, 64, 8, 256, BF16, True, 4, 0, 0),
    ("scalar-f32-4maps", 2, 65, 4, 64, F32, False, 4, 0, 0),
    ("tail-bf16-4maps", 1, 12, 7, 9, BF16, True, 4, 0, 0),
]


def pool_bwd_case(case):
    """(label maps, lut, g, power-of-two counts with slot 0 at count 0, dx after each map in fp64)."""
    name, B, D, H, W, dtype, per_image, n_maps, dx_off, g_off = case
    rng = np.random.default_rng(len(name) * 31 + D + H + W)
    C, n_slots = 23, 9
    segs = [E.pool_segmentation(rng, B, H, W, C) for _ in range(n_maps)]
    lut = E.pool_lut(rng, B, C, n_slots, per_image)
    g64, cnt64 = E.pool_backward_inputs(rng, n_slots, D, n_maps)
    cnt64[0] = 0
    return segs, lut, g64, cnt64, E.pool_backward_reference(g64, cnt64, segs, lut, per_image, D)


@pytest.mark.parametrize("case", POOL_BWD, ids=[c[0] for c in POOL_BWD])
def test_pool_backward_exact(case):
    """dx = sum over the label maps of g[slot] / count[slot], power-of-two counts and dyadic g: bit-identical in the output
    dtype, the four-map bf16 accumulation included; a slot with count 0 contributes nothing."""
    from rangeclip_b200 import _lib
    name, B, D, H, W, dtype, per_image, n_maps, dx_off, g_off = case
    C, n_slots = 23, 9
    segs, lut, g64, cnt64, refs = pool_bwd_case(case)
    ref = refs[-1]
    g = _offset_copy(_t(g64), g_off)
    cnt = _t(cnt64, torch.int32)
    lt = _t(lut, torch.int32)
    sg = [_t(s, torch.int64) for s in segs]
    dx = _offset_copy(torch.full((B, D, H, W), 7.0, device=dev(), dtype=dtype), dx_off)

    def run():
        for i, s in enumerate(sg):
            _lib.check(_lib.lib().rc_pool_bwd(g.data_ptr(), cnt.data_ptr(), B, D, H * W, s.data_ptr(), lt.data_ptr(),
                                              C if per_image else 0, C, n_slots, dx.data_ptr(),
                                              _lib.RC_F32 if dtype == F32 else _lib.RC_BF16, 1 if i else 0, _stream()),
                       "rc_pool_bwd")
    _, names = _kernels(run)
    _ran(names, "pool_bwd_kernel<float>" if dtype == F32 else "pool_bwd_kernel<__nv_bfloat16>")
    _equal(dx.reshape(B, D, H * W), ref, "dx")


# ----------------------------------------------------------------------------------------------------------------------
# 2. smoothness
# ----------------------------------------------------------------------------------------------------------------------

TV = [  # id, B, D, H, W, dtype, x offset, forward kernel, backward kernel (x dtype, dx_in dtype substituted)
    ("f32-vec-seam", 2, 3, 33, 64, F32, 0, "tv_fwd_vec_kernel<float>", "tv_bwd_vec_kernel<float,{i}>"),
    ("f32-vec-w8", 1, 2, 70, 8, F32, 0, "tv_fwd_vec_kernel<float>", "tv_bwd_vec_kernel<float,{i}>"),
    ("f32-vec-h1", 3, 5, 1, 64, F32, 0, "tv_fwd_vec_kernel<float>", "tv_bwd_vec_kernel<float,{i}>"),
    ("f32-vec-planes", 4, 40, 9, 16, F32, 0, "tv_fwd_vec_kernel<float>", "tv_bwd_vec_kernel<float,{i}>"),
    ("bf16-vec-optin", 1, 2, 128, 256, BF16, 0, "tv_fwd_bf16_walk_kernel", "tv_bwd_bf16x2_kernel"),
    ("bf16-vec-seam", 1, 2, 129, 256, BF16, 0, "tv_fwd_bf16_walk_kernel", "tv_bwd_bf16x2_kernel"),
    ("bf16-vec-bwdseam", 1, 3, 94, 256, BF16, 0, "tv_fwd_bf16_walk_kernel", "tv_bwd_bf16x2_kernel"),
    ("bf16-vec-w8", 2, 2, 300, 8, BF16, 0, "tv_fwd_bf16_walk_kernel", "tv_bwd_bf16x2_kernel"),
    ("bf16-vec-h1", 2, 3, 1, 24, BF16, 0, "tv_fwd_bf16_walk_kernel", "tv_bwd_bf16x2_kernel"),
    ("f32-scalar-w13", 2, 3, 33, 13, F32, 0, "tv_fwd_kernel<float>", "tv_bwd_kernel<float,{i}>"),
    ("f32-scalar-w1", 1, 2, 40, 1, F32, 0, "tv_fwd_kernel<float>", "tv_bwd_kernel<float,{i}>"),
    ("bf16-scalar-w20", 2, 2, 35, 20, BF16, 0, "tv_fwd_kernel<__nv_bfloat16>", "tv_bwd_kernel<__nv_bfloat16,{i}>"),
    ("bf16-scalar-h1w1", 2, 3, 1, 1, BF16, 0, "tv_fwd_kernel<__nv_bfloat16>", "tv_bwd_kernel<__nv_bfloat16,{i}>"),
    ("f32-unaligned", 1, 3, 33, 64, F32, 1, "tv_fwd_kernel<float>", "tv_bwd_kernel<float,{i}>"),
    ("bf16-unaligned", 1, 2, 20, 256, BF16, 1, "tv_fwd_kernel<__nv_bfloat16>", "tv_bwd_kernel<__nv_bfloat16,{i}>"),
    ("f32-direct", 1, 2, 3, 6128, F32, 0, "tv_fwd_direct_kernel<float>", "tv_bwd_direct_kernel<float,{i}>"),
    ("bf16-direct", 1, 1, 3, 17032, BF16, 0, "tv_fwd_direct_kernel<__nv_bfloat16>", "tv_bwd_direct_kernel<__nv_bfloat16,{i}>"),
]
TV_MODES = ["none", "same", "bf16in"]
TV_PARAMS = [pytest.param(c, m, id=f"{c[0]}-{m}") for c in TV for m in TV_MODES if not (m == "bf16in" and c[5] == BF16)]
SH, SV = 2.0 ** -4, 2.0 ** -5


def _tv_call(x, scale, dx_in, ds, out, fn="rc_tv_bwd_from"):
    from rangeclip_b200 import _lib
    from rangeclip_b200.ops import _dt
    B, D, H, W = x.shape
    L = _lib.lib()
    if fn == "rc_tv_fwd":
        _lib.check(L.rc_tv_fwd(x.data_ptr(), _dt(x), B * D, H, W, out.data_ptr(), _stream()), fn)
    elif dx_in is None:
        _lib.check(L.rc_tv_bwd(x.data_ptr(), _dt(x), B * D, H, W, scale.data_ptr(), out.data_ptr(), 0, None, _stream()), fn)
    else:
        _lib.check(L.rc_tv_bwd_from(x.data_ptr(), _dt(x), B * D, H, W, scale.data_ptr(), dx_in.data_ptr(), _dt(dx_in),
                                    None if ds is None else ds.data_ptr(), out.data_ptr(), _stream()), fn)


def tv_case(case, mode):
    """(x, dx_in or None, ds, dx_in dtype or None) float64, for a TV case and dx_in mode."""
    name, B, D, H, W, dtype = case[:6]
    rng = np.random.default_rng(len(name) * 7 + B + D + H + W)
    x64 = E.tv_input(rng, B, D, H, W)
    if mode == "none":
        return x64, None, 1.0, None
    return x64, E.dyadic(rng, x64.shape), float(2.0 ** rng.integers(-2, 2)), BF16 if mode == "bf16in" else dtype


@pytest.mark.parametrize("case,mode", TV_PARAMS)
def test_tv_forward_backward(case, mode):
    """tv_sums bit-identical to fp64; dx = ds * dx_in + sh * (sign differences) + sv * (...) bit-identical to the closed
    form (sign(0) = 0) with s_h = 2^-4, s_v = 2^-5, ds a power of two and dyadic dx_in."""
    name, B, D, H, W, dtype, off, kf, kb = case
    x64, dx_in64, ds64, in_dtype = tv_case(case, mode)
    x = _offset_copy(_t(x64, dtype), off)
    sums = torch.zeros(2, device=dev(), dtype=torch.float64)
    _, names = _kernels(lambda: _tv_call(x, None, None, None, sums, "rc_tv_fwd"))
    _ran(names, kf)
    assert torch.equal(sums.cpu(), torch.from_numpy(E.tv_sums_reference(x64))), (sums.cpu(), E.tv_sums_reference(x64))

    scale = torch.tensor([SH, SV], device=dev())
    dx_in = None if dx_in64 is None else _t(dx_in64, in_dtype)
    ds = None if dx_in64 is None else torch.tensor([ds64], device=dev())
    out = torch.full(x.shape, 3.0, device=dev(), dtype=dtype)
    _, names = _kernels(lambda: _tv_call(x, scale, dx_in, ds, out))
    tn = {F32: "float", BF16: "__nv_bfloat16", None: "float" if dtype == F32 else "__nv_bfloat16"}
    _ran(names, kb.format(i=tn[in_dtype]))
    _equal(out, E.tv_grad_reference(x64, SH, SV, dx_in64, ds64), "dx")


def test_tv_backward_unaligned_dx_in():
    """x aligned, dx_in at an odd element offset: the scalar tiled kernel, filling its tile with 16-byte loads of x."""
    rng = np.random.default_rng(3)
    x64 = E.tv_input(rng, 2, 3, 33, 64)
    dx_in64 = E.dyadic(rng, x64.shape)
    x = _t(x64)
    dx_in = _offset_copy(_t(dx_in64), 1)
    out = torch.empty_like(x)
    ds = torch.tensor([0.5], device=dev())
    _, names = _kernels(lambda: _tv_call(x, torch.tensor([SH, SV], device=dev()), dx_in, ds, out))
    _ran(names, "tv_bwd_kernel<float,float>", absent=("tv_bwd_vec_kernel",))
    _equal(out, E.tv_grad_reference(x64, SH, SV, dx_in64, 0.5), "dx")


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_tv_backward_in_place(dtype):
    """rc_tv_bwd with accumulate = 1: dx = dx_scale * dx + TV' in place."""
    from rangeclip_b200 import _lib
    from rangeclip_b200.ops import _dt
    rng = np.random.default_rng(4)
    B, D, H, W = 1, 3, 40, 64
    x64 = E.tv_input(rng, B, D, H, W)
    dx64 = E.dyadic(rng, x64.shape)
    x, dx = _t(x64, dtype), _t(dx64, dtype)
    scale, ds = torch.tensor([SH, SV], device=dev()), torch.tensor([2.0], device=dev())
    _, names = _kernels(lambda: _lib.check(_lib.lib().rc_tv_bwd(x.data_ptr(), _dt(x), B * D, H, W, scale.data_ptr(), dx.data_ptr(),
                                                                1, ds.data_ptr(), _stream()), "rc_tv_bwd"))
    _ran(names, "tv_bwd_vec_kernel<float,float>" if dtype == F32 else "tv_bwd_bf16x2_kernel")
    _equal(dx, E.tv_grad_reference(x64, SH, SV, dx64, 2.0), "dx")


def test_tv_backward_rejects_f32_dx_in_under_bf16_x():
    from rangeclip_b200 import ops
    x = torch.zeros(1, 1, 8, 8, device=dev(), dtype=BF16)
    with pytest.raises(RuntimeError, match="f32 dx_in"):
        ops.tv_backward(x, torch.tensor([SH, SV], device=dev()), torch.zeros(1, 1, 8, 8, device=dev()))


def _prepass_tv(x, want_codes=True):
    """rc_infonce_prepass_tv on an fp32 [B, D, H, W] x: (tv_sums, codes or None, workspace bf16 copy of x)."""
    from rangeclip_b200 import _lib
    L = _lib.lib()
    B, D, H, W = x.shape
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, H * W, 0, _lib.RC_F32))
    ws = torch.zeros(ws_bytes + 256, device=dev(), dtype=torch.uint8)
    sums = torch.zeros(2, device=dev(), dtype=torch.float64)
    codes = torch.zeros(B, D, H, W // 8, device=dev(), dtype=torch.int32) if want_codes else None
    _lib.check(L.rc_infonce_prepass_tv(x.data_ptr(), B, D, H, W, ws.data_ptr(), ws_bytes, sums.data_ptr(),
                                       None if codes is None else codes.data_ptr(), _stream()), "rc_infonce_prepass_tv")
    base = (-ws.data_ptr()) % 256
    M = B * H * W
    xb_off = base + (M * 4 + 255) // 256 * 256
    xb = ws[xb_off:xb_off + M * D * 2].view(BF16).view(B, D, H, W)
    return sums, codes, xb


CODES = [  # id, B, D, H, W, input kind
    ("w8-h10", 2, 3, 10, 8, "dyadic"),
    ("w200-h7", 1, 2, 7, 200, "dyadic"),
    ("w264-h9", 1, 2, 9, 264, "dyadic"),
    ("w256-h12", 2, 1, 12, 256, "dyadic"),
    ("w64-edges", 1, 2, 6, 64, "edges"),
    ("w8-edges", 1, 3, 5, 8, "edges"),
]
CODE_PARAMS = [pytest.param(c, m, id=f"{c[0]}-{m}") for c in CODES for m in ("none", "f32in", "bf16in")]


def codes_case(case, mode):
    """(fp32 x, dx_in float64 or None, ds) for a sign-code case."""
    name, B, D, H, W, kind = case
    rng = np.random.default_rng(len(name) + B * D * H * W)
    x32 = E.tv_input(rng, B, D, H, W).astype(np.float32) if kind == "dyadic" else E.tv_sign_edge_input(B, D, H, W)
    if mode == "none":
        return x32, None, 1.0
    return x32, E.dyadic(rng, x32.shape), 0.25


@pytest.mark.parametrize("case,mode", CODE_PARAMS)
def test_tv_sign_codes(case, mode):
    """The fused fp32 pre-pass: code words equal to the documented layout of the fp32 signs (+0 vs -0 is no difference;
    neighbours equal only after bf16 rounding are +-1; tiny and huge differences keep their sign), tv_sums bit-identical,
    the bf16 copy equal to x.to(bf16); tv_bwd_codes bit-identical to the closed form, not just to tv_backward."""
    from rangeclip_b200 import ops
    kind = case[5]
    x32, dx_in64, ds64 = codes_case(case, mode)
    x = _t(x32)
    (sums, codes, xb), names = _kernels(lambda: _prepass_tv(x))
    _ran(names, "rownorm_tv_kernel")
    assert torch.equal(codes.cpu(), torch.from_numpy(E.tv_codes_reference(x32)))
    assert torch.equal(xb.cpu(), x.cpu().to(BF16))
    if kind == "dyadic":
        assert torch.equal(sums.cpu(), torch.from_numpy(E.tv_sums_reference(x32)))
    dx_in = None if dx_in64 is None else _t(dx_in64, BF16 if mode == "bf16in" else F32)
    ds = None if dx_in64 is None else torch.tensor([ds64], device=dev())
    out, names = _kernels(lambda: ops.tv_backward_codes(codes, torch.tensor([SH, SV], device=dev()), dx_in, ds))
    _ran(names, "tv_bwd_codes_kernel<__nv_bfloat16>" if mode == "bf16in" else "tv_bwd_codes_kernel<float>")
    _equal(out, E.tv_grad_reference(x32, SH, SV, dx_in64, ds64), "dx")


def test_prepass_tv_without_codes():
    rng = np.random.default_rng(8)
    x32 = E.tv_input(rng, 2, 3, 11, 40).astype(np.float32)
    (sums, _, xb), names = _kernels(lambda: _prepass_tv(_t(x32), want_codes=False))
    _ran(names, "rownorm_tv_kernel")
    assert torch.equal(sums.cpu(), torch.from_numpy(E.tv_sums_reference(x32)))
    assert torch.equal(xb.cpu(), torch.from_numpy(x32).to(BF16))


# ----------------------------------------------------------------------------------------------------------------------
# 3. row normalisation
# ----------------------------------------------------------------------------------------------------------------------

NORM = [  # B, D, H, W, dtype
    (2, 256, 3, 8, F32), (1, 256, 1, 64, BF16), (3, 65, 2, 16, F32), (2, 16, 4, 24, BF16), (1, 1, 2, 8, F32),
]


def norm_case(B, D, H, W):
    """(x with rows of power-of-two norm and some zero rows, dyadic g) float64; g is 0 on the zero rows, whose
    dx = g / 1e-12 is not exact."""
    rng = np.random.default_rng(B * 100 + D + H + W)
    x64 = E.exact_rows(rng, B, D, H, W, zero_frac=0.1)
    return x64, E.dyadic(rng, x64.shape) * (x64 != 0).any(1, keepdims=True)


@pytest.mark.parametrize("B,D,H,W,dtype", NORM)
def test_normalize_exact(B, D, H, W, dtype):
    """Rows of power-of-two norm (and zero rows): x_hat and inv bit-identical; the backward with dyadic g bit-identical to
    the single rounding of the exact fp64 result."""
    from rangeclip_b200 import ops
    x64, g64 = norm_case(B, D, H, W)
    xhat64, inv64 = E.normalize_reference(x64)
    x = _t(x64, dtype)
    (xhat, inv), names = _kernels(lambda: ops.normalize_rows_raw(x))
    _ran(names, "normalize_rows_fwd_kernel<float>" if dtype == F32 else "normalize_rows_fwd_kernel<__nv_bfloat16>")
    _equal(xhat, xhat64, "x_hat")
    _equal(inv, inv64, "inv")
    dx, names = _kernels(lambda: ops.normalize_rows_backward(xhat, _t(g64), inv, dtype))
    _ran(names, "normalize_rows_bwd_kernel<float>" if dtype == F32 else "normalize_rows_bwd_kernel<__nv_bfloat16>")
    _equal(dx, E.normalize_backward_reference(xhat64, g64, inv64)[0], "dx")


def _norm_bounds(x64, xhat, inv, g64, dxk, D, dtype):
    ref, absdot = E.normalize_backward_reference(xhat, g64, inv)
    invb = np.asarray(inv, np.float64).reshape((x64.shape[0], 1) + x64.shape[2:])
    e32 = (2 * D + 8) * 2.0 ** -24 * (np.abs(g64) + np.abs(xhat) * absdot) * invb
    return np.abs(dxk - ref) <= e32 + 0.5 * _ulp(np.abs(ref) + e32, dtype)


@pytest.mark.parametrize("B,D,H,W,dtype", [(2, 256, 4, 8, F32), (1, 33, 1, 24, BF16), (3, 512, 2, 16, BF16), (1, 7, 3, 8, F32)])
def test_normalize_bound(B, D, H, W, dtype):
    """Random rows (a few zero rows): forward within (D + 4) 2^-24 relative per element; backward within
    (2D + 8) 2^-24 (|g_j| + |x_hat_j| sum |x_hat g|) inv + half an ulp of the output dtype, per element; zero rows also
    against F.normalize's autograd."""
    from rangeclip_b200 import ops
    g = torch.Generator().manual_seed(B + D + H + W)
    x = torch.randn(B, D, H, W, generator=g).to(dtype)
    x[:, :, 0, :2] = 0
    x64 = x.double().numpy()
    (xhat, inv), names = _kernels(lambda: ops.normalize_rows_raw(x.to(dev())))
    xhat64, inv64 = E.normalize_reference(x64)
    assert (np.abs(xhat.cpu().double().numpy() - xhat64) <= (D + 4) * 2.0 ** -24 * np.abs(xhat64)).all()
    gin = torch.randn(B, D, H, W, generator=g)
    dx = ops.normalize_rows_backward(xhat, gin.to(dev()), inv, dtype)
    ok = _norm_bounds(x64, xhat.cpu().double().numpy(), inv.cpu().double().numpy(), gin.double().numpy(),
                      dx.cpu().double().numpy(), D, dtype)
    assert ok.all(), np.argwhere(~ok)[:4]
    # zero rows through PyTorch's own F.normalize autograd: g / 1e-12
    xt = x.float().clone().requires_grad_(True)
    torch.nn.functional.normalize(xt, dim=1).backward(gin)
    zr = xt.grad[:, :, 0, :2].double().numpy()
    got = dx[:, :, 0, :2].cpu().double().numpy()
    e32 = (2 * D + 8) * 2.0 ** -24 * np.abs(zr)
    assert (np.abs(got - zr) <= e32 + 0.5 * _ulp(np.abs(zr) + e32, dtype)).all()


TVN = [(2, 256, 5, 16, F32), (1, 256, 7, 8, BF16), (3, 16, 1, 32, F32), (2, 65, 3, 8, BF16)]


@pytest.mark.parametrize("B,D,H,W,dtype", TVN)
def test_tv_normalize_backward_exact(B, D, H, W, dtype):
    """rc_tv_normalize_bwd with s_h = 2^-4, s_v = 2^-5 on exactly normalised rows: bit-identical to the single rounding
    of the fp64 composition of the closed-form TV gradient and the normalisation backward."""
    from rangeclip_b200 import ops
    x64 = E.exact_rows(np.random.default_rng(B * 10 + D + H + W), B, D, H, W)
    xhat64, inv64 = E.normalize_reference(x64)
    xhat, inv = _t(xhat64), _t(inv64)
    dx, names = _kernels(lambda: ops.tv_normalize_backward(xhat, inv, torch.tensor([SH, SV], device=dev()), dtype))
    _ran(names, "tv_normalize_bwd_kernel<float>" if dtype == F32 else "tv_normalize_bwd_kernel<__nv_bfloat16>")
    _equal(dx, E.tv_normalize_backward_reference(xhat64, inv64, SH, SV), "dx")


# ----------------------------------------------------------------------------------------------------------------------
# 4. sampling and helpers
# ----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("B,HW,n,C,draws", [(3, 600, 1000, 50, True), (2, 777, 0, 50, False), (2, 4096, 400000, 300, True),
                                            (1, 5000, 3000, 12000, True)])
def test_sample_label_counts(B, HW, n, C, draws):
    """Histogram of the drawn pixels' labels against np.bincount: duplicate draws, draws outside [0, HW), labels < 0 and
    >= C, label 0 counted, rand_idx = None, a grid-stride loop that wraps, and C = 12000 (the shared-memory limit)."""
    from rangeclip_b200 import ops
    rng = np.random.default_rng(B + HW + n + C)
    seg = rng.integers(-3, C + 3, size=(B, HW))
    seg[:, :10] = 0
    r = E.sample_draws(rng, B, HW, n) if draws else None
    counts, names = _kernels(lambda: ops.sample_label_counts(_t(seg, torch.int64), None if r is None else _t(r, torch.int64), C))
    _ran(names, "sample_label_count_kernel")
    assert torch.equal(counts.cpu(), torch.from_numpy(E.sample_label_counts_reference(seg, r, C)).to(torch.int32))


def test_sample_label_counts_limit():
    from rangeclip_b200 import ops
    seg = torch.zeros(1, 64, device=dev(), dtype=torch.int64)
    with pytest.raises(RuntimeError, match="shared-memory histogram"):
        ops.sample_label_counts(seg, None, 12001)


@pytest.mark.parametrize("draws", [True, False])
def test_sample_weights(draws):
    """w = draw multiplicity (a few hundred draws of one pixel), y = label_map[seg] for 0 < seg < C with -1 entries in the
    map, w = 0 wherever y < 0."""
    from rangeclip_b200 import ops
    rng = np.random.default_rng(11)
    B, HW, C = 2, 48 * 64, 40
    seg = rng.integers(-2, C + 2, size=(B, HW))
    lm = rng.integers(0, 30, size=C).astype(np.int32)
    lm[rng.random(C) < 0.25] = -1
    r = E.sample_draws(rng, B, HW, 5000) if draws else None
    (w, y), names = _kernels(lambda: ops.sample_weights(_t(seg, torch.int64), None if r is None else _t(r, torch.int64),
                                                        _t(lm, torch.int32)))
    _ran(names, "sample_map_kernel", *(("sample_count_kernel",) if draws else ()),
         absent=() if draws else ("sample_count_kernel",))
    w_ref, y_ref = E.sample_weights_reference(seg, r, lm)
    assert torch.equal(y.cpu(), torch.from_numpy(y_ref).to(torch.int32))
    _equal(w, w_ref, "w")


@pytest.mark.parametrize("masked", [True, False])
def test_weight_sum(masked):
    """rc_weight_sum on dyadic weights with the y mask: the exact double sum."""
    from rangeclip_b200 import _lib
    rng = np.random.default_rng(12)
    n = 300001
    w64 = rng.integers(0, 4096, size=n) / 64.0
    y = rng.integers(-1, 5, size=n).astype(np.int32)
    wt, yt = _t(w64), _t(y, torch.int32)
    acc = torch.zeros(1, device=dev(), dtype=torch.float64)
    _, names = _kernels(lambda: _lib.check(_lib.lib().rc_weight_sum(wt.data_ptr(), yt.data_ptr() if masked else None, n,
                                                                    acc.data_ptr(), _stream()), "rc_weight_sum"))
    _ran(names, "weight_sum_kernel")
    assert float(acc) == float(w64[y >= 0].sum() if masked else w64.sum())


@pytest.mark.parametrize("ti,to", [(F32, F32), (F32, BF16), (BF16, F32), (BF16, BF16)])
@pytest.mark.parametrize("n,offset,scale", [(1003, 0, 0.3), (1003, 1, 0.3), (4096, 0, None), (17, 1, None)])
def test_scale_to(ti, to, n, offset, scale):
    """out = scale * x in out's dtype: one fp32 product rounded once; vector body, scalar tail, unaligned bases, scale None."""
    from rangeclip_b200 import _lib
    from rangeclip_b200.ops import _dt
    g = torch.Generator().manual_seed(n + offset)
    x = _offset_copy(torch.randn(n, generator=g).to(ti).to(dev()), offset)
    out = _offset_copy(torch.zeros(n, device=dev(), dtype=to), offset)
    s = None if scale is None else torch.tensor([scale], device=dev())
    _, names = _kernels(lambda: _lib.check(_lib.lib().rc_scale_to(x.data_ptr(), _dt(x), out.data_ptr(), _dt(out), n,
                                                                  None if s is None else s.data_ptr(), _stream()), "rc_scale_to"))
    tn = {F32: "float", BF16: "__nv_bfloat16"}
    _ran(names, f"scale_to_kernel<{tn[ti]},{tn[to]}>")
    ref = (x.cpu().float() * (np.float32(scale) if scale is not None else np.float32(1))).to(to)
    assert torch.equal(out.cpu(), ref)


@pytest.mark.parametrize("D,K", [(33, 70), (520, 5), (64, 64)])
def test_text_prepare(D, K):
    """F.normalize(text[idx]): f32 rows within (D + 4) 2^-24 relative per element of fp64; the bf16 copy exactly
    t32.to(bf16) and the transposed copy its transpose; pad rows zero; index -1 a zero row, other out-of-range indices NaN."""
    from rangeclip_b200 import ops
    rng = np.random.default_rng(D + K)
    n_rows = 90
    text = rng.standard_normal((n_rows, D)).astype(np.float32)
    text[3] = 0
    idx = rng.integers(0, n_rows, size=K)
    idx[0] = 3
    if K > 3:
        idx[1], idx[2], idx[3] = -1, n_rows, -2
    (t32, tb, ttb), names = _kernels(lambda: ops.text_prepare(_t(text), _t(idx, torch.int64), True, True))
    _ran(names, "text_prepare_kernel")
    ref = E.text_reference(text, idx)
    got = t32.cpu().double().numpy()
    nan = np.isnan(ref).all(1)
    assert np.isnan(got[nan]).all()
    ok = np.abs(got[~nan] - ref[~nan]) <= (D + 4) * 2.0 ** -24 * np.abs(ref[~nan])
    assert ok.all(), np.argwhere(~ok)[:4]
    Kp = (K + 63) // 64 * 64
    assert tb.shape == (Kp, D) and ttb.shape == (D, Kp)
    valid = ~torch.from_numpy(nan)
    tbc, ttbc = tb.cpu(), ttb.cpu()
    assert torch.equal(tbc[:K][valid], t32.cpu()[valid].to(BF16))
    assert torch.isnan(tbc[:K][~valid].float()).all()
    assert torch.equal(tbc[K:], torch.zeros(Kp - K, D, dtype=BF16))
    assert torch.equal(ttbc.t().nan_to_num(0), tbc.nan_to_num(0)) and torch.equal(ttbc.t().isnan(), tbc.isnan())
