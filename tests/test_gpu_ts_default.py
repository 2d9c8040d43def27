"""Backward launches run the TS-mode InfoNCE kernel (csrc/infonce_ts.cu: softmax tile as a tensor-memory operand of the dX GEMM)
by default; RC_INFONCE_SS_KERNEL selects the CTA-pair SS kernel (csrc/infonce_umma2.cu).  Both round every element the same
way, so dX and the per-row log-sum-exp must agree bit for bit on every schedule corner of the TS kernel (pairs per cluster odd / even, fewer pairs than clusters, a half-empty last
pair, HW not a multiple of 128, D = 256, four targets per row, the K-blocked rounds).  The loss / weight / dlogtau sums are
float64 atomics whose order varies from launch to launch, so they are compared to 1e-12."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TS, SS = 0, 32      # the default (TS), RC_INFONCE_SS_KERNEL


def dev():
    return torch.device("cuda:0")


def n_clusters():
    return torch.cuda.get_device_properties(0).multi_processor_count // 2


def _case(B, D, H, W, K, rep=1, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, H, W, generator=g).to(torch.bfloat16)
    t = torch.nn.functional.normalize(torch.randn(K, D, generator=g), dim=1)
    y = torch.randint(-1, K, (B * H * W, rep) if rep > 1 else (B, H * W), generator=g, dtype=torch.int32)
    w = torch.randint(0, 3, tuple(y.shape), generator=g).float()
    return x.to(dev()), t.to(dev()), y.to(dev()), w.to(dev())


def _run(x, t, y, w, rep, flags):
    from rangeclip_b200 import ops
    r = ops.infonce_raw(x, t, y, w, 1 / 0.07, True, False, "bf16", rep=rep, flags=flags)
    torch.cuda.synchronize()
    return r


def _assert_same(ts, ss):
    assert torch.equal(ts["dx"].view(torch.int16), ss["dx"].view(torch.int16))
    assert torch.equal(ts["lse"].view(torch.int32), ss["lse"].view(torch.int32))
    for k in ("loss_sum", "w_sum", "dlogtau"):
        a, b = float(ts[k]), float(ss[k])
        assert abs(a - b) <= 1e-12 * max(1.0, abs(b)), (k, a, b)


def _tile_shapes():
    """(name, B, D, H, W, K, rep): W = 128 makes one row of pixels one tile, so H sets the tile count."""
    nc = n_clusters()
    return [
        ("headline_one_image", 1, 512, 256, 256, 256, 1),
        ("two_pairs_per_cluster", 1, 512, 4 * nc, 128, 256, 1),
        ("three_pairs_per_cluster", 1, 512, 6 * nc, 128, 256, 1),
        ("odd_even_mix_half_empty_last_pair", 1, 512, 2 * nc + 3, 128, 200, 1),
        ("fewer_pairs_than_clusters", 1, 512, 16, 40, 33, 1),
        ("hw_not_multiple_of_128", 3, 256, 25, 40, 100, 1),
        ("d256", 2, 256, 64, 64, 200, 1),
        ("rep4", 2, 256, 16, 24, 200, 4),
        ("rep4_d512", 1, 512, 64, 64, 256, 4),
    ]


@pytest.mark.parametrize("idx", range(9))
def test_ts_equals_ss_bitwise(idx):
    name, B, D, H, W, K, rep = _tile_shapes()[idx]
    x, t, y, w = _case(B, D, H, W, K, rep, seed=idx)
    _assert_same(_run(x, t, y, w, rep, TS), _run(x, t, y, w, rep, SS))


def test_ts_equals_ss_kblocked_accumulate_round():
    """Round 2 of the K-blocked loss: a block's fwd+bwd launch with the row lse given and the weights kept, ADDING its dX to
    the previous block's (TMA reduce-add stores)."""
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    B, D, H, W, K = 2, 512, 32, 64, 256
    HW, M = H * W, 2 * 32 * 64
    x, t, y, w = _case(B, D, H, W, K, seed=11)
    y, w = y.reshape(-1), w.reshape(-1)
    tb, ttb = ops.text_to_bf16(t)
    lse_in = _run(x, t, y, w, 1, 0)["lse"]
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, _lib.RC_BF16))
    ws = torch.empty(ws_bytes, device=dev(), dtype=torch.uint8)
    st = torch.cuda.current_stream().cuda_stream
    base = torch.randn(B, D, HW, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16).to(dev())
    fl = 1 | ops.RC_INFONCE_KEEP_WEIGHT | ops.RC_INFONCE_LSE_GIVEN | ops.RC_INFONCE_ACCUMULATE_DX
    out = []
    for extra in (TS, SS):
        dx = base.clone()
        acc = torch.zeros(4, device=dev(), dtype=torch.float64)
        acc[3] = w.double().sum()
        lse = lse_in.clone()
        _lib.check(L.rc_infonce_bf16(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), K, y.data_ptr(), w.data_ptr(),
                                     1 / 0.07, lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr(), None,
                                     dx.data_ptr(), None, acc[2:].data_ptr(), ws.data_ptr(), ws_bytes, fl | extra, st), "rc_infonce_bf16")
        torch.cuda.synchronize()
        out.append(dict(dx=dx, lse=lse, loss_sum=acc[0], w_sum=acc[1], dlogtau=acc[2]))
    assert M == y.numel()
    _assert_same(*out)


def test_ts_equals_ss_kblocks_launch():
    """rc_infonce_bf16_kblocks backward (one image, every candidate block of 256 rows in one launch)."""
    from rangeclip_b200 import _lib, ops
    L = _lib.lib()
    D, H, W, K = 256, 32, 64, 300
    HW = H * W
    x, t, y, w = _case(1, D, H, W, K, seed=12)
    y, w = y.reshape(-1), (w.reshape(-1) * (y.reshape(-1) >= 0))
    nb = (K + 255) // 256
    tb_all = torch.zeros(nb * 256, D, device=dev(), dtype=torch.bfloat16)
    tb_all[:K] = t.to(torch.bfloat16)
    ttb_all = tb_all.t().contiguous()
    y_rel = (y[None, :] - 256 * torch.arange(nb, device=dev(), dtype=torch.int32)[:, None]).contiguous()
    w_rep = w[None, :].expand(nb, HW).contiguous()
    lse = torch.logsumexp(torch.randn(HW, 2, generator=torch.Generator().manual_seed(4)), dim=1).to(dev()) + 10.0
    ws_bytes = int(L.rc_infonce_workspace_bytes(1, D, HW, 256, _lib.RC_BF16))
    ws = torch.empty(ws_bytes, device=dev(), dtype=torch.uint8)
    st = torch.cuda.current_stream().cuda_stream
    out = []
    for extra in (TS, SS):
        dxb = torch.empty(nb, D, HW, device=dev(), dtype=torch.bfloat16)
        acc = torch.zeros(4, device=dev(), dtype=torch.float64)
        acc[3] = w.double().sum()
        _lib.check(L.rc_infonce_bf16_kblocks(x.data_ptr(), _lib.RC_BF16, D, HW, tb_all.data_ptr(), ttb_all.data_ptr(), K, nb,
                                             y_rel.data_ptr(), w_rep.data_ptr(), 1 / 0.07, lse.data_ptr(), acc[0:].data_ptr(),
                                             acc[1:].data_ptr(), acc[3:].data_ptr(), None, dxb.data_ptr(), acc[2:].data_ptr(),
                                             ws.data_ptr(), ws_bytes, 1 | ops.RC_INFONCE_LSE_GIVEN | extra, st), "rc_infonce_bf16_kblocks")
        torch.cuda.synchronize()
        out.append(dict(dx=dxb, lse=lse, loss_sum=acc[0], w_sum=acc[1], dlogtau=acc[2]))
    _assert_same(*out)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.key for e in prof.key_averages()]


@pytest.mark.parametrize("flags,kernel,other", [(0, "infonce_ts_kernel", "infonce_umma_pair_kernel"),
                                                 (8, "infonce_ts_kernel", "infonce_umma_pair_kernel"),
                                                 (32, "infonce_umma_pair_kernel", "infonce_ts_kernel")])
def test_backward_kernel_selection(flags, kernel, other):
    """The default backward launch (and RC_INFONCE_TS_KERNEL) runs the TS kernel; RC_INFONCE_SS_KERNEL runs the SS kernel."""
    x, t, y, w = _case(1, 512, 16, 128, 256, seed=13)
    names = _kernel_names(lambda: _run(x, t, y, w, 1, flags))
    assert any(kernel in n for n in names), names
    assert not any(other in n for n in names), names


def test_forward_only_and_dtext_stay_on_ss_kernel():
    from rangeclip_b200 import ops
    x, t, y, w = _case(1, 512, 16, 128, 256, seed=14)
    for need_dx, need_dt in ((False, False), (True, True)):
        names = _kernel_names(lambda: ops.infonce_raw(x, t, y, w, 1 / 0.07, need_dx, need_dt, "bf16"))
        assert any("infonce_umma_pair_kernel" in n for n in names), names
        assert not any("infonce_ts_kernel" in n for n in names), names
