"""PyTorch-facing layer over the C ABI (``include/rangeclip_b200.h``).

Three tiers, top to bottom of this file:
  * ``*_raw`` / plain helpers: allocate outputs with torch, pass pointers + the current stream to the C ABI (ctypes);
  * ``torch.ops.rangeclip.*``: the same calls registered as PyTorch custom operators (``torch.library.custom_op`` with
    fake-tensor rules and autograd formulas), so that the dispatcher, ``torch.compile`` and fake-tensor tracing see
    them as single opaque nodes (north_star: "exposed as PyTorch custom ops");
  * the public functions the drop-ins call (``infonce``, ``pixel_losses``, ``smoothness``, ``masked_pool``, ...), thin
    shims over the registered operators.
Which InfoNCE kernel family a call takes (CUDA-core, one tensor-core launch, or tensor cores over blocks of 256 candidate
rows) is decided in one place, ``_infonce_plan``: ``infonce_raw`` dispatches on it, the fake-tensor rules of
``rangeclip::infonce`` / ``rangeclip::pixel_losses`` derive their outputs from it, and the loss drop-ins ask it whether a
kernel takes a call.
PyTorch is used for device memory, streams and autograd plumbing only; every computation is a kernel in
``librangeclip_b200.so``.  All functions require CUDA tensors on an sm_100 device and raise ``RuntimeError``
otherwise -- there is no CPU or eager-PyTorch fallback.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import RC_BF16, RC_F32, check

_I32_MAX = 2**31 - 1


def _need_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("rangeclip_b200 ops need CUDA tensors (no CPU fallback exists)")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return RC_F32
    if t.dtype == torch.bfloat16:
        return RC_BF16
    raise RuntimeError(f"rangeclip_b200: unsupported embedding dtype {t.dtype} (float32 or bfloat16)")


def _emb3(x: torch.Tensor) -> Tuple[torch.Tensor, int, int, int]:
    """[B, D, H, W] (or [B, D, HW]) contiguous view -> (x, B, D, HW)."""
    if x.dim() not in (3, 4):
        raise RuntimeError("pixel embeddings must be [B, D, H, W]")
    x = x.contiguous()
    B, D = x.shape[0], x.shape[1]
    return x, B, D, x[0, 0].numel() if B and D else 0


# ----------------------------------------------------------------------------------------------
# text preparation / sampling weights
# ----------------------------------------------------------------------------------------------

def text_prepare(text: torch.Tensor, idx: Optional[torch.Tensor], want_f32=True, want_bf16=False):
    """F.normalize(text[idx], dim=1) (model.py:272) as f32 [K,D] and/or bf16 [Kp,D] + [D,Kp]."""
    _need_cuda(text, idx)
    text = text.float().contiguous()
    K = int(idx.numel()) if idx is not None else text.shape[0]
    D = text.shape[1]
    Kp = (K + 63) // 64 * 64
    t32 = torch.empty(K, D, device=text.device, dtype=torch.float32) if want_f32 else None
    tb = torch.empty(Kp, D, device=text.device, dtype=torch.bfloat16) if want_bf16 else None
    ttb = torch.empty(D, Kp, device=text.device, dtype=torch.bfloat16) if want_bf16 else None
    if idx is not None:
        idx = idx.to(torch.int64).contiguous()
    # n_rows: an index outside [0, n_rows) yields a NaN row (the reference raises an index error at
    # candidate_text_embeddings[index_tensor]; a kernel cannot raise, and a silent out-of-bounds read is worse)
    check(_lib.lib().rc_text_prepare(_p(text), text.stride(0), text.shape[0], _p(idx), K, D, _p(t32), _p(tb), _p(ttb),
                                     _stream(text)), "rc_text_prepare")
    return t32, tb, ttb


def text_to_bf16(t_norm: torch.Tensor):
    """bf16 [Kp,D] and transposed [D,Kp] copies of already-normalised rows (tiny; plumbing only)."""
    K, D = t_norm.shape
    Kp = (K + 63) // 64 * 64
    tb = torch.zeros(Kp, D, device=t_norm.device, dtype=torch.bfloat16)
    tb[:K] = t_norm.detach().to(torch.bfloat16)
    return tb, tb.t().contiguous()


def sample_weights(seg: torch.Tensor, rand_idx: Optional[torch.Tensor], label_map: torch.Tensor):
    """Dense form of model.py:220-228,276-284: w[b,p] = multiplicity of p among rand_idx[b] (1 when
    rand_idx is None) zeroed on background / unmapped labels; y[b,p] = label_map[seg] or -1."""
    _need_cuda(seg, rand_idx, label_map)
    B = seg.shape[0]
    HW = seg[0].numel() if B else 0
    seg = seg.to(torch.int64).contiguous()
    label_map = label_map.to(torch.int32).contiguous()
    w = torch.empty(B, HW, device=seg.device, dtype=torch.float32)
    y = torch.empty(B, HW, device=seg.device, dtype=torch.int32)
    n_s = 0
    if rand_idx is not None:
        rand_idx = rand_idx.to(torch.int64).contiguous()
        n_s = rand_idx.shape[1]
    check(_lib.lib().rc_sample_weights(_p(seg), _p(rand_idx), B, HW, n_s, _p(label_map), label_map.numel(),
                                       _p(w), _p(y), _stream(seg)), "rc_sample_weights")
    return w, y


def sample_label_counts(seg: torch.Tensor, rand_idx: Optional[torch.Tensor], C: int) -> torch.Tensor:
    """int32 [C]: how many sampled pixels carry each label (model.py:222-226's gathered labels as a histogram)."""
    _need_cuda(seg, rand_idx)
    B = seg.shape[0]
    HW = seg[0].numel() if B else 0
    seg = seg.to(torch.int64).contiguous()
    counts = torch.zeros(C, device=seg.device, dtype=torch.int32)
    n_s = 0
    if rand_idx is not None:
        rand_idx = rand_idx.to(torch.int64).contiguous()
        n_s = rand_idx.shape[1]
    check(_lib.lib().rc_sample_label_counts(_p(seg), _p(rand_idx), B, HW, n_s, C, _p(counts), _stream(seg)), "rc_sample_label_counts")
    return counts


def clip_crops(images: torch.Tensor, boxes: torch.Tensor, image_index: torch.Tensor, shortest_edge: int, crop_size: int,
               mean, std) -> torch.Tensor:
    """All object crops of a batch as CLIP pixel values in one launch (rc_clip_crops; dataloader.py:254,276 with the
    torchvision-backend CLIP processor): images [B,C,H,W] (f32 / bf16), boxes int [n,4] = xmin, ymin, xmax, ymax,
    image_index int [n] -> f32 [n, C, crop_size, crop_size]."""
    _need_cuda(images, boxes, image_index)
    if images.dim() != 4:
        raise RuntimeError("clip_crops: images must be [B, C, H, W]")
    if images.dtype not in (torch.float32, torch.bfloat16):
        images = images.float()
    images = images.contiguous()
    B, C, H, W = images.shape
    n = int(image_index.numel())
    boxes = boxes.to(torch.int32).contiguous()
    image_index = image_index.to(torch.int32).contiguous()
    if boxes.numel() != 4 * n:
        raise RuntimeError("clip_crops: boxes must be [n, 4]")
    m = torch.as_tensor(list(mean), dtype=torch.float32).to(images.device, non_blocking=True)
    sd = torch.as_tensor(list(std), dtype=torch.float32).to(images.device, non_blocking=True)
    if m.numel() != C or sd.numel() != C:
        raise RuntimeError(f"clip_crops: mean / std must have {C} entries")
    out = torch.empty(n, C, int(crop_size), int(crop_size), device=images.device, dtype=torch.float32)
    check(_lib.lib().rc_clip_crops(_p(images), _dt(images), B, C, H, W, _p(boxes), _p(image_index), n, int(shortest_edge),
                                   int(crop_size), _p(m), _p(sd), _p(out), _stream(images)), "rc_clip_crops")
    return out


def contrast_build(counts: torch.Tensor, sim_off: Optional[torch.Tensor], sim_items: Optional[torch.Tensor], n_curriculum: int,
                   n_rand: int, k_cap: int, seed: int, seed_dev: Optional[torch.Tensor] = None, include_label0: bool = False):
    """Device-side contrast set (rc_contrast_build; model.py:234-268 without host round trips): from the label histogram of
    the sampled pixels to (label_map int32 [C], contrast int64 [k_cap] sorted ids padded with -1, kinfo int32 [4] =
    K, flags, #present, #distractors) in one launch, nothing read back."""
    _need_cuda(counts, sim_off, sim_items)
    C = counts.numel()
    counts = counts.to(torch.int32).contiguous()
    label_map = torch.empty(C, device=counts.device, dtype=torch.int32)
    contrast = torch.empty(int(k_cap), device=counts.device, dtype=torch.int64)
    kinfo = torch.empty(4, device=counts.device, dtype=torch.int32)
    if seed_dev is not None:
        seed_dev = seed_dev.to(torch.int64).contiguous()
    check(_lib.lib().rc_contrast_build(_p(counts), C, _p(sim_off), _p(sim_items), int(n_curriculum), int(n_rand), int(k_cap),
                                       int(seed) & 0xFFFFFFFFFFFFFFFF, _p(seed_dev), 1 if include_label0 else 0, _p(label_map), _p(contrast),
                                       _p(kinfo), _stream(counts)),
          "rc_contrast_build")
    return label_map, contrast, kinfo


# ----------------------------------------------------------------------------------------------
# InfoNCE
# ----------------------------------------------------------------------------------------------

def _infonce_plan(x: torch.Tensor, K: int, need_dt: bool, precision: str, rep: int, need_dx: bool = True,
                  dev_params: bool = False, dev_blocks: bool = False) -> Optional[str]:
    """The route of one InfoNCE call; the only place that chooses it.  ``infonce_raw`` runs it, the fake-tensor rules of
    rangeclip::infonce / pixel_losses derive dX's dtype from it and the loss drop-ins ask it whether a kernel takes a call.
      'fp32'      the CUDA-core kernel (rc_infonce_f32): D <= 1024, one target per row, host K and tau;
      'bf16'      one tensor-core launch (rc_infonce_bf16 / _rep4 / _dyn): K <= 256, D in (128, 256, 384, 512, 768, 1024),
                  HW % 8 == 0; four targets and the device-parameter form only on the CTA-pair kernel (D in _PAIR_D), dText
                  (with dX) only at D in (256, 512);
      'kblocked'  tensor cores over blocks of 256 candidate rows (``infonce_kblocked_raw``): D in _PAIR_D, HW % 8 == 0, no
                  dText, host K and tau; what "auto" (and, for four targets, "bf16") takes above 256 candidates; with
                  ``dev_blocks`` also for K and tau in device memory, up to 1024 rows (rc_infonce_bf16_dyn_kblock);
      None        no kernel covers the call.
    x: a tensor or meta tensor [B, D, H, W] / [B, D, HW]; K: rows of t_norm; precision: 'auto', 'fp32', 'bf16' or 'kblocked';
    need_dx: dX is wanted (the autograd operators always want it with dText); dev_params: K and log(tau) are read from device
    memory (k_dev / log_tau_dev).  dev_blocks (opt-in, implies dev_params): K is the CAPACITY of the contrast set (its valid
    row count stays in device memory); above 256 the K-blocked rounds read it from there -- 'kblocked' up to 1024 rows,
    'bf16' (the one-launch form) up to 256."""
    if rep not in (1, 4) or precision not in ("auto", "fp32", "bf16", "kblocked"):
        return None
    D = x.shape[1]
    HW = x[0, 0].numel() if x.shape[0] and D else 0
    if dev_blocks:
        if precision == "fp32" or need_dt or not kblocked_supported(D, HW) or not 1 <= K <= _DEV_BLOCKS_MAX_ROWS:
            return None
        return "kblocked" if (K > 256 or precision == "kblocked") else "bf16"
    kblocked = kblocked_supported(D, HW) and not need_dt and not dev_params
    if precision == "kblocked":
        return "kblocked" if kblocked else None
    fp32 = rep == 1 and not dev_params and D <= _F32_MAX_D
    if precision == "fp32":
        return "fp32" if fp32 else None
    if kblocked and K > 256 and (precision == "auto" or rep == 4):
        return "kblocked"
    one_launch = 1 <= K <= 256 and D in (128, 384) + _PAIR_D and HW % 8 == 0 and HW > 0
    if rep == 4 or need_dt or dev_params:         # forms only the CTA-pair kernel has
        one_launch = one_launch and D in _PAIR_D
    if need_dt:                                   # tensor-core dText: pair kernel + split-K GEMM (all channels in 512 TMEM columns)
        one_launch = one_launch and need_dx and not dev_params and D in _DTEXT_D
    if one_launch:
        return "bf16"
    return "fp32" if precision == "auto" and fp32 else None


def _infonce_route(x: torch.Tensor, K: int, need_dx: bool, need_dt: bool, precision: str, rep: int, dev_params: bool,
                   dev_blocks: bool = False) -> str:
    """``_infonce_plan``, or the error of a call no kernel covers (raised alike by the op and by its fake-tensor rules)."""
    route = _infonce_plan(x, K, need_dt, precision, rep, need_dx, dev_params, dev_blocks)
    if route is None:
        D = x.shape[1]
        HW = x[0, 0].numel() if x.shape[0] and D else 0
        raise RuntimeError(f"infonce: no kernel covers D={D}, HW={HW}, K={K}, precision={precision!r}, rep={rep} "
                           f"(need_dx={need_dx}, need_dt={need_dt}, device parameters={dev_params}, device blocks={dev_blocks}); "
                           "see _infonce_plan")
    return route


def _fused_tv(x: torch.Tensor, route: Optional[str]) -> bool:
    """Whether the launch's pre-pass over x also gives the smoothness sums of x -- and, with dX, the difference signs for
    tv_backward_codes (rc_infonce_prepass_tv): an fp32 NCHW x with W % 8 == 0 on the tensor-core route."""
    return route == "bf16" and x.dim() == 4 and x.dtype == torch.float32 and x.shape[3] % 8 == 0 and x.numel() > 0


def infonce_raw(x: torch.Tensor, t_norm: torch.Tensor, y: torch.Tensor, w: torch.Tensor, inv_tau: float,
                need_dx: bool, need_dt: bool, precision: str = "auto",
                grad_scale: Optional[torch.Tensor] = None, t_bf16=None, rep: int = 1, keep_bf16: bool = False,
                flags: int = 0, k_dev: Optional[torch.Tensor] = None, log_tau_dev: Optional[torch.Tensor] = None,
                fuse_tv: bool = False, dev_blocks: bool = False):
    """One fused pass: returns dict(loss_sum, w_sum (double[1] tensors), lse, dx, dt, dlogtau).
    loss = loss_sum / w_sum; dx/dt/dlogtau are gradients of that mean loss times grad_scale.  The kernel family is
    ``_infonce_plan``'s route; a call no kernel covers raises ``RuntimeError``.
    rep = 4: every row of x is the embedding shared by a 2x2 block of pixels (decoder.py:113, Q8);
    y / w are [rows, 4] and dx is the gradient w.r.t. the shared row (tensor-core paths only).
    keep_bf16: leave the tensor-core launch's dx in bf16 whatever x's dtype (the autograd wrappers widen and scale it
    in one pass at backward time); flags: extra RC_INFONCE_* bits for rc_infonce_bf16 (e.g. RC_INFONCE_SS_KERNEL).
    k_dev / log_tau_dev (device int32[>=1] / float[1]): the sync-free form (rc_infonce_bf16_dyn) -- the number of valid rows of
    t_norm and log(tau) are read by the kernel from device memory; ``inv_tau`` is ignored; CTA-pair kernel shapes only.
    dev_blocks (with k_dev / log_tau_dev): t_norm may hold up to 1024 rows; above 256 the K-blocked rounds run on them
    (``infonce_kblocked_raw``), each launch reading its valid rows from k_dev.
    fuse_tv: the caller also wants tv_sums(x); where the launch has a pre-pass over x anyway (``_fused_tv``) the sums come
    out of that pass (rc_infonce_prepass_tv) as ``tv_sums`` -- and with need_dx the difference signs for tv_backward_codes
    as ``tv_codes`` --, else both keys are None."""
    _need_cuda(x, t_norm, y, w)
    x_in = x
    x, B, D, HW = _emb3(x)
    K = t_norm.shape[0]
    dev_params = log_tau_dev is not None
    if dev_blocks and (k_dev is None or not dev_params):
        raise RuntimeError("infonce: dev_blocks needs k_dev and log_tau_dev")
    route = _infonce_route(x, K, need_dx, need_dt, precision, rep, dev_params, dev_blocks)
    tv_hw = tuple(x_in.shape[2:]) if (fuse_tv and _fused_tv(x_in, route)) else None
    dev = x.device
    M = B * HW
    y = y.reshape(-1).to(torch.int32).contiguous()
    w = w.reshape(-1).to(torch.float32).contiguous()
    if y.numel() != M * rep or w.numel() != M * rep:
        raise RuntimeError("infonce: y / w must have `rep` entries per embedding row")
    if route == "kblocked":
        # more candidates than one launch takes: tensor cores over blocks of 256 candidate rows instead of the CUDA-core
        # kernel (which needs ~100x longer at full size)
        r = infonce_kblocked_raw(x, t_norm, y, w, inv_tau, need_dx, rep=rep, k_dev=k_dev, log_tau_dev=log_tau_dev)
        dx = r["dx"]
        if dx is not None and grad_scale is not None:
            dx = dx * grad_scale.detach().reshape(1).to(device=dev, dtype=dx.dtype)
        dlt = r["dlogtau"] if r["dlogtau"] is not None else torch.zeros((), device=dev, dtype=torch.float64)
        if grad_scale is not None:
            dlt = dlt * grad_scale.detach().reshape(()).to(device=dev, dtype=torch.float64)
        return dict(loss_sum=r["loss_sum"], w_sum=r["w_sum"], dlogtau=dlt, lse=r["lse"], dx=dx, dt=None,
                    precision="bf16-kblocked", tv_sums=None, tv_codes=None)
    acc = torch.zeros(4, device=dev, dtype=torch.float64)        # loss_sum, w_sum, dlogtau, w_sum_in
    lse = torch.empty(M, device=dev, dtype=torch.float32)
    need_grad = need_dx or need_dt
    L = _lib.lib()
    st = _stream(x)
    if need_grad:
        check(L.rc_weight_sum(_p(w), _p(y), M * rep, acc[3:].data_ptr(), st), "rc_weight_sum")
    gs = None
    if grad_scale is not None:
        gs = grad_scale.detach().reshape(1).to(device=dev, dtype=torch.float32)
    dt = torch.zeros(K, D, device=dev, dtype=torch.float32) if need_dt else None
    tv = tv_codes = None
    if route == "fp32":
        xf = x if x.dtype == torch.float32 else x.float()
        tf = t_norm.detach().float().contiguous()
        dx = torch.empty_like(xf) if need_dx else None
        check(L.rc_infonce_f32(_p(xf), B, D, HW, D * HW, _p(tf), K, _p(y), _p(w), float(inv_tau), _p(lse),
                               acc[0:].data_ptr(), acc[1:].data_ptr(),
                               acc[3:].data_ptr() if need_grad else None, _p(gs),
                               _p(dx), _p(dt), acc[2:].data_ptr() if need_grad else None, st), "rc_infonce_f32")
        if dx is not None and dx.dtype != x.dtype:
            dx = dx.to(x.dtype)
    else:
        if t_bf16 is None:
            t_bf16 = text_to_bf16(t_norm)
        tb, ttb = t_bf16
        xdt = _dt(x)
        ws_bytes = int((L.rc_infonce_workspace_bytes_dt if need_dt else L.rc_infonce_workspace_bytes)(B, D, HW, K, xdt))
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        dxb = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16) if need_dx else None
        if tv_hw is not None:
            # fp32 x: the bf16 copy, the row norms, the smoothness sums and (for the backward) the signs of the differences,
            # 4 bits per element, from one read of x
            tv = torch.zeros(2, device=dev, dtype=torch.float64)
            if need_dx:
                tv_codes = torch.empty(B, D, int(tv_hw[0]), int(tv_hw[1]) // 8, device=dev, dtype=torch.int32)
            check(L.rc_infonce_prepass_tv(_p(x), B, D, int(tv_hw[0]), int(tv_hw[1]), _p(ws), ws_bytes, _p(tv), _p(tv_codes), st),
                  "rc_infonce_prepass_tv")
            flags = int(flags) | RC_INFONCE_PREPASS_DONE
        sums = (_p(lse), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr() if need_grad else None, _p(gs), _p(dxb))
        if dev_params:
            kd = k_dev.to(torch.int32) if k_dev is not None else None
            lt = log_tau_dev.detach().reshape(1).to(device=dev, dtype=torch.float32)
            entry, args = "rc_infonce_bf16_dyn", (_p(kd), _p(y), _p(w), _p(lt), rep) + sums
        else:
            entry = "rc_infonce_bf16" if rep == 1 else "rc_infonce_bf16_rep4"
            args = (_p(y), _p(w), float(inv_tau)) + sums + (_p(dt),)
        check(getattr(L, entry)(_p(x), xdt, B, D, HW, _p(tb), _p(ttb), K, *args, acc[2:].data_ptr() if need_dx else None,
                                _p(ws), ws_bytes, int(flags), st), entry)
        dx = None
        if dxb is not None:
            dx = dxb.view(x.shape) if (x.dtype == torch.bfloat16 or keep_bf16) else scale_to(dxb.view(x.shape), x.dtype)
    return dict(loss_sum=acc[0], w_sum=acc[1], dlogtau=acc[2], lse=lse, dx=dx, dt=dt, precision=route, tv_sums=tv,
                tv_codes=tv_codes)


RC_INFONCE_PREPASS_DONE, RC_INFONCE_KEEP_WEIGHT, RC_INFONCE_LSE_GIVEN, RC_INFONCE_TS_KERNEL, RC_INFONCE_ACCUMULATE_DX = 1, 2, 4, 8, 16
RC_INFONCE_SS_KERNEL = 32


_DEV_BLOCKS_MAX_ROWS = 1024      # contrast-set capacity of the device-parameter K-blocked rounds: four blocks, dX summed in-kernel
_PAIR_D = (256, 512, 768, 1024)  # widths of the CTA-pair kernels (CLIP ViT-B/32: 512, ViT-L/14: 768, ViT-H/14: 1024)
_DTEXT_D = (256, 512)            # widths of the tensor-core dText GEMM
_F32_MAX_D = 1024                # widest row of the CUDA-core kernels


def kblocked_supported(D: int, HW: int) -> bool:
    return D in _PAIR_D and HW % 8 == 0 and HW > 0


def infonce_kblocked_raw(x: torch.Tensor, t_norm: torch.Tensor, y: torch.Tensor, w: torch.Tensor, inv_tau: float,
                         need_dx: bool, block: int = 256, keep_bf16: bool = False, rep: int = 1,
                         k_dev: Optional[torch.Tensor] = None, log_tau_dev: Optional[torch.Tensor] = None):
    """InfoNCE against MORE than 256 candidates on the tensor cores (model.py:304-321 at thousands of objects): the
    candidate rows are split into launches of <= 256.  Round 1: forward launches give the per-block logsumexp; their
    logsumexp is the row's lse over all candidates.  Round 2: fwd+bwd launches with that lse given produce per-block dx /
    dlogtau that add up to the full gradient.  Returns dict(loss, loss_sum, lse, dx, dlogtau, w_sum), loss = loss_sum / w_sum;
    bf16 operands, fp32 sums.
    rep = 4: every row of x is the embedding shared by a 2x2 block of pixels, y / w are [rows, 4] (rc_infonce_bf16_rep4,
    one launch per block and round); lse is per row and a row's weight is the sum of its four.
    k_dev / log_tau_dev (device int32, first entry / float[1]; both or neither): the sync-free form.  t_norm's rows are the
    CAPACITY of the contrast set (<= 1024, the rows past k_dev[0] are zero pads) and shape the launches; each launch
    (rc_infonce_bf16_dyn_kblock) reads how many of its block's rows are valid and log(tau) from device memory, and a block
    past the valid rows is an empty launch.  The blocks are combined on the device with that block mask: nothing is read
    back, ``inv_tau`` is ignored."""
    _need_cuda(x, t_norm, y, w, k_dev, log_tau_dev)
    x, B, D, HW = _emb3(x)
    if not kblocked_supported(D, HW):
        raise RuntimeError(f"infonce_kblocked: needs D in {_PAIR_D} and HW % 8 == 0; got D={D}, HW={HW}")
    if rep not in (1, 4):
        raise RuntimeError("infonce_kblocked: rep must be 1 or 4")
    K = t_norm.shape[0]
    M = B * HW
    dev = x.device
    dyn = k_dev is not None or log_tau_dev is not None
    if dyn:
        if k_dev is None or log_tau_dev is None:
            raise RuntimeError("infonce_kblocked: k_dev and log_tau_dev go together")
        if block != 256 or K > _DEV_BLOCKS_MAX_ROWS:
            raise RuntimeError(f"infonce_kblocked: the device-parameter form takes blocks of 256 and at most "
                               f"{_DEV_BLOCKS_MAX_ROWS} rows; got K={K}")
        kd = k_dev.reshape(-1)[:1].to(torch.int32)
        lt = log_tau_dev.detach().reshape(1).to(device=dev, dtype=torch.float32)
    y = y.reshape(-1, 4) if rep == 4 else y.reshape(-1)
    if y.numel() != M * rep or w.numel() != M * rep:
        raise RuntimeError("infonce_kblocked: y / w must have `rep` entries per embedding row")
    y = y.to(torch.int32)
    # ignored targets: weight 0 (targets may leave the block)
    w = (w.reshape(y.shape).to(torch.float32) * (y >= 0)).contiguous()
    w_row = w.double().sum(dim=1) if rep == 4 else w.double()           # the weight each row's lse carries
    L = _lib.lib()
    st = _stream(x)
    xdt = _dt(x)
    ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, block, xdt))
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    if x.dtype != torch.bfloat16:
        # the bf16 copy of an fp32 x, once for all launches (a bf16 x needs no pre-pass: the CTA-pair kernel, the only one
        # these shapes reach, takes the row norms from its operand tiles)
        check(L.rc_infonce_prepass(_p(x), xdt, B, D, HW, _p(ws), ws_bytes, st), "rc_infonce_prepass")
    starts = list(range(0, K, block))
    nb = len(starts)
    if rep == 1 and B == 1 and HW % 256 == 0 and block == 256 and not dyn:
        # one image of rows (the area-image loss): every candidate block in ONE launch per round -- the kernel's image
        # index runs over the blocks (rc_infonce_bf16_kblocks)
        tb_all = torch.zeros(nb * 256, D, device=dev, dtype=torch.bfloat16)
        tb_all[:K] = t_norm.detach().to(torch.bfloat16)
        ttb_all = tb_all.t().contiguous()
        y_rel = (y[None, :] - 256 * torch.arange(nb, device=dev, dtype=torch.int32)[:, None]).contiguous()
        w_rep = w[None, :].expand(nb, M).contiguous()
        wsum = w.double().sum()
        acc = torch.zeros(4, device=dev, dtype=torch.float64)
        acc[3] = wsum * nb                       # (unused by the forward round)
        lse_blk = torch.empty(nb, M, device=dev, dtype=torch.float32)
        check(L.rc_infonce_bf16_kblocks(_p(x), xdt, D, HW, _p(tb_all), _p(ttb_all), K, nb, _p(y_rel), _p(w_rep), float(inv_tau),
                                        _p(lse_blk), acc[0:].data_ptr(), acc[1:].data_ptr(), None, None, None, None, _p(ws),
                                        ws_bytes, 1, st), "rc_infonce_bf16_kblocks(forward)")
        lse = torch.logsumexp(lse_blk, dim=0)
        wz = (lse_blk.double() * w.double()[None, :]).sum() - acc[0]
        loss_sum = (lse.double() * w.double()).sum() - wz
        loss = torch.where(wsum > 0, loss_sum / wsum.clamp_min(1e-300), torch.zeros_like(wsum))
        dx = dlogtau = None
        if need_dx:
            dxb = torch.empty(nb, D, HW, device=dev, dtype=torch.bfloat16)
            acc2 = torch.zeros(4, device=dev, dtype=torch.float64)
            acc2[3] = wsum
            check(L.rc_infonce_bf16_kblocks(_p(x), xdt, D, HW, _p(tb_all), _p(ttb_all), K, nb, _p(y_rel), _p(w_rep), float(inv_tau),
                                            _p(lse), acc2[0:].data_ptr(), acc2[1:].data_ptr(), acc2[3:].data_ptr(), None, _p(dxb),
                                            acc2[2:].data_ptr(), _p(ws), ws_bytes, 1 | RC_INFONCE_LSE_GIVEN, st),
                  "rc_infonce_bf16_kblocks(backward)")
            dx = dxb.float().sum(dim=0).view(x.shape).to(x.dtype)
            dlogtau = acc2[2].clone()
        return dict(loss=loss, loss_sum=loss_sum, lse=lse, dx=dx, dlogtau=dlogtau, w_sum=wsum)
    # bf16 operand copies of the candidate blocks: all full blocks with two tensor ops, a shorter last block on its own
    n_full = K // block if block % 64 == 0 else 0
    texts = []
    if n_full:
        tb_full = t_norm[:n_full * block].detach().to(torch.bfloat16).contiguous()
        ttb_full = tb_full.view(n_full, block, D).transpose(1, 2).contiguous()
        texts = [(tb_full[i * block:(i + 1) * block], ttb_full[i]) for i in range(n_full)]
    texts += [text_to_bf16(t_norm[s0:s0 + block]) for s0 in starts[n_full:]]
    ys = [(y - s0).contiguous() for s0 in starts]
    entry = L.rc_infonce_bf16 if rep == 1 else L.rc_infonce_bf16_rep4

    def launch(i, s0, lse_ptr, a, w_sum_in, dx_ptr, dlt_ptr, fl, what):
        Kb = min(block, K - s0)
        if dyn:       # the valid rows and log(tau) come from device memory; an empty block's launch returns at once
            check(L.rc_infonce_bf16_dyn_kblock(_p(x), xdt, B, D, HW, _p(texts[i][0]), _p(texts[i][1]), Kb, _p(kd), s0, _p(ys[i]),
                                               _p(w), _p(lt), rep, lse_ptr, a[0:].data_ptr(), a[1:].data_ptr(), w_sum_in, None,
                                               dx_ptr, dlt_ptr, _p(ws), ws_bytes, fl, st), f"rc_infonce_bf16_dyn_kblock({what})")
        else:
            check(entry(_p(x), xdt, B, D, HW, _p(texts[i][0]), _p(texts[i][1]), Kb, _p(ys[i]), _p(w), float(inv_tau),
                        lse_ptr, a[0:].data_ptr(), a[1:].data_ptr(), w_sum_in, None, dx_ptr, None, dlt_ptr,
                        _p(ws), ws_bytes, fl, st), f"rc_infonce_bf16({what})")

    lse_blk = torch.empty(nb, M, device=dev, dtype=torch.float32)
    acc = torch.zeros(nb, 4, device=dev, dtype=torch.float64)             # per block: loss_sum, w_sum, dlogtau, w_sum_in
    wsum = w.double().sum()
    acc[:, 3] = wsum
    for i, s0 in enumerate(starts):
        launch(i, s0, lse_blk[i].data_ptr(), acc[i], None, None, None, 1 | RC_INFONCE_KEEP_WEIGHT, "K block, forward")
    # sum_p w z[p, y_p] from the blocks that own the targets: loss_sum_b = sum_p w lse_b - sum_{y in b} w z_y
    wz_blk = (lse_blk.double() * w_row).sum(dim=1) - acc[:, 0]
    if dyn:
        # blocks past the valid rows were empty launches: their lse (never written) counts as -inf, their terms as 0
        first_rows = torch.arange(0, K, block, device=dev, dtype=torch.int32)
        live = (kd > first_rows) | (first_rows == 0)          # (the first block is never empty)
        lse_blk = torch.where(live[:, None], lse_blk, torch.full((), float("-inf"), device=dev))
        wz_blk = torch.where(live, wz_blk, torch.zeros((), device=dev, dtype=torch.float64))
    lse = torch.logsumexp(lse_blk, dim=0)
    wz = wz_blk.sum()
    loss_sum = (lse.double() * w_row).sum() - wz
    loss = torch.where(wsum > 0, loss_sum / wsum.clamp_min(1e-300), torch.zeros_like(wsum))
    dx = dlogtau = None
    if need_dx:
        dxb = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16)     # the tensor-core kernel always writes bf16
        acc2 = torch.zeros(nb, 4, device=dev, dtype=torch.float64)
        acc2[:, 3] = wsum
        # up to four blocks: every launch after the first ADDS its gradient to the same bf16 tensor inside the kernel
        # (RC_INFONCE_ACCUMULATE_DX, TMA reduce-add stores: one extra rounding per block, launch order = summation order);
        # more blocks are summed in fp32 here, block by block.  The device-parameter form (at most four blocks) always
        # accumulates in the kernel: an empty launch leaves dX as it is, where the fp32 sum would add a stale buffer.
        in_kernel = nb <= 4
        dx = None
        for i, s0 in enumerate(starts):
            fl = 1 | RC_INFONCE_KEEP_WEIGHT | RC_INFONCE_LSE_GIVEN | (RC_INFONCE_ACCUMULATE_DX if (in_kernel and i > 0) else 0)
            launch(i, s0, _p(lse), acc2[i], acc2[i, 3:].data_ptr(), _p(dxb), acc2[i, 2:].data_ptr(), fl, "K block, backward")
            if not in_kernel:
                dx = dxb.float() if dx is None else dx.add_(dxb)
        dlogtau = acc2[:, 2].sum()
        if in_kernel:
            dx = dxb.view(x.shape) if (x.dtype == torch.bfloat16 or keep_bf16) else scale_to(dxb.view(x.shape), x.dtype)
        else:
            dx = dx.view(x.shape).to(x.dtype)
    return dict(loss=loss, loss_sum=loss_sum, lse=lse, dx=dx, dlogtau=dlogtau, w_sum=wsum)


# ----------------------------------------------------------------------------------------------
# smoothness (TV-L1)
# ----------------------------------------------------------------------------------------------

def tv_sums(x: torch.Tensor) -> torch.Tensor:
    """double[2]: sum |dx_w|, sum |dx_h| over [B,D,H,W] (model.py:332-333 numerators)."""
    _need_cuda(x)
    x = x.contiguous()
    B, D, H, W = x.shape
    sums = torch.zeros(2, device=x.device, dtype=torch.float64)
    check(_lib.lib().rc_tv_fwd(_p(x), _dt(x), B * D, H, W, _p(sums), _stream(x)), "rc_tv_fwd")
    return sums


def tv_denominators(shape) -> Tuple[float, float]:
    B, D, H, W = shape
    return float(B * D * H * (W - 1)), float(B * D * (H - 1) * W)


def tv_backward(x: torch.Tensor, scale: torch.Tensor, dx: Optional[torch.Tensor] = None,
                dx_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A FRESH tensor (x's dtype) = dx_scale * dx + scale[0] * d(sum_h)/dx + scale[1] * d(sum_v)/dx.  ``dx`` (optional)
    is the gradient to accumulate onto and is left untouched (autograd may run a backward twice); it may be bf16
    under an fp32 x -- the tensor-core InfoNCE gradient -- so the fused backward of an fp32 embedding tensor reads x
    once, dx once and writes the result once (rc_tv_bwd_from)."""
    _need_cuda(x, scale, dx)
    x = x.contiguous()
    B, D, H, W = x.shape
    out = torch.empty_like(x)
    scale = scale.detach().to(device=x.device, dtype=torch.float32).contiguous()
    if dx is None:
        check(_lib.lib().rc_tv_bwd(_p(x), _dt(x), B * D, H, W, _p(scale), _p(out), 0, None, _stream(x)), "rc_tv_bwd")
        return out
    dx = dx.contiguous()
    if dx.numel() != x.numel():
        raise RuntimeError("tv_backward: dx must have x's shape")
    ds = None if dx_scale is None else dx_scale.detach().reshape(1).to(device=x.device, dtype=torch.float32)
    check(_lib.lib().rc_tv_bwd_from(_p(x), _dt(x), B * D, H, W, _p(scale), _p(dx), _dt(dx), _p(ds), _p(out), _stream(x)),
          "rc_tv_bwd_from")
    return out


def tv_backward_codes(codes: torch.Tensor, scale: torch.Tensor, dx: Optional[torch.Tensor] = None,
                      dx_scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """tv_backward of an fp32 x from the difference signs kept by the fused pre-pass (``codes`` int32 [B, D, H, W/8],
    rc_infonce_prepass_tv) instead of from x: a FRESH fp32 [B, D, H, W] tensor (rc_tv_bwd_codes)."""
    _need_cuda(codes, scale, dx)
    B, D, H, W8 = codes.shape
    out = torch.empty(B, D, H, W8 * 8, device=codes.device, dtype=torch.float32)
    scale = scale.detach().to(device=codes.device, dtype=torch.float32).contiguous()
    if dx is not None:
        dx = dx.contiguous()
        if dx.numel() != out.numel():
            raise RuntimeError("tv_backward_codes: dx must have x's shape")
    ds = None if (dx is None or dx_scale is None) else dx_scale.detach().reshape(1).to(device=codes.device, dtype=torch.float32)
    check(_lib.lib().rc_tv_bwd_codes(_p(codes), B * D, H, W8 * 8, _p(scale), _p(dx), _dt(dx) if dx is not None else _lib.RC_F32, _p(ds),
                                     _p(out), _stream(codes)), "rc_tv_bwd_codes")
    return out


def scale_to(x: torch.Tensor, out_dtype: torch.dtype, scale: Optional[torch.Tensor] = None) -> torch.Tensor:
    """A FRESH tensor of ``out_dtype`` = scale * x (scale: device scalar, None = 1): the late upstream scaling of a
    saved gradient and the bf16 -> fp32 widening of the tensor-core gradient in ONE pass (rc_scale_to)."""
    _need_cuda(x, scale)
    x = x.contiguous()
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    sc = None if scale is None else scale.detach().reshape(1).to(device=x.device, dtype=torch.float32)
    check(_lib.lib().rc_scale_to(_p(x), _dt(x), _p(out), _dt(out), x.numel(), _p(sc), _stream(x)), "rc_scale_to")
    return out


# ----------------------------------------------------------------------------------------------
# L2-normalised rows (decoder.py:114)
# ----------------------------------------------------------------------------------------------

# One step normalises the same decoder output twice: under no_grad for the area pooling (prepare_image_contrast_data,
# dataloader.py:205 is @torch.no_grad) and again, with autograd, for the smoothness term of compute_loss_shared2x2.  The
# no_grad result is kept until the NEXT call and handed over if that call asks for the same data: same address, layout and
# version counter -- and the entry holds a reference to the input, so its storage cannot have been freed and re-used.
_NORM_HANDOVER = None


def normalize_rows_raw(x: torch.Tensor):
    """(F.normalize(x, p=2, dim=1), 1 / max(|x|, 1e-12) per pixel) for an NCHW tensor, one kernel (rc_normalize_rows_fwd)."""
    global _NORM_HANDOVER
    _need_cuda(x)
    x, B, D, HW = _emb3(x)
    kept, _NORM_HANDOVER = _NORM_HANDOVER, None
    if kept is not None:
        xr, version, out, inv = kept
        if (xr.data_ptr() == x.data_ptr() and xr.shape == x.shape and xr.stride() == x.stride() and xr.dtype == x.dtype
                and xr.device == x.device and version == x._version):
            return out, inv
    out = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    inv = torch.empty(B, HW, device=x.device, dtype=torch.float32)
    check(_lib.lib().rc_normalize_rows_fwd(_p(x), _dt(x), B, D, HW, _p(out), _p(inv), _stream(x)), "rc_normalize_rows_fwd")
    if not torch.is_grad_enabled():
        _NORM_HANDOVER = (x, x._version, out, inv)
    return out, inv


def normalize_rows_backward(xhat: torch.Tensor, g: torch.Tensor, inv: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    xhat, B, D, HW = _emb3(xhat)
    g = g.float().contiguous()
    dx = torch.empty(xhat.shape, device=xhat.device, dtype=dtype)
    check(_lib.lib().rc_normalize_rows_bwd(_p(xhat), _p(g), _p(inv), _dt(dx), B, D, HW, _p(dx), _stream(xhat)), "rc_normalize_rows_bwd")
    return dx


# ----------------------------------------------------------------------------------------------
# masked pooling
# ----------------------------------------------------------------------------------------------

def _seg_views(seg: torch.Tensor, B: int):
    """One label map per pass: a tensor, or a list of tensors that label the SAME embedding rows (shared 2x2
    blocks: the four full-resolution label sub-grids of a half-resolution embedding map)."""
    segs = list(seg) if isinstance(seg, (list, tuple)) else [seg]
    return [s_.reshape(B, -1).to(torch.int64).contiguous() for s_ in segs]


def pool_forward(x: torch.Tensor, seg, lut: torch.Tensor, lut_per_image: bool, n_slots: int):
    """sum/count per slot then mean; lut [B,C] (per image) or [C] (batch-wide) int32, -1 = none.
    ``seg`` may be a list of label maps over the same rows: every pass adds into the same sums and counts."""
    _need_cuda(x, lut)
    x, B, D, HW = _emb3(x)
    segs = _seg_views(seg, B)
    lut = lut.to(torch.int32).contiguous()
    C = lut.shape[-1]
    out = torch.zeros(n_slots, D, device=x.device, dtype=torch.float32)
    cnt = torch.zeros(max(n_slots, 1), device=x.device, dtype=torch.int32)
    L = _lib.lib()
    for sg in segs:
        _need_cuda(sg)
        check(L.rc_pool_fwd(_p(x), _dt(x), B, D, HW, _p(sg), _p(lut), C if lut_per_image else 0, C, n_slots,
                            _p(out), _p(cnt), _stream(x)), "rc_pool_fwd")
    check(L.rc_pool_finish(_p(out), _p(cnt), n_slots, D, _stream(x)), "rc_pool_finish")
    return out, cnt


def pool_backward(g: torch.Tensor, cnt: torch.Tensor, seg, lut: torch.Tensor, lut_per_image: bool,
                  shape, dtype) -> torch.Tensor:
    B, D = shape[0], shape[1]
    HW = 1
    for s in shape[2:]:
        HW *= s
    segs = _seg_views(seg, B)
    lut = lut.to(torch.int32).contiguous()
    C = lut.shape[-1]
    g = g.float().contiguous()
    dx = torch.empty(shape, device=g.device, dtype=dtype)
    for i, sg in enumerate(segs):          # later passes accumulate: a row's gradient is the sum over its label maps
        check(_lib.lib().rc_pool_bwd(_p(g), _p(cnt), B, D, HW, _p(sg), _p(lut), C if lut_per_image else 0, C,
                                     g.shape[0], _p(dx), RC_F32 if dtype == torch.float32 else RC_BF16, 1 if i else 0,
                                     _stream(g)), "rc_pool_bwd")
    return dx


# ----------------------------------------------------------------------------------------------
# evaluation
# ----------------------------------------------------------------------------------------------

def topk_bf16_supported(D: int, HW: int) -> bool:
    return D % 64 == 0 and 64 <= D <= 1024 and HW % 8 == 0 and HW > 0


def eval_topk(x: torch.Tensor, t_norm: torch.Tensor, index_map: torch.Tensor, k: int, precision="auto", t_bf16=None):
    """out[b, j, h, w] = index_map[j-th best text row by cosine logit] (model.py:164-173).
    precision 'fp32' = CUDA-core kernel (reference arithmetic), 'bf16' = tcgen05 kernel, 'auto' = bf16 when
    the shape allows it."""
    _need_cuda(x, t_norm, index_map)
    x, B, D, HW = _emb3(x)
    K = t_norm.shape[0]
    k = min(k, K)
    out = torch.empty((B, k) + tuple(x.shape[2:]), device=x.device, dtype=torch.int64)
    index_map = index_map.to(torch.int64).contiguous()
    if precision == "auto":
        precision = "bf16" if topk_bf16_supported(D, HW) else "fp32"
    L = _lib.lib()
    if precision == "fp32":
        xf = x if x.dtype == torch.float32 else x.float()
        tf = t_norm.float().contiguous()
        check(L.rc_eval_topk_f32(_p(xf), B, D, HW, D * HW, _p(tf), K, _p(index_map), k, _p(out), _stream(x)),
              "rc_eval_topk_f32")
    elif precision == "bf16":
        if not topk_bf16_supported(D, HW):
            raise RuntimeError(f"eval_topk: bf16 tensor-core path does not cover D={D}, HW={HW}")
        tb = t_bf16 if t_bf16 is not None else text_to_bf16(t_norm)[0]
        xdt = _dt(x)
        ws, ws_bytes = None, 0
        if xdt == RC_F32:
            ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, xdt))
            ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
        check(L.rc_eval_topk_bf16(_p(x), xdt, B, D, HW, _p(tb), K, _p(index_map), k, _p(out), _p(ws), ws_bytes, _stream(x)),
              "rc_eval_topk_bf16")
    else:
        raise RuntimeError(f"eval_topk: unknown precision {precision!r}")
    return out


def eval_topk_hist(x: torch.Tensor, t_norm: torch.Tensor, index_map: torch.Tensor, k: int, gt: torch.Tensor,
                   E_u8: torch.Tensor, cmap: torch.Tensor, hist: torch.Tensor, counters: torch.Tensor, t_bf16=None,
                   want_ids: bool = True):
    """Fused evaluation batch (model.py:164-173 + validate.py:88-139): top-k on the tensor cores with the five class
    histograms and three counters built from the ids while they are still in registers (added to ``hist`` /
    ``counters``, int64).  Returns the ids [B,k,H,W] when ``want_ids`` (the drop-in ``predict`` needs them), else None.
    Tensor-core path only (D % 64 == 0, D <= 1024, HW % 8 == 0)."""
    _need_cuda(x, t_norm, index_map, gt, E_u8, cmap, hist, counters)
    x, B, D, HW = _emb3(x)
    if not topk_bf16_supported(D, HW):
        raise RuntimeError(f"eval_topk_hist: the fused kernel does not cover D={D}, HW={HW}; use eval_topk + eval_hist")
    K = t_norm.shape[0]
    k = min(k, K)
    C = cmap.numel()
    gt = gt.reshape(-1).to(torch.int64).contiguous()
    if gt.numel() != B * HW:
        raise RuntimeError("eval_topk_hist: gt must have one entry per pixel")
    if hist.dtype != torch.int64 or counters.dtype != torch.int64 or tuple(hist.shape) != (5, C) or counters.numel() != 3:
        raise RuntimeError("eval_topk_hist: hist must be int64 [5, C] and counters int64 [3]")
    out = torch.empty((B, k) + tuple(x.shape[2:]), device=x.device, dtype=torch.int64) if want_ids else None
    index_map = index_map.to(torch.int64).contiguous()
    tb = t_bf16 if t_bf16 is not None else text_to_bf16(t_norm)[0]
    L = _lib.lib()
    xdt = _dt(x)
    ws, ws_bytes = None, 0
    if xdt == RC_F32:
        ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, xdt))
        ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
    check(L.rc_eval_topk_hist_bf16(_p(x), xdt, B, D, HW, _p(tb), K, _p(index_map), k, _p(out), _p(gt), _p(E_u8.contiguous()),
                                   _p(cmap.to(torch.int64).contiguous()), C, _p(hist), _p(counters), _p(ws), ws_bytes,
                                   _stream(x)), "rc_eval_topk_hist_bf16")
    return out


def eval_topk_dyn(x: torch.Tensor, t_bf16: torch.Tensor, k_dev: torch.Tensor, index_map: torch.Tensor, k: int, gt=None, E_u8=None,
                  cmap=None, hist=None, counters=None, want_ids: bool = True):
    """``eval_topk`` / ``eval_topk_hist`` for a candidate set built on the device (rc_contrast_build): ``t_bf16`` [Kp, D] holds the
    normalised rows of the padded index list ``index_map`` [K], ``k_dev`` (int32, first entry) how many of them are valid -- read by
    the kernel from device memory, nothing is read back here (rc_eval_topk_dyn_bf16).  With ``hist`` / ``counters`` the metrics
    are fused as in ``eval_topk_hist``."""
    _need_cuda(x, t_bf16, k_dev, index_map)
    x, B, D, HW = _emb3(x)
    if not topk_bf16_supported(D, HW):
        raise RuntimeError(f"eval_topk_dyn: the tensor-core kernel does not cover D={D}, HW={HW}")
    K = int(index_map.numel())
    k = min(int(k), K)
    out = torch.empty((B, k) + tuple(x.shape[2:]), device=x.device, dtype=torch.int64) if (want_ids or hist is None) else None
    index_map = index_map.to(torch.int64).contiguous()
    C = 0
    if hist is not None:
        C = cmap.numel()
        gt = gt.reshape(-1).to(torch.int64).contiguous()
        if gt.numel() != B * HW or hist.dtype != torch.int64 or tuple(hist.shape) != (5, C) or counters.numel() != 3:
            raise RuntimeError("eval_topk_dyn: gt must have one entry per pixel, hist must be int64 [5, C], counters int64 [3]")
        E_u8, cmap = E_u8.contiguous(), cmap.to(torch.int64).contiguous()
    L = _lib.lib()
    xdt = _dt(x)
    ws, ws_bytes = None, 0
    if xdt == RC_F32:
        ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, xdt))
        ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
    check(L.rc_eval_topk_dyn_bf16(_p(x), xdt, B, D, HW, _p(t_bf16), K, _p(k_dev.to(torch.int32)), _p(index_map), k, _p(out), _p(gt),
                                  _p(E_u8), _p(cmap), C, _p(hist), _p(counters), _p(ws), ws_bytes, _stream(x)),
          "rc_eval_topk_dyn_bf16")
    return out


def eval_topk_rep4(x: torch.Tensor, t_bf16: torch.Tensor, index_map: torch.Tensor, k: int, gt=None, E_u8=None, cmap=None,
                   hist=None, counters=None, k_dev=None, want_ids: bool = True):
    """``eval_topk_dyn`` on the decoder's half-resolution rows (the ``output_conv`` result, SURVEY 8f-1): ``x`` [B,D,h,w] bf16 or
    fp32 stands for its nearest-x2 upsampled, normalised map, whose 2x2 blocks share one embedding and hence one top-k.  The
    ranking runs once per row; the ids [B,k,2h,2w] (returned when ``want_ids``) and, with ``hist`` / ``counters``, the metrics
    of the four pixels against the full-resolution ``gt`` [B,2h,2w] are those of the upsampled launch (rc_eval_topk_bf16_rep4).
    ``t_bf16`` [Kp,D] holds the normalised rows of ``index_map`` [K]; ``k_dev`` (int32, first entry, optional) how many are valid."""
    _need_cuda(x, t_bf16, k_dev, index_map, gt, E_u8, cmap, hist, counters)
    if x.dim() != 4:
        raise RuntimeError("eval_topk_rep4: x must be [B, D, h, w]")
    B, D, h, w = x.shape
    x = x.contiguous()
    if not topk_bf16_supported(D, h * w):
        raise RuntimeError(f"eval_topk_rep4: the tensor-core kernel does not cover D={D}, h*w={h * w}")
    K = int(index_map.numel())
    k = min(int(k), K)
    out = torch.empty((B, k, 2 * h, 2 * w), device=x.device, dtype=torch.int64) if (want_ids or hist is None) else None
    index_map = index_map.to(torch.int64).contiguous()
    if (gt is not None or hist is not None) and (gt is None or tuple(gt.shape) != (B, 2 * h, 2 * w)):
        raise RuntimeError(f"eval_topk_rep4: gt must be the full-resolution [B, 2h, 2w] = [{B}, {2 * h}, {2 * w}] segmentation")
    C = 0
    if hist is not None:
        C = cmap.numel()
        if hist.dtype != torch.int64 or tuple(hist.shape) != (5, C) or counters.dtype != torch.int64 or counters.numel() != 3:
            raise RuntimeError("eval_topk_rep4: hist must be int64 [5, C], counters int64 [3]")
        gt = gt.to(torch.int64).contiguous()
        if gt.data_ptr() % 16:               # the kernel loads the gt words of two adjacent pixels at once
            gt = gt.clone()
        E_u8, cmap = E_u8.contiguous(), cmap.to(torch.int64).contiguous()
    L = _lib.lib()
    xdt = _dt(x)
    ws, ws_bytes = None, 0
    if xdt == RC_F32:
        ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, h * w, K, xdt))
        ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
    kd = k_dev.to(torch.int32) if k_dev is not None else None
    check(L.rc_eval_topk_bf16_rep4(_p(x), xdt, B, D, h, w, _p(t_bf16), K, _p(kd), _p(index_map), k, _p(out), _p(gt), _p(E_u8),
                                   _p(cmap), C, _p(hist), _p(counters), _p(ws), ws_bytes, _stream(x)),
          "rc_eval_topk_bf16_rep4")
    return out


def eval_topk_scores(x: torch.Tensor, t_bf16: torch.Tensor, index_map: torch.Tensor, k: int, log_tau: torch.Tensor,
                     shared2x2: bool = False):
    """Top-k over a vocabulary with scores (rc_eval_topk_scores_bf16 / _rep4): ``t_bf16`` [Kp,D] holds the L2-normalised rows
    of ``index_map`` [K] (``text_prepare``), ``log_tau`` (device float, one element) the log of the softmax temperature.
    Returns (ids int64, cosine fp32, prob fp32), each [B,k,H,W]: the ids of ``eval_topk`` mapped through ``index_map``, the
    cosine of every ranked row and its softmax probability over all K rows at tau.  ``shared2x2``: ``x`` [B,D,h,w] is the
    decoder's ``output_conv`` result and the outputs are [B,k,2h,2w].  Nothing is read back to the host."""
    _need_cuda(x, t_bf16, index_map, log_tau)
    if shared2x2:
        if x.dim() != 4:
            raise RuntimeError("eval_topk_scores: shared2x2 needs x [B, D, h, w]")
        x = x.contiguous()
        B, D, h, w = x.shape
        HW, out_hw = h * w, (2 * h, 2 * w)
    else:
        x, B, D, HW = _emb3(x)
        out_hw = tuple(x.shape[2:])
    if not topk_bf16_supported(D, HW):
        raise RuntimeError(f"eval_topk_scores: the tensor-core kernel does not cover D={D}, HW={HW}")
    K = int(index_map.numel())
    if K < 1 or t_bf16.dtype != torch.bfloat16 or t_bf16.dim() != 2 or t_bf16.shape[1] != D or t_bf16.shape[0] < (K + 63) // 64 * 64:
        raise RuntimeError(f"eval_topk_scores: t_bf16 must be bf16 [round_up(K, 64), D] = [{(K + 63) // 64 * 64}, {D}]")
    if log_tau.numel() != 1:
        raise RuntimeError("eval_topk_scores: log_tau must hold one value")
    k = min(int(k), K)
    index_map = index_map.to(torch.int64).contiguous()
    lt = log_tau.detach().reshape(1).to(torch.float32).contiguous()
    ids = torch.empty((B, k) + out_hw, device=x.device, dtype=torch.int64)
    cos = torch.empty((B, k) + out_hw, device=x.device, dtype=torch.float32)
    prob = torch.empty((B, k) + out_hw, device=x.device, dtype=torch.float32)
    L = _lib.lib()
    xdt = _dt(x)
    ws, ws_bytes = None, 0
    if xdt == RC_F32:
        ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, xdt))
        ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
    tb = t_bf16.contiguous()
    if shared2x2:
        check(L.rc_eval_topk_scores_bf16_rep4(_p(x), xdt, B, D, h, w, _p(tb), K, _p(index_map), k, _p(lt), _p(ids), _p(cos),
                                              _p(prob), _p(ws), ws_bytes, _stream(x)), "rc_eval_topk_scores_bf16_rep4")
    else:
        check(L.rc_eval_topk_scores_bf16(_p(x), xdt, B, D, HW, _p(tb), K, _p(index_map), k, _p(lt), _p(ids), _p(cos), _p(prob),
                                         _p(ws), ws_bytes, _stream(x)), "rc_eval_topk_scores_bf16")
    return ids, cos, prob


def eval_hist(gt: torch.Tensor, topk: torch.Tensor, E_u8: torch.Tensor, cmap: torch.Tensor,
              hist: Optional[torch.Tensor] = None, counters: Optional[torch.Tensor] = None):
    """One batch of validate.py:88-139 as five class histograms + three counters (int64, added to)."""
    _need_cuda(gt, topk, E_u8, cmap)
    B, k = topk.shape[0], topk.shape[1]
    HW = topk[0, 0].numel()
    C = cmap.numel()
    gt = gt.reshape(-1).to(torch.int64).contiguous()
    topk = topk.to(torch.int64).contiguous()
    if gt.numel() != B * HW:
        raise RuntimeError("eval_hist: gt and topk disagree on the number of pixels")
    if hist is None:
        hist = torch.zeros(5, C, device=gt.device, dtype=torch.int64)
    if counters is None:
        counters = torch.zeros(3, device=gt.device, dtype=torch.int64)
    check(_lib.lib().rc_eval_hist(_p(gt), _p(topk), B, HW, k, _p(E_u8), _p(cmap), C, _p(hist), _p(counters),
                                  _stream(gt)), "rc_eval_hist")
    return hist, counters


def eval_fold(batch_hist: torch.Tensor, batch_index: int, acc: torch.Tensor, first_seen: torch.Tensor) -> None:
    C = batch_hist.shape[1]
    check(_lib.lib().rc_eval_fold(_p(batch_hist), C, int(batch_index), _p(acc), _p(first_seen), _stream(acc)),
          "rc_eval_fold")


# ----------------------------------------------------------------------------------------------
# torch.ops.rangeclip.* : the kernels as PyTorch custom operators (dispatcher / torch.compile / fake tensors)
# ----------------------------------------------------------------------------------------------

_DT_CODE = {torch.float32: 0, torch.bfloat16: 1}
_CODE_DT = {0: torch.float32, 1: torch.bfloat16}
_op = torch.library.custom_op


def _empty(like: torch.Tensor) -> torch.Tensor:
    return like.new_empty(0)


def _mean_loss(r) -> torch.Tensor:
    wsum = r["w_sum"]
    return torch.where(wsum > 0, r["loss_sum"] / wsum.clamp_min(1e-300), torch.zeros_like(wsum)).float().reshape(())


@_op("rangeclip::infonce", mutates_args=(), device_types="cuda")
def _op_infonce(x: torch.Tensor, t_norm: torch.Tensor, log_tau: torch.Tensor, y: torch.Tensor, w: torch.Tensor,
                need_grad: bool, need_dt: bool, precision: str, rep: int, t_bf16: Optional[torch.Tensor],
                tt_bf16: Optional[torch.Tensor], k_dev: Optional[torch.Tensor] = None,
                dev_blocks: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(loss, dx, dt, dlogtau): weighted InfoNCE(x, t_norm, y, w) / tau with the gradients of the MEAN loss produced by
    the same fused launch (single pass over x).  dx stays in the kernel's dtype (bf16 on the tensor-core path).
    ``k_dev`` (int32 device tensor, first entry = valid rows of t_norm): the sync-free form -- the kernel reads the row
    count and log(tau) from device memory, nothing is read back here.  ``dev_blocks`` (with k_dev, opt-in): t_norm's rows are
    the contrast set's capacity, up to 1024; above 256 the K-blocked rounds run on them (``_infonce_plan``)."""
    return _infonce_forward(x, t_norm, log_tau, y, w, need_grad, need_dt, precision, rep, t_bf16, tt_bf16, k_dev, False,
                            dev_blocks)[:4]


def _infonce_forward(x, t_norm, log_tau, y, w, need_grad, need_dt, precision, rep, t_bf16, tt_bf16, k_dev, fuse_tv,
                     dev_blocks=False):
    """Body of rangeclip::infonce (and of the InfoNCE half of rangeclip::pixel_losses): (loss, dx, dt, dlogtau, tv_sums | None, tv_codes | None)."""
    tb = (t_bf16, tt_bf16) if (t_bf16 is not None and tt_bf16 is not None) else None
    dyn = k_dev is not None
    inv_tau = 0.0 if dyn else float(torch.exp(-log_tau.detach().float()))      # one scalar sync, as .item() in the reference
    r = infonce_raw(x, t_norm, y, w, inv_tau, need_grad, need_dt, precision, t_bf16=tb, rep=rep, keep_bf16=True, k_dev=k_dev,
                    log_tau_dev=log_tau if dyn else None, fuse_tv=fuse_tv, dev_blocks=dev_blocks)
    dx, dt = r["dx"], r["dt"]
    return (_mean_loss(r), dx if dx is not None else _empty(x), dt if dt is not None else _empty(t_norm),
            r["dlogtau"].float().reshape(()), r.get("tv_sums"), r.get("tv_codes"))


@_op_infonce.register_fake
def _(x, t_norm, log_tau, y, w, need_grad, need_dt, precision, rep, t_bf16, tt_bf16, k_dev=None, dev_blocks=False):
    route = _infonce_route(x, t_norm.shape[0], need_grad, need_dt, precision, rep, k_dev is not None, dev_blocks)
    dx_dtype = torch.bfloat16 if route == "bf16" else x.dtype
    f32 = dict(device=x.device, dtype=torch.float32)
    return (torch.empty((), **f32), torch.empty(x.shape, device=x.device, dtype=dx_dtype) if need_grad else _empty(x),
            torch.empty(t_norm.shape, **f32) if need_dt else _empty(t_norm), torch.empty((), **f32))


def _infonce_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1], output[2], output[3])
    ctx.x_dtype = inputs[0].dtype
    # the auxiliary outputs (dx: the size of x) never carry an upstream gradient; without this autograd materialises a
    # ZERO tensor of that size for each of them on every backward (a 4.3 GB fill at the headline size)
    ctx.set_materialize_grads(False)


def _graph_is_retained() -> bool:
    """True unless the running backward was started with retain_graph=False (then the graph's saved tensors are released
    after this pass and may be consumed in place).  Unknown (tracing, no graph task) counts as retained."""
    try:
        if torch.compiler.is_compiling():
            return True
        return bool(torch._C._autograd._get_current_graph_task_keep_graph())
    except Exception:  # noqa: BLE001
        return True


def _infonce_backward(ctx, g, *_unused):
    dx, dt, dlt = ctx.saved_tensors
    need = ctx.needs_input_grad
    gx = None
    if g is None:
        return (None,) * 13
    if need[0]:
        if dx.dtype == ctx.x_dtype and not _graph_is_retained():
            # the common training case (loss.backward()): nobody can run this node again, so the saved gradient is scaled
            # in place -- and rc_scale returns after reading the scalar when the upstream gradient is exactly 1
            torch.ops.rangeclip.scale_(dx, g)
            gx = dx
        else:
            # retain_graph / autograd.grad: the saved gradient stays READ-ONLY, the scaled (and widened) copy is a fresh
            # tensor, so a second backward through the same graph sees the same dx again
            gx = torch.ops.rangeclip.scale_to(dx, g, _DT_CODE[ctx.x_dtype])
    gt = dt * g if need[1] else None
    gl = (dlt * g).reshape(()) if need[2] else None
    return (gx, gt, gl) + (None,) * 10


_op_infonce.register_autograd(_infonce_backward, setup_context=_infonce_setup)


@_op("rangeclip::pixel_losses", mutates_args=(), device_types="cuda")
def _op_pixel_losses(x: torch.Tensor, t_norm: torch.Tensor, log_tau: torch.Tensor, y: torch.Tensor, w: torch.Tensor,
                     need_grad: bool, need_dt: bool, precision: str, t_bf16: Optional[torch.Tensor],
                     tt_bf16: Optional[torch.Tensor], k_dev: Optional[torch.Tensor] = None,
                     dev_blocks: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """(text InfoNCE, smoothness, dx_text, dt, dlogtau, tv_codes) of the SAME pixel embeddings: one autograd node for both
    terms, so that the backward is a single pass (model.py:272-291, 332-334 and their autograd).  tv_codes: the difference
    signs the backward needs, when the fp32 pre-pass produced them with the sums (else empty)."""
    loss, dx, dt, dlt, sums, codes = _infonce_forward(x, t_norm, log_tau, y, w, need_grad, need_dt, precision, 1, t_bf16, tt_bf16,
                                                      k_dev, True, dev_blocks)
    if sums is None:
        sums = tv_sums(x)
    if codes is None:
        codes = torch.empty(0, device=x.device, dtype=torch.int32)
    dh, dv = tv_denominators(x.shape)
    nan = torch.full((), float("nan"), device=x.device, dtype=torch.float64)
    smooth = ((sums[0] / dh if dh > 0 else nan) + (sums[1] / dv if dv > 0 else nan)).float().reshape(())
    return loss, smooth, dx, dt, dlt, codes


@_op_pixel_losses.register_fake
def _(x, t_norm, log_tau, y, w, need_grad, need_dt, precision, t_bf16, tt_bf16, k_dev=None, dev_blocks=False):
    route = _infonce_route(x, t_norm.shape[0], need_grad, need_dt, precision, 1, k_dev is not None, dev_blocks)
    dx_dtype = torch.bfloat16 if route == "bf16" else x.dtype
    f32 = dict(device=x.device, dtype=torch.float32)
    fused = need_grad and _fused_tv(x, route)
    return (torch.empty((), **f32), torch.empty((), **f32),
            torch.empty(x.shape, device=x.device, dtype=dx_dtype) if need_grad else _empty(x),
            torch.empty(t_norm.shape, **f32) if need_dt else _empty(t_norm), torch.empty((), **f32),
            torch.empty(tuple(x.shape[:3]) + (x.shape[3] // 8,) if fused else (0,), device=x.device, dtype=torch.int32))


def _pixel_losses_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0], output[2], output[3], output[4], output[5])
    ctx.set_materialize_grads(False)         # see _infonce_setup


def _pixel_losses_backward(ctx, g_text, g_smooth, *_unused):
    x, dx, dt, dlt, codes = ctx.saved_tensors
    need = ctx.needs_input_grad
    gx = None
    if g_text is None and g_smooth is None:
        return (None,) * 12
    if g_text is None:
        g_text = torch.zeros((), device=x.device, dtype=torch.float32)
    if g_smooth is None:
        g_smooth = torch.zeros((), device=x.device, dtype=torch.float32)
    if need[0]:
        dh, dv = tv_denominators(x.shape)
        gs = g_smooth.float()
        scale = torch.stack([gs / dh if dh > 0 else gs * 0, gs / dv if dv > 0 else gs * 0])
        # dX = g_text * dX_text (from the forward launch) + g_smooth * d(TV)/dX in ONE pass, into a fresh tensor
        if codes.numel():        # fp32 x: from the difference signs of the fused pre-pass, x is not read again
            gx = torch.ops.rangeclip.tv_bwd_codes(codes, scale, dx, g_text.float())
        else:
            gx = torch.ops.rangeclip.tv_bwd(x, scale, dx, g_text.float())
    gt = dt * g_text if need[1] else None
    gl = (dlt * g_text).reshape(()) if need[2] else None
    return (gx, gt, gl) + (None,) * 9


_op_pixel_losses.register_autograd(_pixel_losses_backward, setup_context=_pixel_losses_setup)


@_op("rangeclip::scale_to", mutates_args=(), device_types="cuda")
def _op_scale_to(x: torch.Tensor, scale: Optional[torch.Tensor], out_dtype: int) -> torch.Tensor:
    return scale_to(x, _CODE_DT[out_dtype], scale)


@_op_scale_to.register_fake
def _(x, scale, out_dtype):
    return torch.empty(x.shape, device=x.device, dtype=_CODE_DT[out_dtype])


@_op("rangeclip::scale_", mutates_args=("x",), device_types="cuda")
def _op_scale_inplace(x: torch.Tensor, scale: torch.Tensor) -> None:
    """x *= scale (device scalar), in place; no pass over memory when the scalar is exactly 1 (rc_scale)."""
    sc = scale.detach().reshape(1).to(device=x.device, dtype=torch.float32)
    check(_lib.lib().rc_scale(_p(x), _dt(x), x.numel(), _p(sc), _stream(x)), "rc_scale")


@_op("rangeclip::tv_sums", mutates_args=(), device_types="cuda")
def _op_tv_sums(x: torch.Tensor) -> torch.Tensor:
    return tv_sums(x)


@_op_tv_sums.register_fake
def _(x):
    return torch.empty(2, device=x.device, dtype=torch.float64)


@_op("rangeclip::tv_bwd", mutates_args=(), device_types="cuda")
def _op_tv_bwd(x: torch.Tensor, scale: torch.Tensor, dx: Optional[torch.Tensor], dx_scale: Optional[torch.Tensor]) -> torch.Tensor:
    return tv_backward(x, scale, dx if (dx is not None and dx.numel()) else None, dx_scale)


@_op_tv_bwd.register_fake
def _(x, scale, dx, dx_scale):
    return torch.empty_like(x)


@_op("rangeclip::tv_bwd_codes", mutates_args=(), device_types="cuda")
def _op_tv_bwd_codes(codes: torch.Tensor, scale: torch.Tensor, dx: Optional[torch.Tensor], dx_scale: Optional[torch.Tensor]) -> torch.Tensor:
    return tv_backward_codes(codes, scale, dx if (dx is not None and dx.numel()) else None, dx_scale)


@_op_tv_bwd_codes.register_fake
def _(codes, scale, dx, dx_scale):
    return torch.empty(tuple(codes.shape[:3]) + (codes.shape[3] * 8,), device=codes.device, dtype=torch.float32)


@_op("rangeclip::smoothness", mutates_args=(), device_types="cuda")
def _op_smoothness(x: torch.Tensor, den_h: float, den_v: float) -> torch.Tensor:
    """sum_h / den_h + sum_v / den_v (model.py:332-333); NaN for an empty slice (W == 1 or H == 1), as l1_loss."""
    sums = tv_sums(x)
    nan = torch.full((), float("nan"), device=x.device, dtype=torch.float64)
    return ((sums[0] / den_h if den_h > 0 else nan) + (sums[1] / den_v if den_v > 0 else nan)).float().reshape(())


@_op_smoothness.register_fake
def _(x, den_h, den_v):
    return torch.empty((), device=x.device, dtype=torch.float32)


def _smoothness_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[0])
    ctx.den = (inputs[1], inputs[2])


def _smoothness_backward(ctx, g):
    (x,) = ctx.saved_tensors
    dh, dv = ctx.den
    gf = g.float()
    scale = torch.stack([gf / dh if dh > 0 else gf * 0, gf / dv if dv > 0 else gf * 0])
    return torch.ops.rangeclip.tv_bwd(x, scale, None, None), None, None


_op_smoothness.register_autograd(_smoothness_backward, setup_context=_smoothness_setup)


def tv_normalize_backward(xhat: torch.Tensor, inv: torch.Tensor, scale: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """d/dx of scale[0] * sum_h + scale[1] * sum_v of normalize(x) from the saved xhat / inv (rc_tv_normalize_bwd): one kernel
    instead of rc_tv_bwd -> gradient tensor -> rc_normalize_rows_bwd."""
    _need_cuda(xhat, inv, scale)
    B, D, H, W = xhat.shape
    dx = torch.empty(xhat.shape, device=xhat.device, dtype=dtype)
    scale = scale.detach().to(device=xhat.device, dtype=torch.float32).contiguous()
    check(_lib.lib().rc_tv_normalize_bwd(_p(xhat), _p(inv), _p(scale), _dt(dx), B, D, H, W, _p(dx), _stream(xhat)), "rc_tv_normalize_bwd")
    return dx


@_op("rangeclip::smoothness_normalized", mutates_args=(), device_types="cuda")
def _op_smoothness_normalized(x: torch.Tensor, den_h: float, den_v: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(smoothness of F.normalize(x, dim=1), xhat, 1/|x|): model.py:332-333 on the decoder tail's output (decoder.py:114) with the
    normalisation inside the operator, so that its backward is ONE kernel (rc_tv_normalize_bwd)."""
    xhat, inv = normalize_rows_raw(x)
    sums = tv_sums(xhat)
    nan = torch.full((), float("nan"), device=x.device, dtype=torch.float64)
    loss = ((sums[0] / den_h if den_h > 0 else nan) + (sums[1] / den_v if den_v > 0 else nan)).float().reshape(())
    return loss, xhat, inv


@_op_smoothness_normalized.register_fake
def _(x, den_h, den_v):
    return (torch.empty((), device=x.device, dtype=torch.float32), torch.empty(x.shape, device=x.device, dtype=torch.float32),
            torch.empty(x.shape[0], x[0, 0].numel(), device=x.device, dtype=torch.float32))


@_op("rangeclip::tv_normalize_bwd", mutates_args=(), device_types="cuda")
def _op_tv_normalize_bwd(xhat: torch.Tensor, inv: torch.Tensor, scale: torch.Tensor, dtype_code: int) -> torch.Tensor:
    return tv_normalize_backward(xhat, inv, scale, _CODE_DT[dtype_code])


@_op_tv_normalize_bwd.register_fake
def _(xhat, inv, scale, dtype_code):
    return torch.empty(xhat.shape, device=xhat.device, dtype=_CODE_DT[dtype_code])


def _smoothness_normalized_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1], output[2])
    ctx.den = (inputs[1], inputs[2])
    ctx.x_dtype = inputs[0].dtype
    ctx.set_materialize_grads(False)


def _smoothness_normalized_backward(ctx, g, _g_xhat, _g_inv):
    if g is None:
        return None, None, None
    xhat, inv = ctx.saved_tensors
    dh, dv = ctx.den
    gf = g.float()
    scale = torch.stack([gf / dh if dh > 0 else gf * 0, gf / dv if dv > 0 else gf * 0])
    return torch.ops.rangeclip.tv_normalize_bwd(xhat, inv, scale, _DT_CODE[ctx.x_dtype]), None, None


_op_smoothness_normalized.register_autograd(_smoothness_normalized_backward, setup_context=_smoothness_normalized_setup)


@_op("rangeclip::normalize_rows", mutates_args=(), device_types="cuda")
def _op_normalize_rows(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(F.normalize(x, p=2, dim=1), per-pixel 1 / max(|x|, 1e-12)) of an NCHW tensor -- the decoder tail (decoder.py:114)."""
    return normalize_rows_raw(x)


@_op_normalize_rows.register_fake
def _(x):
    return (torch.empty(x.shape, device=x.device, dtype=torch.float32),
            torch.empty(x.shape[0], x[0, 0].numel(), device=x.device, dtype=torch.float32))


@_op("rangeclip::normalize_rows_bwd", mutates_args=(), device_types="cuda")
def _op_normalize_rows_bwd(xhat: torch.Tensor, g: torch.Tensor, inv: torch.Tensor, dtype_code: int) -> torch.Tensor:
    return normalize_rows_backward(xhat, g, inv, _CODE_DT[dtype_code])


@_op_normalize_rows_bwd.register_fake
def _(xhat, g, inv, dtype_code):
    return torch.empty(xhat.shape, device=xhat.device, dtype=_CODE_DT[dtype_code])


def _normalize_rows_setup(ctx, inputs, output):
    ctx.save_for_backward(output[0], output[1])
    ctx.x_dtype = inputs[0].dtype
    ctx.set_materialize_grads(False)


def _normalize_rows_backward(ctx, g, _g_inv):
    xhat, inv = ctx.saved_tensors
    if g is None:
        return None
    return torch.ops.rangeclip.normalize_rows_bwd(xhat, g, inv, _DT_CODE[ctx.x_dtype])


_op_normalize_rows.register_autograd(_normalize_rows_backward, setup_context=_normalize_rows_setup)


@_op("rangeclip::masked_pool", mutates_args=(), device_types="cuda")
def _op_masked_pool(x: torch.Tensor, segs: Sequence[torch.Tensor], lut: torch.Tensor, lut_per_image: bool,
                    n_slots: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(mean [n_slots, D] in x's dtype, count [n_slots] int32) of the segment-masked average pooling."""
    out, cnt = pool_forward(x, list(segs), lut, lut_per_image, n_slots)
    return (out.to(x.dtype) if x.dtype != torch.float32 else out), cnt


@_op_masked_pool.register_fake
def _(x, segs, lut, lut_per_image, n_slots):
    return (torch.empty(n_slots, x.shape[1], device=x.device, dtype=x.dtype),
            torch.empty(max(n_slots, 1), device=x.device, dtype=torch.int32))


@_op("rangeclip::masked_pool_bwd", mutates_args=(), device_types="cuda")
def _op_masked_pool_bwd(g: torch.Tensor, cnt: torch.Tensor, segs: Sequence[torch.Tensor], lut: torch.Tensor,
                        lut_per_image: bool, shape: Sequence[int], dtype_code: int) -> torch.Tensor:
    return pool_backward(g, cnt, list(segs), lut, lut_per_image, tuple(shape), _CODE_DT[dtype_code])


@_op_masked_pool_bwd.register_fake
def _(g, cnt, segs, lut, lut_per_image, shape, dtype_code):
    return torch.empty(tuple(shape), device=g.device, dtype=_CODE_DT[dtype_code])


def _masked_pool_setup(ctx, inputs, output):
    x, segs, lut, lut_per_image, _n = inputs
    ctx.save_for_backward(output[1], lut, *segs)
    ctx.meta = (lut_per_image, tuple(x.shape), x.dtype)


def _masked_pool_backward(ctx, g, _g_cnt):
    cnt, lut, *segs = ctx.saved_tensors
    lut_per_image, shape, dtype = ctx.meta
    gx = torch.ops.rangeclip.masked_pool_bwd(g, cnt, segs, lut, lut_per_image, list(shape), _DT_CODE[dtype])
    return gx, [None] * len(segs), None, None, None


_op_masked_pool.register_autograd(_masked_pool_backward, setup_context=_masked_pool_setup)


@_op("rangeclip::sample_weights", mutates_args=(), device_types="cuda")
def _op_sample_weights(seg: torch.Tensor, rand_idx: Optional[torch.Tensor], label_map: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    return sample_weights(seg, rand_idx, label_map)


@_op_sample_weights.register_fake
def _(seg, rand_idx, label_map):
    B = seg.shape[0]
    HW = seg[0].numel() if B else 0
    return (torch.empty(B, HW, device=seg.device, dtype=torch.float32), torch.empty(B, HW, device=seg.device, dtype=torch.int32))


@_op("rangeclip::sample_label_counts", mutates_args=(), device_types="cuda")
def _op_sample_label_counts(seg: torch.Tensor, rand_idx: Optional[torch.Tensor], C: int) -> torch.Tensor:
    return sample_label_counts(seg, rand_idx, C)


@_op_sample_label_counts.register_fake
def _(seg, rand_idx, C):
    return torch.empty(C, device=seg.device, dtype=torch.int32)


@_op("rangeclip::contrast_build", mutates_args=(), device_types="cuda")
def _op_contrast_build(counts: torch.Tensor, sim_off: Optional[torch.Tensor], sim_items: Optional[torch.Tensor], n_curriculum: int,
                       n_rand: int, k_cap: int, seed: int, seed_dev: Optional[torch.Tensor] = None,
                       include_label0: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return contrast_build(counts, sim_off, sim_items, n_curriculum, n_rand, k_cap, seed, seed_dev, include_label0)


@_op_contrast_build.register_fake
def _(counts, sim_off, sim_items, n_curriculum, n_rand, k_cap, seed, seed_dev=None, include_label0=False):
    return (torch.empty(counts.numel(), device=counts.device, dtype=torch.int32),
            torch.empty(k_cap, device=counts.device, dtype=torch.int64), torch.empty(4, device=counts.device, dtype=torch.int32))


@_op("rangeclip::text_prepare", mutates_args=(), device_types="cuda")
def _op_text_prepare(text: torch.Tensor, idx: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """F.normalize(text[idx], dim=1) as f32 [K,D], bf16 [Kp,D] and bf16 [D,Kp] (Kp = K rounded up to 64, zero pads)."""
    return text_prepare(text, idx, want_f32=True, want_bf16=True)


@_op_text_prepare.register_fake
def _(text, idx):
    K = idx.numel() if idx is not None else text.shape[0]
    D = text.shape[1]
    Kp = (K + 63) // 64 * 64
    return (torch.empty(K, D, device=text.device, dtype=torch.float32), torch.empty(Kp, D, device=text.device, dtype=torch.bfloat16),
            torch.empty(D, Kp, device=text.device, dtype=torch.bfloat16))


@_op("rangeclip::eval_topk", mutates_args=(), device_types="cuda")
def _op_eval_topk(x: torch.Tensor, t_norm: torch.Tensor, index_map: torch.Tensor, k: int, precision: str,
                  t_bf16: Optional[torch.Tensor]) -> torch.Tensor:
    return eval_topk(x, t_norm, index_map, k, precision, t_bf16)


@_op_eval_topk.register_fake
def _(x, t_norm, index_map, k, precision, t_bf16):
    k = min(k, t_norm.shape[0])
    return torch.empty((x.shape[0], k) + tuple(x.shape[2:]), device=x.device, dtype=torch.int64)


@_op("rangeclip::eval_topk_scores", mutates_args=(), device_types="cuda")
def _op_eval_topk_scores(x: torch.Tensor, t_bf16: torch.Tensor, index_map: torch.Tensor, k: int, log_tau: torch.Tensor,
                         shared2x2: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return eval_topk_scores(x, t_bf16, index_map, k, log_tau, shared2x2)


@_op_eval_topk_scores.register_fake
def _(x, t_bf16, index_map, k, log_tau, shared2x2):
    k = min(k, index_map.numel())
    hw = (2 * x.shape[2], 2 * x.shape[3]) if shared2x2 else tuple(x.shape[2:])
    shape = (x.shape[0], k) + hw
    return (torch.empty(shape, device=x.device, dtype=torch.int64), torch.empty(shape, device=x.device, dtype=torch.float32),
            torch.empty(shape, device=x.device, dtype=torch.float32))


@_op("rangeclip::eval_hist", mutates_args=("hist", "counters"), device_types="cuda")
def _op_eval_hist(gt: torch.Tensor, topk: torch.Tensor, E_u8: torch.Tensor, cmap: torch.Tensor, hist: torch.Tensor,
                  counters: torch.Tensor) -> None:
    eval_hist(gt, topk, E_u8, cmap, hist, counters)


@_op("rangeclip::eval_topk_hist", mutates_args=("hist", "counters"), device_types="cuda")
def _op_eval_topk_hist(x: torch.Tensor, t_norm: torch.Tensor, index_map: torch.Tensor, k: int, gt: torch.Tensor, E_u8: torch.Tensor,
                       cmap: torch.Tensor, hist: torch.Tensor, counters: torch.Tensor, t_bf16: Optional[torch.Tensor],
                       want_ids: bool) -> torch.Tensor:
    ids = eval_topk_hist(x, t_norm, index_map, k, gt, E_u8, cmap, hist, counters, t_bf16=t_bf16, want_ids=want_ids)
    return ids if ids is not None else torch.empty(0, device=x.device, dtype=torch.int64)


@_op_eval_topk_hist.register_fake
def _(x, t_norm, index_map, k, gt, E_u8, cmap, hist, counters, t_bf16, want_ids):
    k = min(k, t_norm.shape[0])
    if not want_ids:
        return torch.empty(0, device=x.device, dtype=torch.int64)
    return torch.empty((x.shape[0], k) + tuple(x.shape[2:]), device=x.device, dtype=torch.int64)


@_op("rangeclip::eval_topk_rep4", mutates_args=("hist", "counters"), device_types="cuda")
def _op_eval_topk_rep4(x: torch.Tensor, t_bf16: torch.Tensor, index_map: torch.Tensor, k: int, gt: Optional[torch.Tensor],
                       E_u8: Optional[torch.Tensor], cmap: Optional[torch.Tensor], hist: Optional[torch.Tensor],
                       counters: Optional[torch.Tensor], k_dev: Optional[torch.Tensor], want_ids: bool) -> torch.Tensor:
    ids = eval_topk_rep4(x, t_bf16, index_map, k, gt, E_u8, cmap, hist, counters, k_dev=k_dev, want_ids=want_ids)
    return ids if ids is not None else torch.empty(0, device=x.device, dtype=torch.int64)


@_op_eval_topk_rep4.register_fake
def _(x, t_bf16, index_map, k, gt, E_u8, cmap, hist, counters, k_dev, want_ids):
    if not want_ids and hist is not None:
        return torch.empty(0, device=x.device, dtype=torch.int64)
    k = min(k, index_map.numel())
    return torch.empty((x.shape[0], k, 2 * x.shape[2], 2 * x.shape[3]), device=x.device, dtype=torch.int64)


@_op("rangeclip::eval_fold", mutates_args=("acc", "first_seen"), device_types="cuda")
def _op_eval_fold(batch_hist: torch.Tensor, batch_index: int, acc: torch.Tensor, first_seen: torch.Tensor) -> None:
    eval_fold(batch_hist, batch_index, acc, first_seen)


# ----------------------------------------------------------------------------------------------
# public autograd-aware entry points (what losses.py / pooling.py call)
# ----------------------------------------------------------------------------------------------

def _tb(t_bf16):
    return (None, None) if t_bf16 is None else (t_bf16[0], t_bf16[1])


def infonce(x, t_norm, log_tau, y, w, precision="auto", rep=1, t_bf16=None, k_dev=None, dev_blocks=False):
    """Autograd-aware fused InfoNCE (torch.ops.rangeclip.infonce); x [B,D,H,W], t_norm [K,D] normalised, y/w per pixel
    (rep = 4: x holds the embeddings shared by 2x2 pixel blocks, y/w are [B*H*W, 4]).  ``precision``: 'auto', 'fp32', 'bf16'
    or 'kblocked', the kernel family as ``_infonce_plan`` routes it.  ``t_bf16`` = (bf16 [Kp,D], bf16 [D,Kp]) copies of
    t_norm from ``text_prepare`` (optional: built on the fly otherwise).  ``k_dev``: the valid rows of t_norm in device memory
    (log(tau) is then read from ``log_tau`` on the device as well); ``dev_blocks``: t_norm may then hold up to 1024 rows
    (the K-blocked rounds above 256)."""
    _need_cuda(x, t_norm, y, w)
    tb, ttb = _tb(t_bf16)
    need_grad = bool(torch.is_grad_enabled() and (x.requires_grad or log_tau.requires_grad))
    need_dt = bool(torch.is_grad_enabled() and t_norm.requires_grad)
    return torch.ops.rangeclip.infonce(x, t_norm, log_tau, y, w, need_grad or need_dt, need_dt, precision, rep, tb, ttb, k_dev,
                                       dev_blocks)[0]


def pixel_losses(x, t_norm, log_tau, y, w, precision="auto", t_bf16=None, k_dev=None, dev_blocks=False):
    """(text InfoNCE, smoothness) with a fused single-pass backward (torch.ops.rangeclip.pixel_losses); k_dev, dev_blocks as
    for ``infonce``."""
    _need_cuda(x, t_norm, y, w)
    tb, ttb = _tb(t_bf16)
    need_grad = bool(torch.is_grad_enabled() and (x.requires_grad or log_tau.requires_grad))
    need_dt = bool(torch.is_grad_enabled() and t_norm.requires_grad)
    out = torch.ops.rangeclip.pixel_losses(x, t_norm, log_tau, y, w, need_grad or need_dt, need_dt, precision, tb, ttb, k_dev,
                                           dev_blocks)
    return out[0], out[1]


def smoothness(x: torch.Tensor, denominators=None) -> torch.Tensor:
    """sum_h / dh + sum_v / dv; the denominators default to the element counts of x's own slices
    (model.py:332-333) and can be overridden when x stands for a larger tensor (shared 2x2 blocks)."""
    _need_cuda(x)
    dh, dv = tv_denominators(x.shape) if denominators is None else denominators
    return torch.ops.rangeclip.smoothness(x, float(dh), float(dv))


def smoothness_normalized(x: torch.Tensor, denominators=None) -> torch.Tensor:
    """``smoothness(F.normalize(x, dim=1), denominators)`` with a fused single-kernel backward (x NCHW f32 / bf16, W % 8 == 0)."""
    _need_cuda(x)
    dh, dv = tv_denominators(x.shape) if denominators is None else denominators
    return torch.ops.rangeclip.smoothness_normalized(x, float(dh), float(dv))[0]


def normalize_rows(x: torch.Tensor) -> torch.Tensor:
    """F.normalize(x, p=2, dim=1) of an NCHW tensor (f32 or bf16) as f32, with autograd, one kernel each way (HW % 8 == 0)."""
    _need_cuda(x)
    return torch.ops.rangeclip.normalize_rows(x)[0]


def masked_pool(x, seg, lut, lut_per_image, n_slots):
    _need_cuda(x, lut)
    segs = list(seg) if isinstance(seg, (list, tuple)) else [seg]
    return torch.ops.rangeclip.masked_pool(x, segs, lut, bool(lut_per_image), int(n_slots))[0]


def _check_bringup(status: int, what: str) -> None:
    if status != 0:
        raise RuntimeError(f"{what} failed (status {status}): {_lib.bringup_lib().rc_last_error().decode('utf-8', 'replace')}")


def debug_umma_gemm(a: torch.Tensor, b: torch.Tensor, variant: int) -> torch.Tensor:
    """Bring-up check of the TMA + tcgen05 + TMEM path: C[128,N] = A B^T in bf16 -> f32."""
    _need_cuda(a, b)
    N, Kd = b.shape
    c = torch.empty(128, N, device=a.device, dtype=torch.float32)
    _check_bringup(_lib.bringup_lib().rc_debug_umma_gemm(_p(a.contiguous()), _p(b.contiguous()), N, Kd, variant, _p(c), _stream(a)),
          "rc_debug_umma_gemm")
    return c


def debug_umma_gemm_2sm(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Bring-up check of the CTA-pair (cta_group::2) path: C[256,N] = A[256,Kd] B[N,Kd]^T."""
    _need_cuda(a, b)
    N, Kd = b.shape
    c = torch.empty(256, N, device=a.device, dtype=torch.float32)
    _check_bringup(_lib.bringup_lib().rc_debug_umma_gemm_2sm(_p(a.contiguous()), _p(b.contiguous()), N, Kd, _p(c), _stream(a)),
          "rc_debug_umma_gemm_2sm")
    return c


def debug_umma_gemm_ts_2sm(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """Bring-up check of the TS-mode path (A in tensor memory): C[256,N] = A[256,Kd] B[N,Kd]^T, Kd <= 256."""
    _need_cuda(a, b)
    N, Kd = b.shape
    c = torch.empty(256, N, device=a.device, dtype=torch.float32)
    _check_bringup(_lib.bringup_lib().rc_debug_umma_gemm_ts_2sm(_p(a.contiguous()), _p(b.contiguous()), N, Kd, _p(c), _stream(a)),
          "rc_debug_umma_gemm_ts_2sm")
    return c
