"""Drop-in for ``DepthUNet.compute_loss`` (RangeCLIP/src/depth_segmentation_model/model.py:178-355).

Same signature, same ``loss_info`` keys, same RNG streams consumed in the same order
(``torch.randint`` on the device, ``np.random.choice``, CPU ``torch.randperm``; SURVEY Q6), same
zero-loss fallbacks with the same warnings (Q14).  The three loss terms run on the CUDA kernels of
this package; only the tiny host-side contrast-set builder (model.py:231-270) stays in Python, as in
the reference.

Use either as a mixin (``class MyUNet(DepthCLIPLossMixin, DepthUNet)``), by assignment
(``DepthUNet.compute_loss = rangeclip_b200.compute_loss``), or as a free function with a model
object that owns ``log_temperature_text`` / ``log_temperature_image``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops


def build_contrast_indices(unique_labels: torch.Tensor, C: int, label_similarity_sets, k_distractors: int,
                           pct_medium: float, pct_hard: float, pct_rand: float, device) -> torch.Tensor:
    """Contrast set = GT labels in the sample + curriculum distractors (model.py:234-268).

    Host logic, kept behaviour-identical to the reference including the ``label in container``
    membership test that silently disables hard/medium distractors for list-form sets (Q3) and
    the order in which ``np.random`` and the CPU torch generator are consumed (Q6).  The index arithmetic
    (model.py:259-268: arange / isin / randperm / cat / unique) runs on HOST tensors here -- same values, same
    generators, but one device transfer of K indices at the end instead of a dozen tiny launches and syncs."""
    present = unique_labels.tolist()
    present_set = set(present)
    n_medium = int(k_distractors * pct_medium)
    n_hard = int(k_distractors * pct_hard)
    n_rand = k_distractors - n_medium - n_hard
    candidates = set()
    for n_wanted, key in ((n_medium, 'medium'), (n_hard, 'hard')):
        if n_wanted > 0:
            table = label_similarity_sets[key]
            for lab in present:
                if lab in table:
                    candidates.update(table[lab])
    candidates = [c for c in list(candidates) if c not in present_set]      # the set's own iteration order, as in the reference
    n_curriculum = n_medium + n_hard
    if len(candidates) >= n_curriculum:
        chosen = np.random.choice(candidates, size=n_curriculum, replace=False)
    else:
        chosen = candidates
    chosen = torch.tensor(chosen, dtype=torch.long)
    uniq_h = torch.tensor(present, dtype=torch.long)
    every = torch.arange(C)
    free = every[~torch.isin(every, torch.cat([uniq_h, chosen], dim=0))]
    if n_rand > 0 and len(free) > 0:
        rand_part = free[torch.randperm(len(free))[:n_rand]]
    else:
        rand_part = torch.tensor([], dtype=torch.long)
    return torch.unique(torch.cat([uniq_h, chosen, rand_part], dim=0)).to(device)


_CSR_CACHE = {}


def similarity_csr(label_similarity_sets, C: int, use_medium: bool, use_hard: bool, device):
    """The similarity tables as device CSR (int32 offsets [C+1], int32 items) for ``rc_contrast_build``: per label the union
    of its 'medium' / 'hard' lists (those whose share of the distractors is non-zero, model.py:240-247).  Tables that are
    not dicts never match a label in the reference (`label in table` on a list compares with its elements, quirk Q3); the
    same here.  Built once per (tables object, C, selection, device) and cached."""
    key = (id(label_similarity_sets), C, bool(use_medium), bool(use_hard), str(device))
    hit = _CSR_CACHE.get(key)
    if hit is not None and hit[0] is label_similarity_sets:
        return hit[1], hit[2]
    rows = [[] for _ in range(C)]
    for use, name in ((use_medium, 'medium'), (use_hard, 'hard')):
        table = label_similarity_sets.get(name) if (use and isinstance(label_similarity_sets, dict)) else None
        if isinstance(table, dict):
            for lab, items in table.items():
                if isinstance(lab, int) and 0 <= lab < C:
                    rows[lab].extend(int(v) for v in items)
    off = np.zeros(C + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(r) for r in rows])
    items = np.fromiter((v for r in rows for v in r), dtype=np.int32, count=int(off[-1]))
    if items.size == 0:
        items = np.zeros(1, dtype=np.int32)
    off_d, items_d = torch.from_numpy(off).to(device), torch.from_numpy(items).to(device)
    if len(_CSR_CACHE) > 16:
        _CSR_CACHE.clear()
    _CSR_CACHE[key] = (label_similarity_sets, off_d, items_d)
    return off_d, items_d


def device_builder_supported(x: torch.Tensor, rep: int, C: int, k_cap: int, text_requires_grad: bool, precision: str) -> bool:
    """Calls the sync-free path covers: label histogram in shared memory (2 <= C <= 12000), not the fp32 parity mode, and
    tensor-core launches that read K and tau from device memory (``ops._infonce_plan`` with ``dev_blocks``: the CTA-pair
    kernel, frozen text, one launch up to 256 contrast rows and the K-blocked rounds up to 1024)."""
    return (2 <= C <= 12000 and precision != "fp32"
            and ops._infonce_plan(x, k_cap, text_requires_grad, "bf16", rep, dev_params=True, dev_blocks=True) is not None)


def text_contrastive_loss(pixel_embeddings, target_indices, candidate_text_embeddings, label_similarity_sets,
                          log_temperature_text, percent_image_sampling=0.7, k_distractors=50, pct_medium=0.0,
                          pct_hard=0.75, pct_rand=0.25, precision="auto", return_aux=False, with_smoothness=False,
                          shared2x2=False, contrast_builder="reference", max_contrast=256):
    """Pixel-text InfoNCE of model.py:199-301 on the fused kernels.

    The reference gathers ``int(0.7*HW)`` pixel rows per image WITH replacement and drops label 0
    (model.py:220-228); here the same ``torch.randint`` draw becomes a per-pixel multiplicity weight
    and the [B,D,H,W] tensor is read in place (no gather, no [N,K] logits).

    ``shared2x2``: ``pixel_embeddings`` is the decoder's PRE-upsample output [B,D,H/2,W/2] (normalised
    or not) while ``target_indices`` stays [B,H,W]; every embedding row then carries the four targets /
    multiplicities of its 2x2 block (decoder.py:113-114, quirk Q8) and the same loss and gradient come
    out of a quarter of the tensor-core work."""
    assert abs(pct_medium + pct_hard + pct_rand - 1.0) < 1e-4, "Sum of text percentages must be 1."
    B, D, H, W = pixel_embeddings.shape
    if shared2x2:
        H, W = 2 * H, 2 * W
        if with_smoothness:
            raise RuntimeError("text_contrastive_loss: with_smoothness is not available with shared2x2")
        if tuple(target_indices.shape[-2:]) != (H, W):
            raise RuntimeError(f"text_contrastive_loss(shared2x2): targets must be {H}x{W}, got {tuple(target_indices.shape)}")
    C = candidate_text_embeddings.shape[0]
    device = pixel_embeddings.device
    zero = lambda: torch.zeros((), device=device)
    hw = H * W
    if hw == 0:
        raise RuntimeError("Input dimensions H or W are zero.")
    n_samples = min(int(percent_image_sampling * H * W), hw)
    if n_samples == 0 and hw > 0:
        n_samples = hw
    rand_indices = torch.randint(0, hw, (B, n_samples), device=device)
    target_flat = target_indices.reshape(B, -1)
    aux = dict(rand_indices=rand_indices, contrast_indices=None)
    if contrast_builder not in ("reference", "device"):
        raise RuntimeError(f"contrast_builder must be 'reference' or 'device', got {contrast_builder!r}")
    k_cap = max(2, min(int(max_contrast), 1024, C))
    if contrast_builder == "device" and device_builder_supported(pixel_embeddings, 4 if shared2x2 else 1, C, k_cap,
                                                                 candidate_text_embeddings.requires_grad, precision):
        # ---- sync-free path (SURVEY 8f-2): label histogram -> contrast set, label map, text operands and the loss launch
        # without one device->host read; the set size and the temperature reach the kernel through device memory
        n_medium = int(k_distractors * pct_medium)
        n_hard = int(k_distractors * pct_hard)
        n_rand = k_distractors - n_medium - n_hard
        sim_off, sim_items = similarity_csr(label_similarity_sets, C, n_medium > 0, n_hard > 0, device)
        seed_dev = None
        if torch.cuda.is_current_stream_capturing():
            # CUDA-graph capture: a host-side seed would be frozen into the graph.  The CUDA generator is graph-safe (its
            # Philox offset advances per replay), so the seed is drawn on the device and read by the kernel from memory.
            seed = 0
            seed_dev = torch.randint(0, 2 ** 62, (1,), device=device, dtype=torch.int64)
        else:
            seed = int(torch.empty((), dtype=torch.int64).random_().item())   # CPU generator (the stream the reference's randperm uses): no device sync
        counts = torch.ops.rangeclip.sample_label_counts(target_flat, rand_indices, C)
        label_map, contrast, kinfo = torch.ops.rangeclip.contrast_build(counts, sim_off, sim_items, n_medium + n_hard, n_rand,
                                                                        k_cap, seed, seed_dev)
        aux["contrast_indices"] = contrast
        aux["contrast_info"] = kinfo
        w, y = torch.ops.rangeclip.sample_weights(target_flat, rand_indices, label_map)
        t_norm, tb, ttb = torch.ops.rangeclip.text_prepare(candidate_text_embeddings, contrast)
        if with_smoothness:
            loss, smooth = ops.pixel_losses(pixel_embeddings, t_norm, log_temperature_text, y, w, "bf16", t_bf16=(tb, ttb),
                                            k_dev=kinfo, dev_blocks=True)
            aux["smoothness"] = smooth
            return loss, aux
        if shared2x2:
            y, w = group_2x2(y.view(B, H, W)), group_2x2(w.view(B, H, W))
        loss = ops.infonce(pixel_embeddings, t_norm, log_temperature_text, y, w, "bf16", rep=4 if shared2x2 else 1,
                           t_bf16=(tb, ttb), k_dev=kinfo, dev_blocks=True)
        return (loss, aux) if return_aux else loss
    # the sampled foreground labels (model.py:222-233: gather, drop label 0, torch.unique) from a label histogram of the
    # sampled pixels: one small kernel instead of a 3M-element gather + boolean index + sort
    if C <= 12000:
        counts = torch.ops.rangeclip.sample_label_counts(target_flat, rand_indices, C)
        unique_labels = torch.nonzero(counts[1:]).reshape(-1) + 1
    else:
        label_samples = torch.gather(target_flat, 1, rand_indices)
        unique_labels = torch.unique(label_samples[label_samples > 0])
    if unique_labels.numel() == 0 or D == 0:
        print("Warning: No valid foreground pixels sampled for text contrastive loss.")
        return (zero(), aux) if return_aux else zero()
    contrast = build_contrast_indices(unique_labels, C, label_similarity_sets, k_distractors, pct_medium,
                                      pct_hard, pct_rand, device)
    aux["contrast_indices"] = contrast
    if len(contrast) <= 1:
        print("Warning: Not enough indices for text contrastive loss (need > 1).")
        return (zero(), aux) if return_aux else zero()
    label_map = torch.full((C,), -1, dtype=torch.int32, device=device)
    label_map[contrast] = torch.arange(contrast.shape[0], device=device, dtype=torch.int32)
    w, y = torch.ops.rangeclip.sample_weights(target_flat, rand_indices, label_map)
    t_bf16 = None
    if candidate_text_embeddings.requires_grad:
        t_norm = torch.nn.functional.normalize(candidate_text_embeddings[contrast].float(), dim=1)
    else:       # one launch: normalised rows as f32 and as the two bf16 operand layouts of the tensor-core kernels
        t_norm, tb, ttb = torch.ops.rangeclip.text_prepare(candidate_text_embeddings, contrast)
        t_bf16 = (tb, ttb)
    if with_smoothness:      # one autograd node for both terms -> one fused backward pass over X / dX
        loss, smooth = ops.pixel_losses(pixel_embeddings, t_norm, log_temperature_text, y, w, precision, t_bf16=t_bf16)
        aux["smoothness"] = smooth
        return loss, aux
    if shared2x2:
        # the four-target kernel: one launch, or blocks of 256 candidate rows for frozen text above 256 contrast rows (their
        # number is data dependent, model.py:268).  The plan is asked with the text's requires_grad, not the grad mode's
        # view of it, so a no_grad call with trainable text takes the same route as the training step
        if ops._infonce_plan(pixel_embeddings, int(contrast.shape[0]), candidate_text_embeddings.requires_grad, precision, 4) is not None:
            y, w = group_2x2(y.view(B, H, W)), group_2x2(w.view(B, H, W))
            loss = ops.infonce(pixel_embeddings, t_norm, log_temperature_text, y, w, precision, rep=4, t_bf16=t_bf16)
        else:
            # outside what the four-target kernel covers (D not 256 / 512 / 768 / 1024, fp32 parity mode, more than 256 contrast rows
            # with trainable text): the loss of the upsampled tensor itself, as the decoder would emit it (decoder.py:113);
            # autograd sums the four pixel gradients of a block below the interpolation
            up = torch.nn.functional.interpolate(pixel_embeddings, scale_factor=2, mode="nearest")
            loss = ops.infonce(up, t_norm, log_temperature_text, y, w, precision, t_bf16=t_bf16)
    else:
        loss = ops.infonce(pixel_embeddings, t_norm, log_temperature_text, y, w, precision, t_bf16=t_bf16)
    return (loss, aux) if return_aux else loss


def group_2x2(t: torch.Tensor) -> torch.Tensor:
    """[B, 2h, 2w] -> [B, h*w, 4]: the four full-resolution entries of every shared-embedding block."""
    B, H, W = t.shape
    return t.reshape(B, H // 2, 2, W // 2, 2).permute(0, 1, 3, 2, 4).reshape(B, (H // 2) * (W // 2), 4).contiguous()


def image_contrastive_loss(area_embeddings, image_embeddings, log_temperature_image, precision="auto"):
    """Area-image InfoNCE of model.py:304-321: rows = pooled area embeddings, candidates = CLIP
    crop embeddings, positives on the diagonal.  n is at most a few thousand, so the rows are
    transposed to the kernels' [D][n] layout first (n*D elements; plumbing).

    ``precision``: "fp32" = CUDA-core kernel (1e-5 path; what the reference's n <= batch size needs -- the call is
    launch-bound there); "bf16" = tensor cores with the candidates in blocks of 256 (``ops.infonce`` with
    ``precision="kblocked"``; the fp32 kernel takes 9 ms at n = 4096); "auto" = bf16 from n = 512 when the shape allows it
    (D in (256, 512, 768, 1024), n % 8 == 0, frozen image embeddings)."""
    n, D = area_embeddings.shape
    x = area_embeddings.float().t().contiguous().view(1, D, n, 1)
    blocked_ok = ops._infonce_plan(x, n, image_embeddings.requires_grad, "kblocked", 1) is not None
    if precision == "auto":
        precision = "bf16" if (blocked_ok and n >= 512) else "fp32"
    if precision == "bf16":
        if not blocked_ok:
            raise RuntimeError(f"image_contrastive_loss: the tensor-core path needs D in (256, 512, 768, 1024), n % 8 == 0 and frozen "
                               f"image embeddings; got n={n}, D={D}")
        precision = "kblocked"
    if image_embeddings.requires_grad:
        t_norm = torch.nn.functional.normalize(image_embeddings.float(), dim=1)
    else:
        t_norm, _, _ = torch.ops.rangeclip.text_prepare(image_embeddings, None)
    y = torch.arange(n, device=x.device, dtype=torch.int32)
    w = torch.ones(n, device=x.device, dtype=torch.float32)
    return ops.infonce(x, t_norm, log_temperature_image, y, w, precision)


def compute_loss(self, pixel_embeddings, target_indices, candidate_text_embeddings, label_similarity_sets,
                 area_embeddings, image_embeddings, W_text=1.0, W_image=0.5, W_smooth=2e2,
                 percent_image_sampling=0.7, k_distractors=50, pct_medium=0.0, pct_hard=0.75, pct_rand=0.25,
                 precision="auto", contrast_builder="reference", max_contrast=256):
    """Hybrid contrastive loss: pixel-text + area-image + smoothness (model.py:178-355).

    ``contrast_builder="device"`` (opt-in, SURVEY 8f-2): the contrast set is drawn on the GPU (``rc_contrast_build``, a
    counter-based stream seeded from the CPU torch generator -- NOT the reference's NumPy / randperm streams, so the drawn
    distractors differ from the reference's for the same seeds), its size and the temperatures stay in device memory, and
    ``loss_info`` is a ``LazyLossInfo`` whose floats are fetched on first access: the call never synchronises with the
    host.  At most ``max_contrast`` (<= 1024) rows; distractors are trimmed to fit.  Up to 256 rows the loss is one
    tensor-core launch; above, K-blocked rounds shaped for ``max_contrast`` rows, each launch reading from device memory how
    many of its rows the drawn set fills."""
    return _compute_loss(self, pixel_embeddings, target_indices, candidate_text_embeddings, label_similarity_sets,
                         area_embeddings, image_embeddings, W_text, W_image, W_smooth, percent_image_sampling,
                         k_distractors, pct_medium, pct_hard, pct_rand, precision, shared2x2=False,
                         contrast_builder=contrast_builder, max_contrast=max_contrast)


def compute_loss_shared2x2(self, decoder_output, target_indices, candidate_text_embeddings, label_similarity_sets,
                           area_embeddings, image_embeddings, W_text=1.0, W_image=0.5, W_smooth=2e2,
                           percent_image_sampling=0.7, k_distractors=50, pct_medium=0.0, pct_hard=0.75,
                           pct_rand=0.25, precision="auto", contrast_builder="reference", max_contrast=256):
    """``compute_loss`` of the tensor the decoder WOULD emit, taken before its tail (SURVEY 8f-1).

    The reference decoder ends in ``output_conv -> F.interpolate(nearest, x2) -> F.normalize``
    (utils/src/decoder.py:112-116), so ``compute_loss`` always sees 2x2 blocks of identical embeddings
    (quirk Q8).  Given ``decoder_output`` = the ``output_conv`` result [B,D,H/2,W/2] (what the decoder holds
    before line 113) and the full-resolution ``target_indices`` [B,H,W], this returns the same
    ``(total_loss, loss_info)`` as ``compute_loss(decoder_tail(decoder_output), ...)`` and back-propagates the
    same gradient into ``decoder_output`` -- without materialising the upsampled tensor:
      * text term: one embedding row per block with its four targets (rc_infonce_bf16_rep4): 1/4 of the GEMM
        work and HBM traffic, row norms taken inside the kernel;
      * smoothness: differences inside a block are exactly 0 and every low-resolution difference appears
        twice, so sum_hi = 2 sum_lo over the normalised low-resolution rows, divided by the full-resolution
        element counts of model.py:332-333.
    Same RNG streams as the reference (the pixel draw is over the full-resolution H*W)."""
    return _compute_loss(self, decoder_output, target_indices, candidate_text_embeddings, label_similarity_sets,
                         area_embeddings, image_embeddings, W_text, W_image, W_smooth, percent_image_sampling,
                         k_distractors, pct_medium, pct_hard, pct_rand, precision, shared2x2=True,
                         contrast_builder=contrast_builder, max_contrast=max_contrast)


def _compute_loss(self, pixel_embeddings, target_indices, candidate_text_embeddings, label_similarity_sets,
                  area_embeddings, image_embeddings, W_text, W_image, W_smooth, percent_image_sampling, k_distractors,
                  pct_medium, pct_hard, pct_rand, precision, shared2x2, contrast_builder="reference", max_contrast=256):
    device = pixel_embeddings.device
    log_tau_text = self.log_temperature_text
    log_tau_image = self.log_temperature_image

    text_loss = torch.zeros((), device=device)              # (a fill kernel: torch.tensor(0.0, device=...) is a blocking copy)
    fused_smooth = None
    if W_text > 0:
        fuse = W_smooth > 0 and pixel_embeddings.requires_grad and not shared2x2
        out = text_contrastive_loss(pixel_embeddings, target_indices, candidate_text_embeddings,
                                    label_similarity_sets, log_tau_text, percent_image_sampling,
                                    k_distractors, pct_medium, pct_hard, pct_rand, precision, return_aux=True,
                                    with_smoothness=fuse, shared2x2=shared2x2, contrast_builder=contrast_builder,
                                    max_contrast=max_contrast)
        text_loss = out[0]
        fused_smooth = out[1].get("smoothness")

    image_loss = torch.zeros((), device=device)
    if area_embeddings is not None and image_embeddings is not None and area_embeddings.shape[0] > 1:
        # "fp32" is the parity mode of every term; an explicit "bf16" asks for the tensor cores where a term's shape allows them
        image_loss = image_contrastive_loss(area_embeddings, image_embeddings, log_tau_image,
                                            precision if precision == "fp32" else "auto")
    elif W_image > 0:
        dummy = torch.ones((), device=device, requires_grad=True)          # model.py:325-326 (Q14)
        image_loss = dummy * torch.exp(log_tau_image) * 0.0

    smooth_loss = torch.zeros((), device=device)
    if W_smooth > 0 and shared2x2:
        B, D, h, w = pixel_embeddings.shape
        H, W = 2 * h, 2 * w
        dens = (B * D * H * (W - 1) / 2.0, B * D * (H - 1) * W / 2.0)
        if w % 8 == 0 and pixel_embeddings.dtype in (torch.float32, torch.bfloat16):
            # decoder.py:114 + model.py:332-333 as one operator: normalise (handed over from the area pooling when it ran on the
            # same tensor), TV sums, and ONE backward kernel through both
            smooth_loss = ops.smoothness_normalized(pixel_embeddings, denominators=dens)
        else:
            if (h * w) % 8 == 0:
                rows = ops.normalize_rows(pixel_embeddings)
            else:
                rows = torch.nn.functional.normalize(pixel_embeddings.float(), p=2, dim=1)
            smooth_loss = ops.smoothness(rows, denominators=dens)
    elif W_smooth > 0:
        smooth_loss = fused_smooth if fused_smooth is not None else ops.smoothness(pixel_embeddings)

    total = W_text * text_loss + W_image * image_loss + W_smooth * smooth_loss

    # one device->host transfer instead of the reference's six .item() syncs (model.py:343-349)
    stacked = torch.stack([total.detach().float(), text_loss.detach().float(), image_loss.detach().float(),
                           smooth_loss.detach().float(), torch.exp(log_tau_text.detach().float()),
                           torch.exp(log_tau_image.detach().float())])
    if contrast_builder == "device":
        # sync-free call: the six floats travel to pinned host memory asynchronously and are read on first access
        return total, LazyLossInfo(stacked, W_text, W_image, W_smooth)
    host = stacked.tolist()
    loss_info = {
        'total_loss': host[0],
        'text_contrastive_loss': host[1] if W_text > 0 else 0,
        'image_contrastive_loss': host[2] if W_image > 0 else 0,
        'smoothness_loss': host[3] if W_smooth > 0 else 0,
        'temperature_text': host[4],
        'temperature_image': host[5],
        'W_text': W_text,
        'W_image': W_image,
        'W_smooth': W_smooth,
    }
    return total, loss_info


class LazyLossInfo(dict):
    """``loss_info`` of ``compute_loss(contrast_builder="device")``: same keys as the reference's dict (model.py:343-353); the
    six device scalars are copied to pinned host memory asynchronously when the object is made and turned into Python floats
    the first time anything is read -- a training loop that logs every n-th step synchronises every n-th step."""
    _KEYS = ('total_loss', 'text_contrastive_loss', 'image_contrastive_loss', 'smoothness_loss', 'temperature_text',
             'temperature_image')

    _ring = []        # [pinned buffer, event of its last copy, weak reference to the owner]: cudaHostAlloc is slow and may block,
                      # so a buffer is reused once its copy has completed and its owner has read it (or is gone)

    @classmethod
    def _slot(cls):
        for slot in cls._ring:
            owner = slot[2]() if slot[2] is not None else None
            if (owner is None or owner._ready) and slot[1].query():
                return slot
        slot = [torch.empty(6, dtype=torch.float32, pin_memory=True), torch.cuda.Event(), None]
        cls._ring.append(slot)
        return slot

    def __init__(self, stacked: torch.Tensor, W_text, W_image, W_smooth):
        super().__init__()
        import weakref
        if torch.cuda.is_current_stream_capturing():
            # inside a CUDA-graph capture: the copy becomes a node of the graph (every replay refreshes the pinned buffer); an
            # event recorded during capture cannot be waited on from the host, so reading the values is the caller's business
            # AFTER it has synchronised with a replay -- until then this object reports itself as not ready
            self._host = torch.empty(6, dtype=torch.float32, pin_memory=True)
            self._host.copy_(stacked, non_blocking=True)
            self._event = None
        else:
            slot = self._slot()
            slot[2] = weakref.ref(self)
            self._host = slot[0]
            self._host.copy_(stacked, non_blocking=True)
            self._event = slot[1]
            self._event.record()
        self._weights = (W_text, W_image, W_smooth)
        self._ready = False

    def _fill(self):
        if not self._ready or self._event is None:       # (captured: re-read the pinned buffer every time -- replays refresh it)
            self._ready = True
            if self._event is not None:
                self._event.synchronize()
            else:
                torch.cuda.current_stream().synchronize()
            h = self._host.tolist()
            W_text, W_image, W_smooth = self._weights
            dict.update(self, {
                'total_loss': h[0],
                'text_contrastive_loss': h[1] if W_text > 0 else 0,
                'image_contrastive_loss': h[2] if W_image > 0 else 0,
                'smoothness_loss': h[3] if W_smooth > 0 else 0,
                'temperature_text': h[4],
                'temperature_image': h[5],
                'W_text': W_text,
                'W_image': W_image,
                'W_smooth': W_smooth,
            })

    def __getitem__(self, k): self._fill(); return dict.__getitem__(self, k)
    def __iter__(self): self._fill(); return dict.__iter__(self)
    def __len__(self): self._fill(); return dict.__len__(self)
    def __contains__(self, k): self._fill(); return dict.__contains__(self, k)
    def __repr__(self): self._fill(); return dict.__repr__(self)
    def __eq__(self, o): self._fill(); return dict.__eq__(self, o)
    def get(self, k, d=None): self._fill(); return dict.get(self, k, d)
    def keys(self): self._fill(); return dict.keys(self)
    def values(self): self._fill(); return dict.values(self)
    def items(self): self._fill(); return dict.items(self)
    def copy(self): self._fill(); return dict(self)
    __hash__ = None


class DepthCLIPLossMixin:
    """Mixin giving a model with ``log_temperature_text`` / ``log_temperature_image`` parameters the
    reference's ``compute_loss`` on the B200 kernels."""
    compute_loss = compute_loss
    compute_loss_shared2x2 = compute_loss_shared2x2
