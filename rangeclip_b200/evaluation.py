"""Drop-ins for the evaluation hot path: the tail of ``DepthUNet.predict`` (model.py:144-173) and
the metric accumulation / finalisation of ``validate_model`` (validate.py:88-139, 194-214).

``MetricAccumulator`` keeps everything on the device as int64 histograms; one transfer at the end
reproduces the reference's four dictionaries (including their insertion order, which fixes the
float summation order of the mIoU, SURVEY Q11) and therefore its four returned floats bit for bit.
Across ranks the histograms are summed with a single all-reduce (see distributed.py)."""
from __future__ import annotations

import random
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import ops

INT32_MAX = 2**31 - 1


def build_reduced_candidates(segmentation: torch.Tensor, total_candidates: int, num_negatives: int):
    """GT labels + ``random.sample`` negatives, sorted (model.py:147-156; Python RNG, Q6)."""
    if segmentation is None:
        raise ValueError("segmentation must be provided for reduced-candidate prediction")
    gt = set(torch.unique(segmentation).tolist())
    pool = list(set(range(total_candidates)) - gt)
    negatives = random.sample(pool, min(num_negatives, len(pool)))
    return sorted(list(gt.union(negatives)))


def device_candidates_supported(pixel_embeddings, total_candidates: int) -> bool:
    D = pixel_embeddings.shape[1]
    hw = pixel_embeddings[0, 0].numel() if pixel_embeddings.shape[0] else 0
    return pixel_embeddings.is_cuda and ops.topk_bf16_supported(D, hw) and 2 <= total_candidates <= 12000


def build_reduced_candidates_device(segmentation: torch.Tensor, candidate_text_embeddings: torch.Tensor, num_negatives: int):
    """model.py:147-161 without the host round trip (SURVEY 8f-2): the label histogram of the batch -> GT labels (label 0
    included, as ``torch.unique(segmentation)`` includes it) + ``num_negatives`` labels drawn without replacement from the
    rest (``rc_contrast_build``'s counter-based stream seeded from Python's ``random`` -- the generator the reference's
    ``random.sample`` uses; not its draws), sorted.  Returns (index list [K_cap] int64 padded with -1, bf16 rows [K_cap', D],
    kinfo int32 [4] with the set size first) -- all on the device, nothing read back."""
    total = candidate_text_embeddings.shape[0]
    seg = segmentation.reshape(segmentation.shape[0], -1)
    counts = torch.ops.rangeclip.sample_label_counts(seg, None, total)
    seed_dev = None
    if torch.cuda.is_current_stream_capturing():
        seed, seed_dev = 0, torch.randint(0, 2 ** 62, (1,), device=seg.device, dtype=torch.int64)
    else:
        seed = random.getrandbits(62)
    _, reduced, kinfo = torch.ops.rangeclip.contrast_build(counts, None, None, 0, int(num_negatives), total, seed, seed_dev, True)
    _, tb, _ = torch.ops.rangeclip.text_prepare(candidate_text_embeddings, reduced)
    return reduced, tb, kinfo


def _check_shared2x2(pixel_embeddings, segmentation):
    """``shared2x2=True`` takes the decoder's ``output_conv`` result [B,D,h,w] and the full-resolution segmentation [B,2h,2w]."""
    if pixel_embeddings.dim() != 4 or segmentation is None or not pixel_embeddings.is_cuda or not segmentation.is_cuda:
        raise RuntimeError("shared2x2: needs CUDA tensors, embeddings [B, D, h, w] and a segmentation")
    B, _, h, w = pixel_embeddings.shape
    if tuple(segmentation.shape) != (B, 2 * h, 2 * w):
        raise RuntimeError(f"shared2x2: the segmentation must be [B, 2h, 2w] = [{B}, {2 * h}, {2 * w}], "
                           f"got {list(segmentation.shape)}")


def predict_from_embeddings(pixel_embeddings, candidate_text_embeddings, segmentation, num_negatives=300, top_k=5,
                            precision="auto", candidate_builder="reference", shared2x2=False):
    """model.py:144-173 given the decoder output: returns (topk ids [B,k,H,W] int64 in the ORIGINAL
    index space, L2-normalised embeddings).  The [B,Kr,HW] logits are never materialised.
    ``candidate_builder="device"``: the reduced candidate set is built on the GPU and its size stays there
    (``build_reduced_candidates_device``): no host synchronisation; a pixel gets -1 where fewer than ``top_k`` candidates exist.
    ``shared2x2=True``: ``pixel_embeddings`` is the decoder's ``output_conv`` result [B,D,H/2,W/2], before the tail
    (nearest x2 -> normalize, decoder.py:113-115) that makes every 2x2 block one embedding; the top-k is ranked once per
    block (rc_eval_topk_bf16_rep4, tensor cores only) and the ids come out at full resolution [B,k,H,W].  The second
    result is then the L2-normalised half-resolution rows."""
    total = candidate_text_embeddings.shape[0]
    if shared2x2:
        if precision == "fp32":
            raise ValueError("shared2x2=True runs on the tensor cores only (precision 'auto' or 'bf16')")
        _check_shared2x2(pixel_embeddings, segmentation)
        if candidate_builder == "device" and device_candidates_supported(pixel_embeddings, total):
            reduced, tb, kinfo = build_reduced_candidates_device(segmentation, candidate_text_embeddings, num_negatives)
            topk = ops.eval_topk_rep4(pixel_embeddings, tb, reduced, min(top_k, total), k_dev=kinfo)
        else:
            reduced = build_reduced_candidates(segmentation, total, num_negatives)
            index_tensor = torch.tensor(reduced, device=pixel_embeddings.device)
            t_norm, _, _ = ops.text_prepare(candidate_text_embeddings, index_tensor, want_f32=True)
            topk = ops.eval_topk_rep4(pixel_embeddings, ops.text_to_bf16(t_norm)[0], index_tensor, min(top_k, len(reduced)))
        return topk, F.normalize(pixel_embeddings, dim=1)
    if candidate_builder == "device" and segmentation is not None and device_candidates_supported(pixel_embeddings, total) \
            and precision != "fp32":
        reduced, tb, kinfo = build_reduced_candidates_device(segmentation, candidate_text_embeddings, num_negatives)
        topk = ops.eval_topk_dyn(pixel_embeddings, tb, kinfo, reduced, min(top_k, total))
        return topk, F.normalize(pixel_embeddings, dim=1)
    reduced = build_reduced_candidates(segmentation, total, num_negatives)
    index_tensor = torch.tensor(reduced, device=pixel_embeddings.device)
    t_norm, _, _ = ops.text_prepare(candidate_text_embeddings, index_tensor, want_f32=True)
    topk = ops.eval_topk(pixel_embeddings, t_norm, index_tensor, min(top_k, len(reduced)), precision)
    return topk, F.normalize(pixel_embeddings, dim=1)


def segment_from_embeddings(pixel_embeddings, text_embeddings, log_temperature, top_k=1, candidates=None, shared2x2=False):
    """Open-vocabulary segmentation of a decoder output against a vocabulary of the caller's choosing -- no ground truth,
    no RNG, no host synchronisation.  ``text_embeddings`` [V,D] (normalised here, as ``F.normalize``); ``candidates``: an
    optional 1-D tensor of vocabulary rows to rank (default: all V); ``log_temperature``: a 0-d tensor (e.g.
    ``model.log_temperature_text``) or a float.  Returns (ids [B,k,H,W] int64 in the vocabulary's index space, cosine
    [B,k,H,W] fp32, prob [B,k,H,W] fp32): the top ``k = min(top_k, K)`` rows of every pixel by cosine similarity, their
    cosines, and their softmax probabilities over all K candidate rows at the temperature -- CLIP-style confidences; the
    cosine is the score to reject "none of these" with.  One tensor-core launch (rc_eval_topk_scores_bf16); the [B,K,HW]
    logits are never materialised.  ``shared2x2=True``: ``pixel_embeddings`` is the decoder's ``output_conv`` result
    [B,D,H/2,W/2] (see ``predict_from_embeddings``) and the outputs are full resolution.  Shapes outside the kernel
    (top_k > 8, D % 64 != 0, D > 1024, H*W % 8 != 0) raise."""
    if shared2x2 and pixel_embeddings.dim() != 4:
        raise RuntimeError("segment_from_embeddings: shared2x2=True takes the output_conv result [B, D, h, w]")
    if not (pixel_embeddings.is_cuda and text_embeddings.is_cuda):
        raise RuntimeError("segment_from_embeddings: needs CUDA tensors (no CPU fallback exists)")
    dev = pixel_embeddings.device
    if candidates is not None:
        if candidates.dim() != 1:
            raise RuntimeError("segment_from_embeddings: candidates must be a 1-D tensor of vocabulary rows")
        index_map = candidates.to(device=dev, dtype=torch.int64)
    else:
        index_map = torch.arange(text_embeddings.shape[0], device=dev)
    _, tb, _ = ops.text_prepare(text_embeddings, index_map if candidates is not None else None, want_f32=False, want_bf16=True)
    if isinstance(log_temperature, torch.Tensor):
        log_tau = log_temperature.detach().to(device=dev, dtype=torch.float32).reshape(1)
    else:
        log_tau = torch.full((1,), float(log_temperature), device=dev, dtype=torch.float32)
    return torch.ops.rangeclip.eval_topk_scores(pixel_embeddings, tb, index_map, int(top_k), log_tau, bool(shared2x2))


def predict_and_accumulate(pixel_embeddings, candidate_text_embeddings, segmentation, accumulator, num_negatives=300, top_k=5,
                           batch_index=None, want_ids=True, candidate_builder="reference", shared2x2=False):
    """``predict_from_embeddings`` + ``MetricAccumulator.update`` as one fused kernel per batch: same reduced candidate
    set (same ``random.sample`` draw, Q6), same ids, same histograms -- the ids never make the round trip through HBM
    between the two steps.  Returns (topk ids or None, L2-normalised embeddings).  ``candidate_builder="device"``: see
    ``predict_from_embeddings`` -- the whole validation batch then runs without a host synchronisation.
    ``shared2x2=True``: ``pixel_embeddings`` is the ``output_conv`` result [B,D,H/2,W/2] (see ``predict_from_embeddings``);
    every full-resolution pixel of ``segmentation`` [B,H,W] is counted, as on the upsampled tensor."""
    total = candidate_text_embeddings.shape[0]
    if shared2x2:
        _check_shared2x2(pixel_embeddings, segmentation)
    if candidate_builder == "device" and device_candidates_supported(pixel_embeddings, total):
        reduced, tb, kinfo = build_reduced_candidates_device(segmentation, candidate_text_embeddings, num_negatives)
        ids = accumulator.update_from_device_candidates(pixel_embeddings, tb, kinfo, reduced, segmentation, min(top_k, total),
                                                        batch_index=batch_index, want_ids=want_ids, shared2x2=shared2x2)
        return ids, F.normalize(pixel_embeddings, dim=1)
    reduced = build_reduced_candidates(segmentation, total, num_negatives)
    index_tensor = torch.tensor(reduced, device=pixel_embeddings.device)
    t_norm, _, _ = ops.text_prepare(candidate_text_embeddings, index_tensor, want_f32=True)
    ids = accumulator.update_from_embeddings(pixel_embeddings, t_norm, index_tensor, segmentation, min(top_k, len(reduced)),
                                             batch_index=batch_index, want_ids=want_ids, shared2x2=shared2x2)
    return ids, F.normalize(pixel_embeddings, dim=1)


def predict(self, depth_maps, candidate_text_embeddings, segmentation, num_negatives=300, top_k=5, candidate_builder="reference"):
    """Drop-in for ``DepthUNet.predict`` (model.py:119-175): backbone in PyTorch, tail on the kernels.
    ``candidate_builder="device"`` (an addition): see ``predict_from_embeddings``."""
    self.eval()
    B, _, H, W = depth_maps.shape
    with torch.no_grad():
        with torch.autocast("cuda", enabled=depth_maps.is_cuda):
            _, encoder_features, final_feature_map = self.depth_encoder(depth_maps)
            pixel_embeddings = self.depth_decoder(final_feature_map, encoder_features, (H, W))
        topk, pixel_embeddings = predict_from_embeddings(pixel_embeddings.float(), candidate_text_embeddings,
                                                         segmentation, num_negatives, top_k, candidate_builder=candidate_builder)
        return topk, pixel_embeddings, self.temperature_text


class MetricAccumulator:
    """Device-side state of validate.py:59-69 / 88-139."""

    def __init__(self, equivalence_tensor: torch.Tensor, equiv_class_map: torch.Tensor, device=None):
        device = device if device is not None else equiv_class_map.device
        self.E = equivalence_tensor.to(device=device, dtype=torch.uint8).contiguous()
        self.cmap = equiv_class_map.to(device=device, dtype=torch.int64).contiguous()
        self.C = int(self.cmap.numel())
        self.acc = torch.zeros(4, self.C, device=device, dtype=torch.int64)        # I1, U1, IK, UK
        self.counters = torch.zeros(3, device=device, dtype=torch.int64)           # correct1, correctk, total
        self.first_seen = torch.full((self.C,), INT32_MAX, device=device, dtype=torch.int32)
        self.n_batches = 0
        self._hist = torch.zeros(5, self.C, device=device, dtype=torch.int64)

    def update(self, segmentation: torch.Tensor, pred_topk: torch.Tensor, batch_index: Optional[int] = None) -> None:
        """One validation batch: segmentation [B,H,W], pred_topk [B,k,H,W] (no host sync)."""
        self._hist.zero_()
        ops.eval_hist(segmentation, pred_topk, self.E, self.cmap, self._hist, self.counters)
        ops.eval_fold(self._hist, self.n_batches if batch_index is None else batch_index, self.acc, self.first_seen)
        self.n_batches += 1

    def update_from_embeddings(self, pixel_embeddings: torch.Tensor, t_norm: torch.Tensor, index_tensor: torch.Tensor,
                               segmentation: torch.Tensor, top_k: int = 5, batch_index: Optional[int] = None,
                               t_bf16=None, want_ids: bool = True, shared2x2: bool = False):
        """One validation batch straight from the pixel embeddings: ONE kernel does the top-k over the text rows and the
        metric histograms (rc_eval_topk_hist_bf16); the ids are returned only if ``want_ids``.  ``shared2x2=True``: the
        embeddings are the ``output_conv`` result [B,D,H/2,W/2] of the full-resolution ``segmentation`` (rc_eval_topk_bf16_rep4)."""
        self._hist.zero_()
        if shared2x2:
            _check_shared2x2(pixel_embeddings, segmentation)
            tb = t_bf16 if t_bf16 is not None else ops.text_to_bf16(t_norm)[0]
            ids = ops.eval_topk_rep4(pixel_embeddings, tb, index_tensor, top_k, segmentation, self.E, self.cmap, self._hist,
                                     self.counters, want_ids=want_ids)
        else:
            ids = ops.eval_topk_hist(pixel_embeddings, t_norm, index_tensor, top_k, segmentation, self.E, self.cmap, self._hist,
                                     self.counters, t_bf16=t_bf16, want_ids=want_ids)
        ops.eval_fold(self._hist, self.n_batches if batch_index is None else batch_index, self.acc, self.first_seen)
        self.n_batches += 1
        return ids

    def update_from_device_candidates(self, pixel_embeddings, t_bf16, kinfo, index_tensor, segmentation, top_k: int = 5,
                                      batch_index: Optional[int] = None, want_ids: bool = True, shared2x2: bool = False):
        """``update_from_embeddings`` for a candidate set whose size lives on the device (``build_reduced_candidates_device``)."""
        self._hist.zero_()
        if shared2x2:
            _check_shared2x2(pixel_embeddings, segmentation)
            ids = ops.eval_topk_rep4(pixel_embeddings, t_bf16, index_tensor, top_k, segmentation, self.E, self.cmap, self._hist,
                                     self.counters, k_dev=kinfo, want_ids=want_ids)
        else:
            ids = ops.eval_topk_dyn(pixel_embeddings, t_bf16, kinfo, index_tensor, top_k, segmentation, self.E, self.cmap,
                                    self._hist, self.counters, want_ids=want_ids)
        ops.eval_fold(self._hist, self.n_batches if batch_index is None else batch_index, self.acc, self.first_seen)
        self.n_batches += 1
        return ids

    def state(self) -> Dict[str, torch.Tensor]:
        return dict(acc=self.acc, counters=self.counters, first_seen=self.first_seen)

    def valid_mask(self, last_segmentation: Optional[torch.Tensor]) -> torch.Tensor:
        """uint8 [C]: classes present in a batch's ground truth -- the label filter of validate.py:206-210 (Q11)."""
        mask = torch.zeros(self.C, device=self.cmap.device, dtype=torch.uint8)
        if last_segmentation is not None:
            mask[self.cmap[last_segmentation.reshape(-1).to(self.cmap.device)]] = 1
        return mask

    def finalize(self, last_segmentation: Optional[torch.Tensor] = None, valid_mask: Optional[torch.Tensor] = None) -> Dict[str, object]:
        """validate.py:194-214: mIoU over labels present in the LAST batch's GT (Q11), averaged in the
        reference's dict insertion order (batch of first appearance, then label id); accuracies.  ``valid_mask``
        (uint8 [C]) replaces ``last_segmentation`` when the globally last batch lives on another rank."""
        mask = valid_mask if valid_mask is not None else self.valid_mask(last_segmentation)
        valid = set(torch.nonzero(mask).reshape(-1).tolist())
        return finalize_metrics(self.acc, self.counters, self.first_seen, valid)


def finalize_metrics(acc_t: torch.Tensor, counters_t: torch.Tensor, first_seen_t: torch.Tensor, valid: set) -> Dict[str, object]:
    """Host-side finalisation (validate.py:194-214) from the integer state; one device->host transfer."""
    acc = acc_t.cpu().tolist()
    counters = counters_t.cpu().tolist()
    first = first_seen_t.cpu().tolist()
    order = sorted((fs, lab) for lab, fs in enumerate(first) if fs != INT32_MAX)
    dicts = {name: {} for name in ("intersection_top1", "union_top1", "intersection_topk", "union_topk")}
    for _, lab in order:
        dicts["intersection_top1"][lab] = acc[0][lab]
        dicts["union_top1"][lab] = acc[1][lab]
        dicts["intersection_topk"][lab] = acc[2][lab]
        dicts["union_topk"][lab] = acc[3][lab]

    def miou(inter, union):
        ious = [inter[lab] / union[lab] for lab in union if lab in valid and union[lab] > 0]
        return sum(ious) / len(ious) if ious else 0.0

    total = counters[2]
    return {
        "mIoU_t1": miou(dicts["intersection_top1"], dicts["union_top1"]),
        "mIoU_tk": miou(dicts["intersection_topk"], dicts["union_topk"]),
        "pixel_accuracy_t1": counters[0] / total if total > 0 else 0.0,
        "pixel_accuracy_tk": counters[1] / total if total > 0 else 0.0,
        "correct_pixels_top1": counters[0], "correct_pixels_topk": counters[1], "total_pixels": total,
        **dicts,
    }


def _log(s: str, filepath: Optional[str] = None) -> None:
    """Same contract as utils/src/log_utils.py:7-30: print, and append to ``filepath`` when given."""
    print(s)
    if filepath is not None:
        import os
        os.makedirs(os.path.dirname(filepath) or ".", exist_ok=True)
        with open(filepath, "a+") as f:
            f.write(s + "\n")


def _unwrap(model):
    return model.module if hasattr(model, "module") else model


def validate_model(model, clip_model, clip_processor, candidate_text_embeddings, candidate_labels, equivalence_tensor,
                   equiv_class_map, similarity_sets, curriculum, dataloader, step, best_results, device, w_text=1.0,
                   w_image=0.5, w_smooth=2e2, summary_writer=None, n_sample_per_summary=16, log_path=None,
                   all_reduce=False):
    """Drop-in for ``validate_model`` (validate.py:34-266).  Same arguments, same ``best_results`` keys and log
    lines; the per-batch metric loops (validate.py:88-139) run as two kernels per batch with no host sync, and the
    finalisation (validate.py:194-214) reads the integer state back once.  ``all_reduce=True`` (an addition) sums
    the state over the default process group first, so that every rank may validate its own shard of the batches:
    ``dataloader`` then yields the batches ``distributed.shard_batches`` assigns to this rank (round robin: the i-th
    local batch is global batch rank + i * world_size), the per-label first-appearance order is kept in GLOBAL batch
    indices, and the class filter of the final mean (the LAST batch's ground truth, Q11) comes from the rank that owns
    the globally last batch -- every rank then returns the single-process result bit for bit."""
    from .losses import compute_loss as _compute_loss
    from .pooling import prepare_image_contrast_data as _prepare

    model.eval()
    acc = MetricAccumulator(equivalence_tensor, equiv_class_map, device=device)
    totals = [0.0, 0.0, 0.0, 0.0]
    n_batches = 0
    segmentation = None
    temperature_text = None
    core = _unwrap(model)
    rank, world = 0, 1
    if all_reduce:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
    with torch.no_grad():
        for batch in dataloader:
            depth = batch['depth'].to(device, non_blocking=True)
            image_processed = batch['image'].to(device, non_blocking=True)
            segmentation = batch['segmentation'].to(device, non_blocking=True)
            object_bbox = batch['object_bbox'].to(device, non_blocking=True)
            object_label = batch['object_label']
            pred_topk, pixel_embeddings, temperature_text = core.predict(
                depth_maps=depth, candidate_text_embeddings=candidate_text_embeddings, segmentation=segmentation,
                num_negatives=50, top_k=5)
            acc.update(segmentation, pred_topk, batch_index=rank + n_batches * world)
            area_embeddings, image_embeddings = _prepare(
                image_processed_batch=image_processed, object_bbox_batch=object_bbox, object_label_batch=object_label,
                segmentation_batch=segmentation, pixel_embeddings_batch=pixel_embeddings, clip_image_encoder=clip_model,
                clip_processor=clip_processor, device=device)
            loss_fn = core.compute_loss if hasattr(core, "compute_loss") else (lambda **kw: _compute_loss(core, **kw))
            _, loss_info = loss_fn(
                pixel_embeddings=pixel_embeddings, target_indices=segmentation,
                candidate_text_embeddings=candidate_text_embeddings, label_similarity_sets=similarity_sets,
                area_embeddings=area_embeddings, image_embeddings=image_embeddings, W_text=w_text, W_image=w_image,
                W_smooth=w_smooth, k_distractors=50, pct_medium=curriculum['pct_medium'], pct_hard=curriculum['pct_hard'],
                pct_rand=curriculum['pct_rand'])
            totals[0] += loss_info['total_loss']
            totals[1] += loss_info.get('text_contrastive_loss', 0)
            totals[2] += loss_info.get('image_contrastive_loss', 0)
            totals[3] += loss_info.get('smoothness_loss', 0)
            n_batches += 1
    valid_mask = acc.valid_mask(segmentation)
    if all_reduce:
        from .distributed import all_reduce_metrics, global_last_batch_mask
        all_reduce_metrics(acc)
        valid_mask = global_last_batch_mask(valid_mask, rank + (n_batches - 1) * world if n_batches else -1)
        tot = torch.tensor(totals + [float(n_batches)], device=acc.acc.device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tot)                  # the logged losses are averages over all batches of all ranks
        totals, n_batches = tot[:4].tolist(), int(tot[4])
    fin = acc.finalize(valid_mask=valid_mask)
    miou_top1, miou_topk = fin["mIoU_t1"], fin["mIoU_tk"]
    pixel_acc_top1, pixel_acc_topk = fin["pixel_accuracy_t1"], fin["pixel_accuracy_tk"]
    avg = [t / max(n_batches, 1) for t in totals]
    _log(f"[Val] [Step {step}] Top-1 pixel accuracy (equiv): {pixel_acc_top1:.4f}", log_path)
    _log(f"[Val] [Step {step}] Top-k pixel accuracy (equiv): {pixel_acc_topk:.4f}", log_path)
    _log(f"[Val] [Step {step}] Top-1 mIoU (equiv): {miou_top1:.4f}", log_path)
    _log(f"[Val] [Step {step}] Top-k mIoU (equiv): {miou_topk:.4f}", log_path)
    _log(f"[Val] Step {step} | # of labels in Top-1 mIoU: {len(fin['intersection_top1'])}", log_path)
    _log(f"[Val] Step {step} | # of labels in Top-k mIoU: {len(fin['intersection_topk'])}", log_path)
    _log(f"[Val] Step {step} | Loss: {avg[0]:.4f}, Text Contrastive: {avg[1]:.4f}, Image Contrastive: {avg[2]:.4f}, "
         f"Smoothness: {avg[3]:.4f}", log_path)
    if best_results.get("mIoU_tk", 0) < miou_topk:
        best_results.update({
            "loss": avg[0], "step": step, "mIoU_t1": miou_top1, "mIoU_tk": miou_topk,
            "pixel_accuracy_t1": pixel_acc_top1, "pixel_accuracy_tk": pixel_acc_topk, "temperature": temperature_text,
            "avg_text_contrastive_loss": avg[1], "avg_image_contrastive_loss": avg[2], "avg_smoothness_loss": avg[3]})
    _log(f"Best validation loss: {best_results['loss']:.4f} at step {best_results['step']}", log_path)
    if summary_writer is not None:
        summary_writer.add_scalar("val/loss", avg[0], global_step=step)
        for name, val in (("val/pixel_accuracy", pixel_acc_top1), ("val/pixel_accuracy_tk", pixel_acc_topk),
                          ("val/mIoU", miou_top1), ("val/mIoU_tk", miou_topk),
                          ("val/avg_text_contrastive_loss", avg[1]), ("val/avg_image_contrastive_loss", avg[2]),
                          ("val/avg_smoothness_loss", avg[3])):
            summary_writer.add_scalar(name, val, global_step=step)
    return best_results
