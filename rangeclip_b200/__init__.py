"""rangeclip_b200 -- B200 (sm_100a) kernels for the DepthCLIP (jinryan/RangeCLIP) loss and
evaluation hot path, behind the reference's own Python call signatures.

    compute_loss / DepthCLIPLossMixin        model.py:178-355
    compute_loss_shared2x2                   model.py:178-355 below the decoder tail (decoder.py:112-116)
    masked_average_pooling                   model.py:15-56
    prepare_image_contrast_data              dataloader.py:205-305
    predict / predict_from_embeddings        model.py:119-175
    segment_from_embeddings                  open-vocabulary inference: top-k labels, cosines and softmax confidences
    MetricAccumulator, validate_model        validate.py:34-266

The CUDA code lives in ``csrc/`` and is reached through the C ABI in ``include/rangeclip_b200.h``
(``_lib.py``).  Importing the package does not require a GPU; calling an op does.
"""
from .losses import (DepthCLIPLossMixin, build_contrast_indices, compute_loss, compute_loss_shared2x2,
                     image_contrastive_loss, text_contrastive_loss)
from .pooling import masked_average_pooling, pool_objects_per_image, prepare_image_contrast_data
from .evaluation import (MetricAccumulator, build_reduced_candidates, finalize_metrics, predict, predict_and_accumulate,
                         predict_from_embeddings, segment_from_embeddings, validate_model)
from . import ops

__all__ = [
    "DepthCLIPLossMixin", "build_contrast_indices", "compute_loss", "compute_loss_shared2x2", "image_contrastive_loss",
    "text_contrastive_loss", "masked_average_pooling", "pool_objects_per_image",
    "prepare_image_contrast_data", "MetricAccumulator", "build_reduced_candidates", "predict",
    "predict_from_embeddings", "segment_from_embeddings", "predict_and_accumulate", "finalize_metrics", "validate_model", "ops",
]
