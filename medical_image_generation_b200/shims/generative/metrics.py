"""generative.metrics (train_ldm.py:32): the validation metrics of train_ldm.py:241-330. SSIMMetric and
MultiScaleSSIMMetric ARE the B200 implementations (medical_image_generation_b200.metrics, fused sm_100a kernel); FID
needs torch.hub feature networks and MMD is not implemented, so both stay placeholders that raise on construction."""
from medical_image_generation_b200.metrics import MultiScaleSSIMMetric, SSIMMetric
from ._placeholder import placeholder

FIDMetric = placeholder("metrics.FIDMetric", "validation metric, needs torch.hub feature networks")
MMDMetric = placeholder("metrics.MMDMetric", "validation metric")

__all__ = ["FIDMetric", "MMDMetric", "SSIMMetric", "MultiScaleSSIMMetric"]
