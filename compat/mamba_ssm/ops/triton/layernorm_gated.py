"""mamba_ssm.ops.triton.layernorm_gated.{RMSNorm, rmsnorm_fn} -> the B200 gated RMSNorm (reference SSD/MedSSD.py:36, used at
:268-269, 393-394)."""
from medical_image_classification_b200.ssd_combined import RMSNormGated as RMSNorm  # noqa: F401
from medical_image_classification_b200.ssd_combined import rmsnorm_fn  # noqa: F401
