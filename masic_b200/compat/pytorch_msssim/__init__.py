"""`import pytorch_msssim` shim: the two functions the reference's eval loop uses, on the masic_b200 MS-SSIM kernel."""
from masic_b200.msssim_compat import __version__, ms_ssim, ssim  # noqa: F401
