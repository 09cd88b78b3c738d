"""Regularisers next to the hot path (SURVEY.md 8(f)2): the projection / repulsion losses of DSS/training/losses.py on top
of the B200 K-NN; and the image objective of the training step as a fused CUDA op (image_loss.dr_image_loss)."""
from .image_loss import DrLoss, dr_image_loss  # noqa: F401
from .losses import BaseLoss, IouLoss, L1Loss, L2Loss, ProjectionLoss, RepulsionLoss, SurfaceLoss  # noqa: F401
