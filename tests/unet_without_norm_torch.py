"""CPU ORACLE (second, independent restatement) -- TEST INFRASTRUCTURE ONLY: the 2-D UNet with --without_norm in
torch-CPU autograd, against the same reference lines as tests/unet_without_norm_ref.py but sharing no code with it
(loss and parameter conversion are oracle/unet_torch.py's own): every 3x3 conv is F.conv2d with its bias, then ReLU."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle import unet_torch as T
from oracle.unet_torch import to_torch_params  # noqa: F401


def forward(p: dict, images: torch.Tensor, cfg):
    """images NCHW -> logits NCHW (training and evaluation are the same graph)."""
    def block(x, scope):
        return F.relu(F.conv2d(x, p[f"{scope}/weights"].permute(3, 2, 0, 1), p[f"{scope}/biases"], padding=1))

    x = images
    skips = []
    for i in range(cfg.num_down_samples):
        for j in (1, 2):
            x = block(x, f"UNet/Encode{i + 1}/Repeat/convolution2d_{j}")
        skips.append(x)
        x = F.max_pool2d(x, 2)
    for j in (1, 2):
        x = block(x, f"UNet/ED-Bridge/ED-Bridge_{j}")
    for i in reversed(range(cfg.num_down_samples)):
        scope = f"UNet/Decode{i + 1}/Conv2d_transpose"
        up = F.relu(F.conv_transpose2d(x, p[f"{scope}/weights"].permute(3, 2, 0, 1), p[f"{scope}/biases"], stride=2))
        x = torch.cat((skips[i], up), dim=1)
        for j in (1, 2):
            x = block(x, f"UNet/Decode{i + 1}/Repeat/convolution2d_{j}")
    scope = "UNet/AdjustChannels"
    return F.conv2d(x, p[f"{scope}/weights"].permute(3, 2, 0, 1), p[f"{scope}/biases"])


def total_loss(p: dict, images, labels, cfg):
    """Data loss + slim L2 terms: weights always, biases unless --bias_decay (base.py:128-135)."""
    logits = forward(p, images, cfg)
    loss = T.data_loss(logits, labels, cfg)
    if cfg.weight_decay_rate > 0:
        names = [k for k in p if k.endswith("/weights") or (k.endswith("/biases") and not cfg.bias_decay)]
        loss = loss + cfg.weight_decay_rate * 0.5 * sum((p[k] ** 2).sum() for k in names)
    return loss, logits
