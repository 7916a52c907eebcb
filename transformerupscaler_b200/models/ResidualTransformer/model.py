"""Drop-in replacement for the reference's models/ResidualTransformer/model.py::TransformerModel
(ctor model.py:69-112, forward :114-165): global attention over exactly 3600 tokens + learned pos_embed."""
from typing import Tuple

import torch
import torch.nn as nn

from .._base import EngineModel, GlobalTransformerBlock


class TransformerModel(EngineModel):
    ENGINE_MODEL = "ResidualTransformer"
    AUTOCAST_OUT_FP32 = True

    def __init__(self, in_channels=3, base_channels=64, embed_dim=64, transformer_dim=128, num_transformer_blocks=8,
                 num_heads=8, mlp_ratio=4.0, dropout=0.1):
        super().__init__()
        if (in_channels, base_channels, mlp_ratio) != (3, 64, 4.0) or transformer_dim != num_heads * 16 \
                or transformer_dim not in (128, 192):
            raise NotImplementedError("libtu_b200 kernels are specialised for in=3, base=64, mlp_ratio=4, head_dim=16")
        self.conv1 = nn.Conv2d(in_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(base_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.downsample = nn.Conv2d(base_channels, base_channels, kernel_size=3, stride=2, padding=1)
        self.patch_embed = nn.Conv2d(base_channels, transformer_dim, kernel_size=8, stride=8)
        self.token_H, self.token_W = 360 // 8, 640 // 8
        self.num_tokens = self.token_H * self.token_W
        self.pos_embed = nn.Parameter(torch.randn(1, self.num_tokens, transformer_dim))
        self.transformer_blocks = nn.ModuleList([
            GlobalTransformerBlock(transformer_dim, num_heads, mlp_ratio, dropout)
            for _ in range(num_transformer_blocks)])
        self.patch_unembed = nn.ConvTranspose2d(transformer_dim, base_channels, kernel_size=8, stride=8)
        self.decoder_conv1 = nn.Conv2d(base_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.decoder_conv2 = nn.Conv2d(base_channels, in_channels, kernel_size=3, stride=1, padding=1)

    def forward(self, x, res_out: Tuple[int, int] = (1080, 1920), upscale_factor: int = None, require_ratio: bool = True,
                in_layout: str = "chw", out_layout: str = "chw", yuv: str = "bt709", out=None):
        return super().forward(x, res_out, upscale_factor, require_ratio, in_layout, out_layout, yuv, out)
