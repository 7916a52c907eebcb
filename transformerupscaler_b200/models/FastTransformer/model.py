"""Drop-in replacement for the reference's models/FastTransformer/model.py::TransformerModel
(ctor model.py:189-229, forward :231-327): no downsample, reflect-padded patch embed, 6 window blocks of
dim 192, sub-pixel (conv + PixelShuffle) branches for scales {2,3,4,6}, optional antialiased Resize."""
from typing import Tuple

import torch
import torch.nn as nn

from .._base import EngineModel, WindowTransformerBlock
from .utils import BasicConv, Upsampler, default_conv


class TransformerModel(EngineModel):
    ENGINE_MODEL = "FastTransformer"
    AUTOCAST_OUT_FP32 = False      # under autocast the reference's last ops are convs -> low-precision output

    def __init__(self, in_channels: int = 3, base_channels: int = 64, transformer_dim: int = 192,
                 num_window_blocks: int = 6, num_heads: int = 12, mlp_ratio: float = 4.0, dropout: float = 0.1,
                 window_size: int = 8):
        super().__init__()
        if (in_channels, base_channels, window_size, mlp_ratio) != (3, 64, 8, 4.0) or transformer_dim != num_heads * 16 \
                or transformer_dim not in (128, 192):
            raise NotImplementedError("libtu_b200 kernels are specialised for in=3, base=64, window=8, mlp_ratio=4, "
                                      "head_dim=16 and transformer_dim in {128,192}")
        self.conv1 = nn.Conv2d(in_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = nn.Conv2d(base_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.up1 = Upsampler(conv=default_conv, n_feats=base_channels)
        self.up1_conv = BasicConv(base_channels, 3, 3, 1, 1)
        self.final_upscale = Upsampler(conv=default_conv, n_feats=3)
        self.final_upscale_conv = default_conv(3, 3, 3)
        self.patch_embed = nn.Conv2d(base_channels, transformer_dim, kernel_size=8, stride=8)
        self.window_size = window_size
        self.window_blocks = nn.ModuleList([
            WindowTransformerBlock(transformer_dim, window_size, num_heads, mlp_ratio, dropout)
            for _ in range(num_window_blocks)])
        self.patch_unembed = nn.ConvTranspose2d(transformer_dim, base_channels, kernel_size=8, stride=8)
        self.decoder_conv1 = nn.Conv2d(base_channels, base_channels, kernel_size=3, stride=1, padding=1)
        self.decoder_conv2 = nn.Conv2d(base_channels, in_channels, kernel_size=3, stride=1, padding=1)

    def forward(self, x: torch.Tensor, res_out: Tuple[int, int] = (1080, 1920), upscale_factor: int = None,
                require_ratio: bool = True, in_layout: str = "chw", out_layout: str = "chw", yuv: str = "bt709", out=None):
        return super().forward(x, res_out, upscale_factor, require_ratio, in_layout, out_layout, yuv, out)
