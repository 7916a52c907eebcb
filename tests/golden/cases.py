"""Golden-vector cases shared by make_golden.py (reference run) and the tests (oracle / engine)."""
CASES = {
    # WindowTransformer: token grid 4x6 -> one padded 8x8 window; default-style res_out (1.5x)
    "window_72x104_r1p5": dict(model="WindowTransformer", shape=(1, 3, 72, 104), wseed=1, xseed=11,
                               kw=dict(res_out=(108, 156))),
    # batch 2, integer factor, 4x5 tokens
    "window_64x80_x2": dict(model="WindowTransformer", shape=(2, 3, 64, 80), wseed=2, xseed=12,
                            kw=dict(upscale_factor=2)),
    # odd input: ceil stride-2, floor patch embed, crop before the skip add; 2x3 windows
    "window_131x189_odd": dict(model="WindowTransformer", shape=(1, 3, 131, 189), wseed=3, xseed=13,
                               kw=dict(res_out=(200, 280))),
    "fast_40x56_x2": dict(model="FastTransformer", shape=(1, 3, 40, 56), wseed=4, xseed=14, kw=dict(upscale_factor=2)),
    "fast_40x56_x3": dict(model="FastTransformer", shape=(1, 3, 40, 56), wseed=4, xseed=15, kw=dict(upscale_factor=3)),
    "fast_40x56_x4": dict(model="FastTransformer", shape=(1, 3, 40, 56), wseed=4, xseed=16, kw=dict(upscale_factor=4)),
    "fast_24x32_x6": dict(model="FastTransformer", shape=(1, 3, 24, 32), wseed=5, xseed=17, kw=dict(upscale_factor=6)),
    # H, W not multiples of 8 -> reflect pad before patch embed, crop after unembed
    "fast_36x52_x2_reflect": dict(model="FastTransformer", shape=(2, 3, 36, 52), wseed=6, xseed=18,
                                  kw=dict(upscale_factor=2)),
    # res_out path: factor = ceil(1.5) = 2, then antialiased Resize down to res_out
    "fast_40x56_res60x84": dict(model="FastTransformer", shape=(1, 3, 40, 56), wseed=7, xseed=19,
                                kw=dict(res_out=(60, 84))),
    # ResidualTransformer only accepts 3600 tokens -> 720p input; store every 8th pixel
    "residual_720p_1080p": dict(model="ResidualTransformer", shape=(1, 3, 720, 1280), wseed=8, xseed=20,
                                kw=dict(res_out=(1080, 1920)), stride=8),
}

# Every BASELINE.json configuration at its real size (VERDICT r01 item 1).  The reference's pre-clamp output is stored on a
# stride-13 lattice (13 is coprime to every sub-pixel factor 2/3/4/6 and to the 8-pixel patch, so all PixelShuffle phases,
# patch positions and strip seams are sampled) plus dense 40x40 crops of the four corners (border handling: conv padding,
# reflect pad, bicubic clamping, the folded up1 ring).  `frames` = which frames of the batch are stored.
_CORNERS = ((0, 0), (0, -40), (-40, 0), (-40, -40))
FULLSIZE = {
    # cfg2 / cfg3: WindowTransformer 720p -> 1080p, batch 8 (first and last frame stored)
    "window_720p_1080p_b8": dict(model="WindowTransformer", shape=(8, 3, 720, 1280), wseed=70, xseed=170, kw=dict(res_out=(1080, 1920)),
                                 stride=13, frames=(0, 7), crops=_CORNERS),
    # cfg4: FastTransformer multi-scale sweep on 720p input
    "fast_720p_x2": dict(model="FastTransformer", shape=(1, 3, 720, 1280), wseed=71, xseed=171, kw=dict(upscale_factor=2),
                         stride=13, frames=(0,), crops=_CORNERS),
    "fast_720p_x3": dict(model="FastTransformer", shape=(1, 3, 720, 1280), wseed=72, xseed=172, kw=dict(upscale_factor=3),
                         stride=13, frames=(0,), crops=_CORNERS),
    "fast_720p_x4": dict(model="FastTransformer", shape=(1, 3, 720, 1280), wseed=73, xseed=173, kw=dict(upscale_factor=4),
                         stride=13, frames=(0,), crops=_CORNERS),
    "fast_720p_x6": dict(model="FastTransformer", shape=(1, 3, 720, 1280), wseed=74, xseed=174, kw=dict(upscale_factor=6),
                         stride=13, frames=(0,), crops=_CORNERS),
    # cfg5b: FastTransformer 1080p -> 4K (token grid 135x240 -> padded to 136x240; reflect pad of the 1080-row map)
    "fast_1080p_x2": dict(model="FastTransformer", shape=(1, 3, 1080, 1920), wseed=75, xseed=175, kw=dict(upscale_factor=2),
                          stride=13, frames=(0,), crops=_CORNERS),
    # cfg5a: ResidualTransformer 720p -> 4K, the call of speed_test.py:64
    "residual_720p_4k": dict(model="ResidualTransformer", shape=(2, 3, 720, 1280), wseed=76, xseed=176, kw=dict(res_out=(2160, 3840)),
                             stride=13, frames=(0, 1), crops=_CORNERS),
    # FastTransformer through its res_out path at 720p -> 1080p: factor 2, then the antialiased Resize (F:323-325)
    "fast_720p_res1080p": dict(model="FastTransformer", shape=(1, 3, 720, 1280), wseed=77, xseed=177, kw=dict(res_out=(1080, 1920)),
                               stride=13, frames=(0,), crops=_CORNERS),
}


def sample_fullsize(t, c):
    """(lattice, [crops]) views of a (B, 3, H, W) array the way the FULLSIZE goldens store it"""
    st = c["stride"]
    t = t[list(c["frames"])]
    H, W = t.shape[-2:]
    crops = []
    for y0, x0 in c["crops"]:
        y0, x0 = (H + y0 if y0 < 0 else y0), (W + x0 if x0 < 0 else x0)
        crops.append(t[..., y0:y0 + 40, x0:x0 + 40])
    return t[..., ::st, ::st], crops


# the seeded ragged-shape sweep (tests/golden/make_ragged.py): pre-clamp output on the lattice of the smallest stride among
# RAGGED_STRIDES that keeps it within RAGGED_LATTICE values (1, or a prime >= 5: coprime to every sub-pixel factor 2/3/4/6 and to
# the 8-pixel patch, so all phases are sampled), plus dense 8x8 crops of the four corners
RAGGED_LATTICE = 2048
RAGGED_STRIDES = (1, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37, 41)
RAGGED_CORNERS = ((0, 0), (0, -8), (-8, 0), (-8, -8))


def ragged_sample(t):
    """(stride, lattice, [crops]) of a (B, 3, H, W) array the way the ragged-sweep goldens store it"""
    B, C, H, W = t.shape
    st = next(s for s in RAGGED_STRIDES if B * C * -(-H // s) * -(-W // s) <= RAGGED_LATTICE)
    crops = []
    for y0, x0 in RAGGED_CORNERS:
        y0, x0 = (H + y0 if y0 < 0 else y0), (W + x0 if x0 < 0 else x0)
        crops.append(t[..., y0:y0 + 8, x0:x0 + 8])
    return st, t[..., ::st, ::st], crops


# natural-image fixtures (tests/golden/make_natural.py): uint8 LR frame, uint8 HR target, the reference's fp32 output as fp16
NATURAL = {
    "natural_window_96x176_r1p5": dict(model="WindowTransformer", wseed=31, kw=dict(res_out=(144, 264))),
    "natural_fast_96x176_x2": dict(model="FastTransformer", wseed=32, kw=dict(upscale_factor=2)),
}

# whole 720p natural frames (make_natural.py --full): HR target and reference output stored on a stride-3 lattice of the output
NATURAL_FULL = {
    "natural_window_720p_1080p": dict(model="WindowTransformer", wseed=33, kw=dict(res_out=(1080, 1920))),
    "natural_fast_720p_x2": dict(model="FastTransformer", wseed=34, kw=dict(upscale_factor=2)),
    "natural_residual_720p_1080p": dict(model="ResidualTransformer", wseed=35, kw=dict(res_out=(1080, 1920))),
}
