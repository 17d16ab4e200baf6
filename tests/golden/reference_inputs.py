"""Seeded inputs of the reference-run fixtures in tests/golden/.

The fixtures store the reference's outputs (sampled where the full tensors would be too large) but
not the inputs: both the generators (make_reference_golden.py, make_reference_geglu_golden.py) and
tests/test_reference_pin.py rebuild them here from a CPU generator, which gives the same values on
every machine.  Each fixture also stores `input_check`, a strided sample of every input, so that a
change in the recipe or in torch's CPU generator fails loudly instead of comparing unrelated data.
"""
import math

import torch

GN_CASES = [
    # (tag, shape, transform of x)
    ("selftest_2x320x32x32", (2, 320, 32, 32), None),
    ("unet_2x1280x8x8", (2, 1280, 8, 8), None),
    ("large_mean_1x320x16x16", (1, 320, 16, 16), "mean50"),
    ("outlier_channel_1x640x8x8", (1, 640, 8, 8), "outlier"),
]
LN_CASES = [("selftest_recipe_257x1280", (257, 1280)), ("tokens_300x320", (300, 320)),
            ("tokens_64x640", (64, 640))]

GEGLU_SHAPES = [(4608, 320, 1280), (1152, 640, 2560), (300, 1280, 5120), (18432, 320, 1280)]

SAMPLES = 4096  # output elements kept per tensor where a whole tensor would be too large


def input_check(*tensors):
    """About 1024 evenly strided values of each tensor, as fp32."""
    return [t.flatten()[::max(1, t.numel() // 1024)].float() for t in tensors]


def sample_index(numel, seed, count=SAMPLES):
    """Sorted indices of `count` of `numel` elements (all of them when there are fewer)."""
    if numel <= count:
        return torch.arange(numel, dtype=torch.int32)
    g = torch.Generator().manual_seed(seed)
    return torch.randperm(numel, generator=g)[:count].sort().values.to(torch.int32)


def norm_cases():
    """GroupNorm cases (x NCHW fp16, weight, bias, groups, eps), then LayerNorm cases (x [rows, c]),
    drawn in this order from one generator: the self-test configuration of the reference's
    group_norm.py (randn(2, 320, 32, 32) fp16, G = 32, randn affine, eps 1e-5), UNet-shaped
    extras (1280 channels at 8x8, a large-mean input, an outlier channel), and LayerNorm on the
    self-test's data recipe of layer_norm.py (x = -2.3 + 0.5 randn, rand affine) at UNet widths."""
    g = torch.Generator().manual_seed(20260923)

    def randn(*s):
        return torch.randn(*s, generator=g)

    gn, ln = [], []
    for tag, shape, tf in GN_CASES:
        x = randn(*shape)
        if tf == "mean50":
            x = x + 50.0
        elif tf == "outlier":
            x[:, 7] *= 100.0
        x = x.half()
        w, b = randn(shape[1]).half(), randn(shape[1]).half()
        gn.append({"tag": tag, "x": x, "weight": w, "bias": b, "groups": 32, "eps": 1e-5})
    for tag, (m, n) in LN_CASES:
        weight = torch.rand(n, generator=g).half()
        bias = torch.rand(n, generator=g).half()
        x = (-2.3 + 0.5 * randn(m, n)).half()
        ln.append({"tag": tag, "x": x, "weight": weight, "bias": bias, "eps": 1e-5})
    return gn, ln


def geglu_inputs(dtype, shape):
    """x [m, k], weight [2 * inner, k] (hidden rows first, gate rows second) and bias of one UNet
    GEGLU projection, on the CPU."""
    m, k, inner = shape
    g = torch.Generator().manual_seed(m + k)
    x = torch.randn(m, k, generator=g).to(dtype)
    w = (torch.randn(2 * inner, k, generator=g) / math.sqrt(k)).to(dtype)
    b = (torch.randn(2 * inner, generator=g) * 0.1).to(dtype)
    return x, w, b
