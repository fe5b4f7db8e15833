"""The library's fp32 NCHW -> bf16 NHWC tile pass in its two identity-prologue forms: the head's feature pack and the
discriminator's gradient layout with a padded, zero-filled channel pitch.  Bit-equality with torch's cast on ragged and
unaligned shapes and special values (-m gpu)."""
import pytest
import torch

from rnd_semantic_segmentation_b200 import _lib

pytestmark = pytest.mark.gpu


def special_values(shape, seed):
    """Random normals with NaN, +-Inf, -0, subnormals and values on bf16 rounding ties sprinkled in."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, device="cuda", generator=g)
    flat = x.view(-1)
    n = flat.numel()
    specials = torch.tensor([float("nan"), float("inf"), float("-inf"), -0.0, 1e-40, -3e-39, 1.0 + 2.0 ** -8,
                             1.0 + 3 * 2.0 ** -8, 3.4e38], device="cuda")
    idx = torch.randint(0, n, (max(n // 50, len(specials)),), device="cuda", generator=g)
    flat[idx] = specials[torch.arange(idx.numel(), device="cuda") % len(specials)]
    return x


def same_bits(a, b):
    """Bit-equal bf16 tensors; a NaN must meet a NaN (the conversion instruction writes the canonical NaN, torch keeps more
    of the payload), every other value -- -0, infinities, subnormals -- must match bit for bit."""
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    return torch.equal(a.view(torch.int16)[~na], b.view(torch.int16)[~nb])


@pytest.mark.parametrize("shape", [(1, 64, 64, 128),        # bench-like, vector path
                                   (2, 256, 65, 129),       # ragged: hw % 4 != 0, partial pixel tiles, N > 1
                                   (3, 40, 7, 9),           # Cin % 8 == 0 but not % 32, hw = 63
                                   (2, 72, 12, 12)])        # Cin = 72: a partial channel tile, hw % 4 == 0
def test_pack_bit_equal(shape):
    x = special_values(shape, 1)
    N, Cin, h, w = shape
    Xp = _lib.aspp_pack_features(x)
    ref = x.to(torch.bfloat16).permute(0, 2, 3, 1).reshape(N * h * w, Cin)
    assert same_bits(Xp, ref)


def test_pack_unaligned_base():
    N, Cin, h, w = 2, 64, 16, 32
    buf = special_values((N * Cin * h * w + 1,), 2)
    x = buf[1:].view(N, Cin, h, w)                          # 4-byte aligned only: the scalar-load path
    assert x.data_ptr() % 16 != 0
    Xp = _lib.aspp_pack_features(x)
    assert same_bits(Xp, x.to(torch.bfloat16).permute(0, 2, 3, 1).reshape(N * h * w, Cin))


@pytest.mark.parametrize("shape,pitch", [((2, 38, 64, 128), 40), ((1, 38, 9, 13), 40), ((2, 19, 5, 7), 24)])
def test_disc_layout_pitch_zero_fill(shape, pitch):
    g = special_values(shape, 3)
    out = _lib.nchw_to_nhwc_bf16(g, pitch)
    N, C, h, w = shape
    ref = torch.zeros(N, h, w, pitch, dtype=torch.bfloat16, device="cuda")
    ref[..., :C] = g.to(torch.bfloat16).permute(0, 2, 3, 1)
    assert same_bits(out, ref)
