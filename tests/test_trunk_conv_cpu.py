"""CPU: the host side of the trunk convolution kernel (csrc/dbaz_trunk.cu) -- its tap tables, weight packing and
per-position bias -- rebuilds SimpleNN's padded and unpadded 3x3 convolutions exactly (float64 against F.conv2d)."""
import pytest
import torch
import torch.nn.functional as F


def _conv_by_taps(x, w, hi, wi, pad):
    """y[b, p] = sum over the table's taps of p: x[b, q] @ W_t^T, in the kernel's order of taps (float64)."""
    from dotsboxesaz_b200.engine import trunk_conv_taps
    from dotsboxesaz_b200.nn import trunk_conv_pack
    ho, wo, taps, order = trunk_conv_taps(hi, wi, pad)
    wp = trunk_conv_pack(w).double().view(9, 256, 256)  # [t][cout][cin]
    xf = x.double().reshape(x.shape[0], hi * wi, 256)
    y = torch.zeros((x.shape[0], ho * wo, 256), dtype=torch.float64)
    for p in range(ho * wo):
        for q, t in taps[p]:
            y[:, p] += xf[:, q] @ wp[t].t()
    return y.view(-1, ho, wo, 256), taps, order


@pytest.mark.parametrize("grid", [(4, 4), (6, 6), (3, 4), (8, 8), (2, 32), (1, 3)])
@pytest.mark.parametrize("pad", [1, 0])
def test_taps_and_packing_rebuild_conv2d(grid, pad):
    hi, wi = grid
    if pad == 0 and (hi < 3 or wi < 3):
        pytest.skip("no output position")
    g = torch.Generator().manual_seed(hi * 100 + wi + pad)
    x = torch.randn(3, hi, wi, 256, generator=g).to(torch.bfloat16)
    w = (torch.randn(256, 256, 3, 3, generator=g) * 0.02).to(torch.bfloat16).float()
    y, taps, order = _conv_by_taps(x, w, hi, wi, pad)
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), w.double(), None, padding=pad).permute(0, 2, 3, 1)
    assert y.shape == ref.shape
    assert (y - ref).abs().max().item() < 1e-9
    ho, wo = ref.shape[1], ref.shape[2]
    for p in range(ho * wo):
        oy, ox = divmod(p, wo)
        inside = [(ky, kx) for ky in range(3) for kx in range(3) if 0 <= oy + ky - pad < hi and 0 <= ox + kx - pad < wi]
        assert [t for _, t in taps[p]] == [3 * ky + kx for ky, kx in inside]  # every in-board tap once, in (ky, kx) order
    counts = [len(taps[p]) for p in order]
    assert sorted(order) == list(range(ho * wo)) and counts == sorted(counts, reverse=True)


def test_tap_counts_of_the_3x3_board():
    from dotsboxesaz_b200.engine import trunk_conv_taps
    ho, wo, taps, order = trunk_conv_taps(4, 4, 1)
    assert (ho, wo) == (4, 4) and sum(len(t) for t in taps) == 100  # (10 / 12)^2 of the 144 taps of the padded conv
    assert [len(taps[p]) for p in order] == [9] * 4 + [6] * 8 + [4] * 4
    ho, wo, taps, _ = trunk_conv_taps(4, 4, 0)
    assert (ho, wo) == (2, 2) and all(len(t) == 9 for t in taps)


def test_unsupported_grids_are_refused():
    from dotsboxesaz_b200.engine import trunk_conv_taps
    for args in [(9, 8, 1), (4, 4, 2), (2, 2, 0), (0, 4, 1)]:
        with pytest.raises(ValueError):
            trunk_conv_taps(*args)


def test_biases_are_the_library_plans():
    """bias_pos = bf16(conv(t, W) over the grid) and bias = bf16(b): the z map and bias of cuDNN's conv-add-bias-ReLU in the
    library plan.  With zero padding applied after the BatchNorm, conv(s x + t) + b = conv(s x) + bias_pos + bias up to
    those roundings; for pad 0 the map is one constant, folded into the bias."""
    from dotsboxesaz_b200.nn import trunk_conv_bias
    g = torch.Generator().manual_seed(5)
    w = torch.randn(256, 256, 3, 3, generator=g, dtype=torch.float64) * 0.02
    b, s, t = (torch.randn(256, generator=g, dtype=torch.float64) for _ in range(3))
    x = torch.randn(2, 256, 4, 4, generator=g, dtype=torch.float64)
    for pad in (1, 0):
        tmap = t.view(1, -1, 1, 1).expand(1, 256, 4, 4)
        bpos = F.conv2d(tmap, w, None, padding=pad)[0]
        bias_pos, bias = trunk_conv_bias(b, bpos, pad)
        for v in (bias_pos, bias):
            assert v.dtype == torch.float32 and torch.equal(v, v.to(torch.bfloat16).float())
        if pad == 1:
            assert torch.equal(bias_pos, bpos.permute(1, 2, 0).reshape(16, 256).to(torch.bfloat16).float())
            assert torch.equal(bias, b.to(torch.bfloat16).float())
        else:
            assert not bias_pos.any()
        ref = F.conv2d(x * s.view(1, -1, 1, 1) + t.view(1, -1, 1, 1), w, b, padding=pad)
        got = F.conv2d(x, w * s.view(1, -1, 1, 1), None, padding=pad)
        ho, wo = got.shape[2:]
        got = got + bias_pos.double().t().reshape(1, 256, ho, wo) + bias.double().view(1, 256, 1, 1)
        assert (got - ref).abs().max().item() < 0.05  # two bf16 roundings of values of a few units
