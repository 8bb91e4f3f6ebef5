"""CPU: the part of oracle/vit_oracle.py that restates reference code (pixel gather) is checked against that code's output
(tests/golden/vit_gather.pt, tools/make_golden_vit_gather.py); the bilinear-gather formula used by the CUDA kernel is checked
against F.interpolate on random maps.  (The timm trunk is unpinned, see the oracle header.)"""
import os

import torch
import torch.nn.functional as F

from oracle import vit_oracle as vo


def gather_inputs():
    g = torch.Generator().manual_seed(0)
    img = torch.randn(2, 16, 20, 24, generator=g)
    choose = torch.randint(0, 20 * 24, (2, 50), generator=g)
    return img, choose


def test_chosen_pixel_feats_matches_reference_function(golden_dir):
    want = torch.load(os.path.join(golden_dir, "vit_gather.pt"), weights_only=False)["feats"]
    assert torch.equal(vo.chosen_pixel_feats(*gather_inputs()), want)


def test_bilinear_gather_formula_matches_interpolate():
    """the closed form the CUDA kernel evaluates (4 taps of the token-major upscaling output, align_corners=False weights)"""
    g = torch.Generator().manual_seed(1)
    B, C, G, sub, H = 2, 8, 14, 4, 224
    up = torch.randn(B, G * G, sub * sub * C, generator=g)
    fmap = up.reshape(B, G, G, sub, sub, C).permute(0, 5, 1, 3, 2, 4).contiguous().reshape(B, C, G * sub, G * sub)
    ref = F.interpolate(fmap, (H, H), mode="bilinear", align_corners=False)
    choose = torch.randint(0, H * H, (B, 300), generator=g)
    choose[0, :4] = torch.tensor([0, H - 1, H * (H - 1), H * H - 1])          # corners: clamped source indices
    want = vo.chosen_pixel_feats(ref, choose)
    Hs = G * sub
    Y, X = choose // H, choose % H
    sy = (0.25 * (Y.float() + 0.5) - 0.5).clamp(min=0)
    sx = (0.25 * (X.float() + 0.5) - 0.5).clamp(min=0)
    y0, x0 = sy.floor().long(), sx.floor().long()
    y1, x1 = y0 + (y0 < Hs - 1).long(), x0 + (x0 < Hs - 1).long()
    ly1, lx1 = sy - y0, sx - x0

    def tap(h, w):
        tok = (h // sub) * G + (w // sub)
        blk = (h % sub) * sub + (w % sub)
        idx = (tok[:, :, None] * (sub * sub * C) + blk[:, :, None] * C + torch.arange(C)).reshape(B, -1)
        return torch.gather(up.reshape(B, -1), 1, idx).reshape(B, -1, C)

    got = ((1 - ly1)[..., None] * ((1 - lx1)[..., None] * tap(y0, x0) + lx1[..., None] * tap(y0, x1)) +
           ly1[..., None] * ((1 - lx1)[..., None] * tap(y1, x0) + lx1[..., None] * tap(y1, x1)))
    torch.testing.assert_close(got, want, atol=1e-6, rtol=1e-5)
