"""oracle/vit_oracle.py -- TEST INFRASTRUCTURE ONLY.

CPU restatement (torch fp32) of the PEM RGB branch, PEM/model/feature_extraction.py:17-181:
    vit_forward         ViT.forward :21-35 on top of timm.models.vision_transformer.VisionTransformer
    vit_ae_forward      ViT_AE.forward :97-111 (up_type 'linear')
    get_img_feats       ViTEncoder.get_img_feats :166-167 = get_chosen_pixel_feats (PEM/utils/model_utils.py:69-81)
Parity status:
  * everything below the ViT trunk (concatenation of the 4 pyramid levels, output_upscaling, the reshape / permute to the
    56 x 56 map, F.interpolate(bilinear, align_corners=False), the pixel gather) follows reference code, and the gather is
    checked against the output of model_utils.get_chosen_pixel_feats (tests/golden/vit_gather.pt) by tests/test_oracle_vit.py;
  * the trunk itself is timm's VisionTransformer, which the reference neither vendors nor pins (PEM/dependencies.sh:4,
    environment.yaml:34) and which is absent here: PARITY UNPINNED.  The restatement follows timm >= 0.6 semantics:
    patch_embed = Conv2d(3, D, 16, 16) -> flatten(2).transpose(1,2); _pos_embed = cat(cls_token, x) + pos_embed;
    norm_pre = Identity; blocks x = x + attn(norm1(x)), x = x + mlp(norm2(x)) with LayerNorm eps 1e-6, attention
    softmax(q k^T / sqrt(64)) v over (B, heads, N, 64), MLP fc1 -> GELU(erf) -> fc2; self.norm applied to the tapped outputs.
"""
import math
from typing import Dict, List

import torch
import torch.nn.functional as F

SD = Dict[str, torch.Tensor]

from sam6d_b200.synth import make_vit_state_dict as make_state_dict  # noqa: E402,F401  (seeded weights: shared with bench.py)


def vit_forward(sd: SD, x: torch.Tensor, depth: int, num_heads: int, prefix="rgb_net.vit.") -> List[torch.Tensor]:
    p = prefix
    D = sd[p + "cls_token"].shape[-1]
    x = F.conv2d(x, sd[p + "patch_embed.proj.weight"], sd[p + "patch_embed.proj.bias"], stride=16).flatten(2).transpose(1, 2)
    x = torch.cat([sd[p + "cls_token"].expand(x.shape[0], -1, -1), x], dim=1) + sd[p + "pos_embed"]
    n = depth // 4
    taps = [depth - 1, depth - n - 1, depth - 2 * n - 1, depth - 3 * n - 1]
    out = []
    hd = D // num_heads
    for i in range(depth):
        b = f"{p}blocks.{i}."
        h = F.layer_norm(x, (D,), sd[b + "norm1.weight"], sd[b + "norm1.bias"], 1e-6)
        B, N, _ = h.shape
        qkv = F.linear(h, sd[b + "attn.qkv.weight"], sd[b + "attn.qkv.bias"]).reshape(B, N, 3, num_heads, hd).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        a = ((q * hd ** -0.5) @ k.transpose(-2, -1)).softmax(dim=-1)
        h = (a @ v).transpose(1, 2).reshape(B, N, D)
        x = x + F.linear(h, sd[b + "attn.proj.weight"], sd[b + "attn.proj.bias"])
        h = F.layer_norm(x, (D,), sd[b + "norm2.weight"], sd[b + "norm2.bias"], 1e-6)
        h = F.linear(F.gelu(F.linear(h, sd[b + "mlp.fc1.weight"], sd[b + "mlp.fc1.bias"])), sd[b + "mlp.fc2.weight"], sd[b + "mlp.fc2.bias"])
        x = x + h
        if i in taps:
            out.append(F.layer_norm(x, (D,), sd[p + "norm.weight"], sd[p + "norm.bias"], 1e-6))
    return out


def upscale_map(sd: SD, vit_outs: List[torch.Tensor], H: int, W: int, out_dim: int, prefix="rgb_net."):
    """ViT_AE.forward :97-111 after the trunk -> ((B,out_dim,H,W) map, cls tokens)"""
    B = vit_outs[0].shape[0]
    cls_tokens = vit_outs[-1][:, 0, :].contiguous()
    x = torch.cat([l[:, 1:, :].contiguous() for l in vit_outs], dim=2)
    x = F.linear(x, sd[prefix + "output_upscaling.weight"], sd[prefix + "output_upscaling.bias"])
    x = x.reshape(B, 14, 14, 4, 4, out_dim).permute(0, 5, 1, 3, 2, 4).contiguous().reshape(B, -1, 56, 56)
    x = F.interpolate(x, (H, W), mode="bilinear", align_corners=False)
    return x, cls_tokens


def chosen_pixel_feats(img: torch.Tensor, choose: torch.Tensor) -> torch.Tensor:
    """get_chosen_pixel_feats, PEM/utils/model_utils.py:69-81"""
    B, C, H, W = img.shape
    img = img.reshape(B, C, H * W)
    return torch.gather(img, 2, choose.unsqueeze(1).repeat(1, C, 1)).contiguous().transpose(1, 2).contiguous()


def get_img_feats(sd: SD, img: torch.Tensor, choose: torch.Tensor, depth=12, num_heads=12, out_dim=256, prefix="rgb_net.") -> torch.Tensor:
    outs = vit_forward(sd, img, depth, num_heads, prefix + "vit.")
    fmap, _ = upscale_map(sd, outs, img.shape[2], img.shape[3], out_dim, prefix)
    return chosen_pixel_feats(fmap, choose)
