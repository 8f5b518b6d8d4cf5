"""CPU/fp32 restatement of the reference networks on the Diff-UNet inference path.

TEST INFRASTRUCTURE ONLY (oracle).  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
``--impl reference`` legs may import this module; the product package never does.

What is restated (functional style over a flat state dict keyed exactly like the reference checkpoint):

  * ``init_state_dict``      parameter creation in the reference's construction order so that
                             ``torch.manual_seed(s)`` yields bit-identical weights to
                             ``DiffUNet(in_channels, out_channels)`` (models/diff_unet.py:33-35).
  * ``encoder_forward``      BasicUNetEncoder.forward   models/basic_unet/pretrained/basic_unet.py:496-512
  * ``time_embedding``       TimeStepEmbedder.forward    models/diffusion/utils.py:6-54
  * ``denoiser_forward``     BasicUNetRDenoiser.forward  models/basic_unet/denoiser.py:284-312
                             (TwoConv :63-67, Down :105-108, UpCat :173-194)

Parity pin: tests/test_oracle_golden.py checks these against tests/golden/*.npz, which
oracle/make_golden.py produced by running the unmodified reference (oracle/ref_loader.py); one full-resolution
case is held to same-machine tolerances (rel-L2 < 1e-6 for the encoder and one denoiser call).
"""
from __future__ import annotations

import hashlib
import math
from collections import OrderedDict
from typing import Dict, List, Sequence

import torch
import torch.nn.functional as F

DEFAULT_FEATURES = (64, 64, 128, 256, 512, 64)  # models/diff_unet.py:17
LEAKY_SLOPE = 0.1                                # models/diff_unet.py:35, pretrained/basic_unet.py:428
IN_EPS = 1e-5                                    # nn.InstanceNorm3d default, used via MONAI ("instance", affine)
TEMB_DIM = 128                                   # models/diffusion/utils.py:34
TEMB_HID = 512                                   # models/diffusion/utils.py:35, denoiser.py:51


# --------------------------------------------------------------------------------------------------------------
# parameter creation (same RNG consumption order as the reference constructors)
# --------------------------------------------------------------------------------------------------------------
def _conv_params(sd, prefix, cin, cout, k):
    m = torch.nn.Conv3d(cin, cout, k, padding=k // 2)
    sd[prefix + ".weight"] = m.weight.detach()
    sd[prefix + ".bias"] = m.bias.detach()


def _convblock_params(sd, prefix, cin, cout):
    # MONAI Convolution = conv (consumes RNG) + ADN(InstanceNorm affine: ones/zeros, no RNG)
    _conv_params(sd, prefix + ".conv", cin, cout, 3)
    sd[prefix + ".adn.N.weight"] = torch.ones(cout)
    sd[prefix + ".adn.N.bias"] = torch.zeros(cout)


def _linear_params(sd, prefix, cin, cout):
    m = torch.nn.Linear(cin, cout)
    sd[prefix + ".weight"] = m.weight.detach()
    sd[prefix + ".bias"] = m.bias.detach()


def _twoconv_params(sd, prefix, cin, cout, with_temb):
    if with_temb:  # denoiser.py:51-52 creates temb_proj before the convs
        _linear_params(sd, prefix + ".temb_proj", TEMB_HID, cout)
    _convblock_params(sd, prefix + ".conv_0", cin, cout)
    _convblock_params(sd, prefix + ".conv_1", cout, cout)


def init_state_dict(in_channels: int = 1, out_channels: int = 16,
                    features: Sequence[int] = DEFAULT_FEATURES, seed: int | None = 0) -> "OrderedDict[str, torch.Tensor]":
    """Random-init weights exactly as ``torch.manual_seed(seed); DiffUNet(in_channels=..., out_channels=...)``."""
    f = list(features)
    assert len(f) == 6
    if seed is not None:
        torch.manual_seed(seed)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    # embed_model = BasicUNetEncoder(3, in_channels, 2, features)      pretrained/basic_unet.py:491-494
    _twoconv_params(sd, "embed_model.conv_0", in_channels, f[0], False)
    for d in range(4):
        _twoconv_params(sd, f"embed_model.down.{d}.convs", f[d], f[d + 1], False)
    # model = BasicUNetRDenoiser(3, out_channels + 1, out_channels, features)      denoiser.py:268-282
    _linear_params(sd, "model.temb.dense.0", TEMB_DIM, TEMB_HID)
    _linear_params(sd, "model.temb.dense.1", TEMB_HID, TEMB_HID)
    _twoconv_params(sd, "model.conv_0", out_channels + 1, f[0], True)
    for lvl in range(1, 5):
        _twoconv_params(sd, f"model.down_{lvl}.convs", f[lvl - 1], f[lvl], True)
    # UpCat(in, cat, out, halves): upsample first, then TwoConv(cat + up, out)      denoiser.py:157-171
    ups = [(4, f[4], f[3], f[3], True), (3, f[3], f[2], f[2], True), (2, f[2], f[1], f[1], True),
           (1, f[1], f[0], f[5], False)]
    for lvl, cin, ccat, cout, halves in ups:
        cup = cin // 2 if halves else cin
        m = torch.nn.ConvTranspose3d(cin, cup, 2, stride=2)
        sd[f"model.upcat_{lvl}.upsample.deconv.weight"] = m.weight.detach()
        sd[f"model.upcat_{lvl}.upsample.deconv.bias"] = m.bias.detach()
        _twoconv_params(sd, f"model.upcat_{lvl}.convs", ccat + cup, cout, True)
    _conv_params(sd, "model.final_conv", f[5], out_channels, 1)
    return sd


# --------------------------------------------------------------------------------------------------------------
# forward restatement
# --------------------------------------------------------------------------------------------------------------
def _conv_in_act(sd, prefix, x):
    """MONAI Convolution with ADN ordering NDA: conv3x3x3(pad 1, bias) -> InstanceNorm(affine) -> LeakyReLU(0.1)."""
    x = F.conv3d(x, sd[prefix + ".conv.weight"], sd[prefix + ".conv.bias"], padding=1)
    x = F.instance_norm(x, weight=sd[prefix + ".adn.N.weight"], bias=sd[prefix + ".adn.N.bias"], eps=IN_EPS)
    return F.leaky_relu(x, LEAKY_SLOPE)


def _swish(x):
    return x * torch.sigmoid(x)  # models/diffusion/utils.py:27-29


def _twoconv(sd, prefix, x, temb=None):
    x = _conv_in_act(sd, prefix + ".conv_0", x)
    if temb is not None:  # denoiser.py:65
        bias = F.linear(_swish(temb), sd[prefix + ".temb_proj.weight"], sd[prefix + ".temb_proj.bias"])
        x = x + bias[:, :, None, None, None]
    return _conv_in_act(sd, prefix + ".conv_1", x)


def encoder_forward(sd: Dict[str, torch.Tensor], image: torch.Tensor) -> List[torch.Tensor]:
    """BasicUNetEncoder.forward (pretrained/basic_unet.py:496-512): five feature maps."""
    xs = [_twoconv(sd, "embed_model.conv_0", image)]
    for d in range(4):
        xs.append(_twoconv(sd, f"embed_model.down.{d}.convs", F.max_pool3d(xs[-1], 2)))
    return xs


def sinusoid_embedding(t: torch.Tensor, dim: int = TEMB_DIM) -> torch.Tensor:
    """get_timestep_embedding (models/diffusion/utils.py:6-25)."""
    half = dim // 2
    freq = torch.exp(torch.arange(half, dtype=torch.float32) * -(math.log(10000) / (half - 1))).to(t.device)
    arg = t.float()[:, None] * freq[None, :]
    return torch.cat([torch.sin(arg), torch.cos(arg)], dim=1)


def time_embedding(sd, t: torch.Tensor) -> torch.Tensor:
    """TimeStepEmbedder.forward (models/diffusion/utils.py:49-54)."""
    e = sinusoid_embedding(t).to(sd["model.temb.dense.0.weight"].dtype)  # no-op in fp32; lets the oracle run in fp64
    e = F.linear(e, sd["model.temb.dense.0.weight"], sd["model.temb.dense.0.bias"])
    return F.linear(_swish(e), sd["model.temb.dense.1.weight"], sd["model.temb.dense.1.bias"])


def temb_bias_table(sd, timesteps: Sequence[int]) -> Dict[str, torch.Tensor]:
    """Per-TwoConv additive bias ``temb_proj(swish(temb(t)))`` for each t: {block prefix: [len(t), Cout]}."""
    temb = time_embedding(sd, torch.tensor(list(timesteps), dtype=torch.int64))
    blocks = ["model.conv_0"] + [f"model.down_{i}.convs" for i in range(1, 5)] + \
             [f"model.upcat_{i}.convs" for i in (4, 3, 2, 1)]
    return {b: F.linear(_swish(temb), sd[b + ".temb_proj.weight"], sd[b + ".temb_proj.bias"]) for b in blocks}


def denoiser_forward(sd, x: torch.Tensor, t: torch.Tensor, image: torch.Tensor,
                     embeddings: List[torch.Tensor], return_intermediates: bool = False):
    """BasicUNetRDenoiser.forward (denoiser.py:284-312).  ``t`` holds ORIGINAL timesteps (after the
    _WrappedModel remap, respace.py:123-129)."""
    temb = time_embedding(sd, t)
    h = torch.cat([image, x], dim=1)                                                   # :298
    x0 = _twoconv(sd, "model.conv_0", h, temb) + embeddings[0]                         # :300
    x1 = _twoconv(sd, "model.down_1.convs", F.max_pool3d(x0, 2), temb) + embeddings[1]
    x2 = _twoconv(sd, "model.down_2.convs", F.max_pool3d(x1, 2), temb) + embeddings[2]
    x3 = _twoconv(sd, "model.down_3.convs", F.max_pool3d(x2, 2), temb) + embeddings[3]
    x4 = _twoconv(sd, "model.down_4.convs", F.max_pool3d(x3, 2), temb) + embeddings[4]

    def upcat(lvl, low, skip):
        up = F.conv_transpose3d(low, sd[f"model.upcat_{lvl}.upsample.deconv.weight"],
                                sd[f"model.upcat_{lvl}.upsample.deconv.bias"], stride=2)   # :181
        # :183-189 replicate-pad by one voxel where the skip is odd-sized; patch edges are multiples of 16
        pad = []
        for i in range(3):
            pad += [0, 1 if skip.shape[-i - 1] != up.shape[-i - 1] else 0]
        up = F.pad(up, pad, "replicate")
        return _twoconv(sd, f"model.upcat_{lvl}.convs", torch.cat([skip, up], dim=1), temb)  # :190

    u4 = upcat(4, x4, x3)
    u3 = upcat(3, u4, x2)
    u2 = upcat(2, u3, x1)
    u1 = upcat(1, u2, x0)
    logits = F.conv3d(u1, sd["model.final_conv.weight"], sd["model.final_conv.bias"])  # :311
    if return_intermediates:
        return logits, {"x0": x0, "x1": x1, "x2": x2, "x3": x3, "x4": x4, "u4": u4, "u3": u3, "u2": u2, "u1": u1}
    return logits


def state_dict_fingerprint(sd) -> Dict[str, str]:
    """Bit-exact fingerprint per tensor: sha256 of dtype, shape and raw bytes.  (Float64 sums are not portable: their
    last bit follows the order in which torch's CPU reduction splits the tensor, which depends on the thread count.)"""
    out = {}
    for k, v in sd.items():
        t = v.detach().cpu().contiguous()
        h = hashlib.sha256(f"{t.dtype} {tuple(t.shape)}".encode())
        h.update(t.numpy().tobytes())
        out[k] = h.hexdigest()
    return out
