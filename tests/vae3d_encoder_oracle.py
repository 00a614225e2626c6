"""CPU reference for VAE3DLarge.encode (the original project's encoder nn.Sequential and fc_mu / fc_logvar, networks.py:2210-2244,
ResidualBlock3D networks.py:471-505), restated with F.conv3d in eval mode.  Imported by the encoder tests and by
tools/bench_vae3d_encode.py; not a test module itself."""
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.pointdiff_oracle import _bn3d_eval

SD = Dict[str, torch.Tensor]


# VAE3DLarge.encode (networks.py:2210-2244, encode just above decode at :2327): (index in the encoder nn.Sequential, kind, cin, cout)
VAE3D_ENCODER = [(0, "conv", 1, 32), (2, "res", 32, 64), (3, "down", 64, 64), (5, "res", 64, 128), (6, "down", 128, 128),
                 (8, "res", 128, 256), (9, "down", 256, 256), (11, "res", 256, 512), (12, "valid", 512, 512)]


def vae3d_encoder_state_dict_spec(latent_dim: int = 256, prefix: str = "vae"):
    """(key, shape, kind) of the encoder half of VAE3DLarge's state_dict (encoder, fc_mu, fc_logvar)."""
    spec = []
    for idx, kind, ci, co in VAE3D_ENCODER:
        name = f"{prefix}.encoder.{idx}"
        if kind == "conv":
            spec += [(f"{name}.weight", (co, ci, 3, 3, 3), "w"), (f"{name}.bias", (co,), "b")]
        elif kind in ("down", "valid"):       # Conv3d(k=4, s=2, p=1) / Conv3d(k=4, p=0)
            spec += [(f"{name}.weight", (co, ci, 4, 4, 4), "w"), (f"{name}.bias", (co,), "b")]
        else:                                 # ResidualBlock3D(ci -> co): conv1, bn1, conv2, bn2, downsample (1x1)
            for j, cj in ((1, ci), (2, co)):
                spec += [(f"{name}.conv{j}.weight", (co, cj, 3, 3, 3), "w"), (f"{name}.conv{j}.bias", (co,), "b"),
                         (f"{name}.bn{j}.weight", (co,), "bn_w"), (f"{name}.bn{j}.bias", (co,), "bn_b"),
                         (f"{name}.bn{j}.running_mean", (co,), "bn_m"), (f"{name}.bn{j}.running_var", (co,), "bn_v"),
                         (f"{name}.bn{j}.num_batches_tracked", (), "nbt")]
            spec += [(f"{name}.downsample.weight", (co, ci, 1, 1, 1), "w"), (f"{name}.downsample.bias", (co,), "b")]
    for head in ("fc_mu", "fc_logvar"):
        spec += [(f"{prefix}.{head}.weight", (latent_dim, 512), "w"), (f"{prefix}.{head}.bias", (latent_dim,), "b")]
    return spec


def make_synthetic_vae3d_encoder_checkpoint(seed: int = 43, latent_dim: int = 256, prefix: str = "vae") -> SD:
    """Seeded encoder weights with variance-preserving scales (fan-in = cin x kernel volume) and randomised BatchNorm
    statistics, as make_synthetic_vae3d_decoder_checkpoint does for the decoder."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for key, shape, kind in vae3d_encoder_state_dict_spec(latent_dim, prefix):
        if kind == "w":
            fan = 1
            for n in shape[1:]:
                fan *= n
            sd[key] = torch.randn(shape, generator=g) * (2.0 / fan) ** 0.5
        elif kind == "b":
            sd[key] = torch.randn(shape, generator=g) * 0.05
        elif kind == "bn_w":
            sd[key] = 1.0 + 0.2 * torch.randn(shape, generator=g)
        elif kind in ("bn_b", "bn_m"):
            sd[key] = 0.1 * torch.randn(shape, generator=g)
        elif kind == "bn_v":
            sd[key] = 0.5 + torch.rand(shape, generator=g)
        else:
            sd[key] = torch.tensor(0, dtype=torch.int64)
    return sd


def _res_block3d_down(sd: SD, name: str, x: torch.Tensor) -> torch.Tensor:
    """ResidualBlock3D.forward, networks.py:488-505 (cin != cout: the shortcut is the biased 1x1 `downsample` conv)."""
    out = F.relu(_bn3d_eval(sd, f"{name}.bn1", F.conv3d(x, sd[f"{name}.conv1.weight"], sd[f"{name}.conv1.bias"], padding=1)))
    out = _bn3d_eval(sd, f"{name}.bn2", F.conv3d(out, sd[f"{name}.conv2.weight"], sd[f"{name}.conv2.bias"], padding=1))
    return F.relu(out + F.conv3d(x, sd[f"{name}.downsample.weight"], sd[f"{name}.downsample.bias"]))


def vae3d_encode(sd: SD, x: torch.Tensor, prefix: str = "vae", taps: Optional[dict] = None):
    """VAE3DLarge.encode: occupancy x [B, 1, 32, 32, 32] -> (mu, logvar), each [B, latent] (eval-mode BatchNorm)."""
    h = x
    for idx, kind, ci, co in VAE3D_ENCODER:
        name = f"{prefix}.encoder.{idx}"
        if kind == "conv":
            h = F.relu(F.conv3d(h, sd[f"{name}.weight"], sd[f"{name}.bias"], padding=1))
        elif kind == "res":
            h = _res_block3d_down(sd, name, h)
        elif kind == "down":
            h = F.relu(F.conv3d(h, sd[f"{name}.weight"], sd[f"{name}.bias"], stride=2, padding=1))
        else:                                  # Conv3d(k=4, p=0) + ReLU + Flatten
            h = F.relu(F.conv3d(h, sd[f"{name}.weight"], sd[f"{name}.bias"])).flatten(1)
        if taps is not None:
            taps[idx] = h
    return (F.linear(h, sd[f"{prefix}.fc_mu.weight"], sd[f"{prefix}.fc_mu.bias"]),
            F.linear(h, sd[f"{prefix}.fc_logvar.weight"], sd[f"{prefix}.fc_logvar.bias"]))
