"""CPU reference for SimplePointNetVAE.encode (the original project's encoder nn.Sequential and fc_mu / fc_logvar,
networks.py:1110-1156; PointNetLayer networks.py:16-49), restated with F.conv1d, eval-mode BatchNorm, amax and F.linear.
Imported by the point-encoder tests and by tools/bench_point_vae_encode.py; not a test module itself."""
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.pointdiff_oracle import _bn_eval, _conv

SD = Dict[str, torch.Tensor]

# encoder.0..3 = PointNetLayer(cin, cout): conv1 cin -> cout, conv2 and conv3 cout -> cout, each + BatchNorm1d + ReLU
POINT_ENCODER = [(0, 3, 64), (1, 64, 128), (2, 128, 256), (3, 256, 512)]


def point_vae_encoder_state_dict_spec(latent_dim: int = 256, hidden_dim: int = 512, prefix: str = "vae"):
    """(key, shape, kind) of the encoder half of SimplePointNetVAE's state_dict (encoder, fc_mu, fc_logvar)."""
    spec = []
    for idx, ci, co in POINT_ENCODER:
        co = hidden_dim if idx == 3 else co
        name = f"{prefix}.encoder.{idx}"
        for j, cj in ((1, ci), (2, co), (3, co)):
            spec += [(f"{name}.conv{j}.weight", (co, cj, 1), "w"), (f"{name}.conv{j}.bias", (co,), "b"),
                     (f"{name}.bn{j}.weight", (co,), "bn_w"), (f"{name}.bn{j}.bias", (co,), "bn_b"),
                     (f"{name}.bn{j}.running_mean", (co,), "bn_m"), (f"{name}.bn{j}.running_var", (co,), "bn_v"),
                     (f"{name}.bn{j}.num_batches_tracked", (), "nbt")]
    spec += [(f"{prefix}.encoder.6.weight", (hidden_dim // 2, hidden_dim), "w"), (f"{prefix}.encoder.6.bias", (hidden_dim // 2,), "b")]
    for head in ("fc_mu", "fc_logvar"):
        spec += [(f"{prefix}.{head}.weight", (latent_dim, hidden_dim // 2), "w"), (f"{prefix}.{head}.bias", (latent_dim,), "b")]
    return spec


def make_synthetic_point_vae_encoder_checkpoint(seed: int = 47, latent_dim: int = 256, hidden_dim: int = 512,
                                                prefix: str = "vae") -> SD:
    """Seeded encoder weights with variance-preserving scales (fan-in) and randomised BatchNorm statistics (scale, shift, mean
    and variance all away from the identity), so a BatchNorm folding bug cannot hide."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for key, shape, kind in point_vae_encoder_state_dict_spec(latent_dim, hidden_dim, prefix):
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


def point_vae_encode(sd: SD, x: torch.Tensor, prefix: str = "vae", taps: Optional[dict] = None):
    """SimplePointNetVAE.encode: clouds x [B, N, 3] -> (mu, logvar), each [B, latent] (eval-mode BatchNorm).

    Assumption (the reference body is not restated here): encode takes x in the [B, N, 3] layout of every cloud in this API and
    of `decode`'s output, and transposes it to channels-first [B, 3, N] for the Conv1d stack.  The reference-gated test in
    tests/test_point_vae_encoder_oracle.py pins it against the original module where that is available.

    taps (optional): 3 * i + j - 1 -> the activation after encoder.<i>.conv<j> (+ BatchNorm + ReLU) as [B, C, N];
    12 -> the pooled [B, 512]; 13 -> encoder.7's output [B, 256]."""
    h = x.transpose(1, 2)
    for idx, _, _ in POINT_ENCODER:
        for j in (1, 2, 3):                             # PointNetLayer.forward: conv -> BatchNorm1d -> ReLU, three times
            name = f"{prefix}.encoder.{idx}"
            h = F.relu(_bn_eval(sd, f"{name}.bn{j}", _conv(sd, f"{name}.conv{j}", h)))
            if taps is not None:
                taps[3 * idx + j - 1] = h
    g = h.amax(dim=2)                                   # AdaptiveMaxPool1d(1) + Flatten
    hid = F.relu(F.linear(g, sd[f"{prefix}.encoder.6.weight"], sd[f"{prefix}.encoder.6.bias"]))
    if taps is not None:
        taps[12], taps[13] = g, hid
    return (F.linear(hid, sd[f"{prefix}.fc_mu.weight"], sd[f"{prefix}.fc_mu.bias"]),
            F.linear(hid, sd[f"{prefix}.fc_logvar.weight"], sd[f"{prefix}.fc_logvar.bias"]))
