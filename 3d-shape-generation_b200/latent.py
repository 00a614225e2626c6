"""Latent-diffusion sampling (reference `LatentDiffusion`, diffusion.py:361-707) on the B200 path:
`SimpleLatentUNetPointNet` (networks.py:962-1106) as the latent denoiser and
`SimplePointNetVAE.decode` (networks.py:1144-1154, 1219-1231) as the fused 2048-point decoder.  `SimplePointNetVAE.encode` /
`forward` run on the per-point tcgen05 GEMMs with a fused max-pool (`pcd_point_encode`, `PointEncoderEngine`).

Module trees are parameter containers with the reference's exact state_dict keys; forward /
decode / the loops run in the CUDA library (`pcd_latent_*`).  The reference's default voxel VAE
(`VAE3DLarge`, is_voxel_based=True) decodes through `pcd_vae3d_decode` and the GPU voxel -> points
compaction (voxel.py); any other VAE module is supported by running the latent loop in the
library and then calling the user's own `vae.decode`."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.nn as nn

from . import _lib
from .diffusion import build_ddim3_table, build_ddim_table, build_ddpm_table
from .networks import PointNetLayer
from . import voxel as _voxel


class _HParams(dict):
    __getattr__ = dict.__getitem__


class SimpleLatentUNetPointNet(nn.Module):
    """Parameter container mirroring reference networks.py:962-1049."""

    def __init__(self, latent_dim, dim=512, time_dim=256, dropout_rate=0.1):
        super().__init__()
        if (latent_dim, dim, time_dim) != (256, 512, 256):
            raise NotImplementedError("the B200 latent kernels are specialised for latent_dim=256, dim=512, time_dim=256 "
                                      "(the reference defaults)")
        self.time_dim = time_dim

        def blk(cin, cout, drop=False):
            layers = [nn.Linear(cin, cout), nn.GroupNorm(8, cout), nn.ReLU()]
            if drop:
                layers.append(nn.Dropout(dropout_rate))
            return nn.Sequential(*layers)
        self.time_mlp = nn.Sequential(nn.Linear(time_dim, time_dim), nn.SiLU(), nn.Linear(time_dim, time_dim))
        self.enc1 = blk(latent_dim + time_dim, dim // 4)
        self.enc2 = blk(dim // 4, dim // 2)
        self.enc3 = blk(dim // 2, dim)
        self.enc4 = blk(dim, dim * 2)
        self.global_feat = nn.Sequential(nn.Linear(dim * 2, dim * 4), nn.GroupNorm(8, dim * 4), nn.ReLU(),
                                         nn.Linear(dim * 4, dim * 8), nn.GroupNorm(8, dim * 8), nn.ReLU())
        self.dec4 = blk(dim * 8 + dim * 2, dim * 2)
        self.dec3 = blk(dim * 2 + dim, dim)
        self.dec2 = blk(dim + dim // 2, dim // 2)
        self.dec1 = blk(dim // 2 + dim // 4, dim // 4, drop=True)
        self.output = nn.Sequential(nn.Linear(dim // 4, dim // 4), nn.ReLU(), nn.Linear(dim // 4, latent_dim))
        self.refine1 = nn.Linear(dim // 4, dim // 4)
        self.refine2 = nn.Linear(dim // 2, dim // 2)
        self.refine3 = nn.Linear(dim, dim)
        self.refine4 = nn.Linear(dim * 2, dim * 2)


class SimplePointNetVAE(nn.Module):
    """Parameter container mirroring reference networks.py:1110-1156 (same state_dict keys, so `load_state_dict(strict=True)`
    works in both directions).  `encode(x)`, `decode(z)` and `forward(x)` run in the library (inference: eval-mode BatchNorm,
    no autograd); training is out of scope.  `precision` selects the encoder's tensor-core precision ('bf16x3', 'f16mix',
    'bf16' or 'f16'); it is not a hyper-parameter of the reference and does not affect `decode`."""

    def __init__(self, num_points, latent_dim=256, hidden_dim=512, lr=1e-4, beta=1e-1, dropout_rate=0.1,
                 chamfer_lambda=1, voxel_lambda=1, focal_alpha=0.25, focal_gamma=2.00, *, precision: str = "bf16x3"):
        super().__init__()
        self.precision = precision
        self._enc_engine = None
        self._enc_engine_key = None
        self.hparams = _HParams(num_points=num_points, latent_dim=latent_dim, hidden_dim=hidden_dim, lr=lr, beta=beta,
                                dropout_rate=dropout_rate, chamfer_lambda=chamfer_lambda, voxel_lambda=voxel_lambda,
                                focal_alpha=focal_alpha, focal_gamma=focal_gamma)
        self.encoder = nn.Sequential(PointNetLayer(3, 64), PointNetLayer(64, 128), PointNetLayer(128, 256),
                                     PointNetLayer(256, hidden_dim), nn.AdaptiveMaxPool1d(1), nn.Flatten(),
                                     nn.Linear(hidden_dim, hidden_dim // 2), nn.ReLU())
        self.fc_mu = nn.Linear(hidden_dim // 2, latent_dim)
        self.fc_logvar = nn.Linear(hidden_dim // 2, latent_dim)
        self.decoder = nn.Sequential(nn.Linear(latent_dim, hidden_dim // 2), nn.ReLU(), nn.Linear(hidden_dim // 2, hidden_dim),
                                     nn.ReLU(), nn.Linear(hidden_dim, num_points * 3), nn.ReLU(), nn.Dropout(dropout_rate))
        self.output_layer = nn.Linear(num_points * 3, num_points * 3)

    def decode(self, z):
        """Reference networks.py:1219-1231: latent [B, 256] -> points [B, num_points, 3], on the library's fused decoder."""
        return _own_decoder_engine(self, self.output_layer.out_features // 3).decode(z)

    def encoder_engine(self) -> "PointEncoderEngine":
        """The encoder handle, rebuilt when the parameters or BatchNorm statistics change."""
        dev = self.fc_mu.weight.device
        if dev.type != "cuda":
            raise _lib.PcdError("SimplePointNetVAE is on %s: the B200 point encoder has no CPU fallback; call .to('cuda')" % dev)
        key = (dev, self.precision, tuple(p._version for p in self.parameters()), tuple(b._version for b in self.buffers()))
        if self._enc_engine is None or key != self._enc_engine_key:
            if self._enc_engine is not None:
                self._enc_engine.close()
            self._enc_engine = PointEncoderEngine(self.state_dict(), dev, self.precision)
            self._enc_engine_key = key
        return self._enc_engine

    @torch.no_grad()
    def encode(self, x: torch.Tensor):
        """Reference SimplePointNetVAE.encode: clouds x [B, N, 3] (any N >= 1) -> (mu, logvar), each [B, latent_dim].
        BatchNorm runs in eval mode (running statistics) whatever the module's mode.  A cloud with a NaN or infinite coordinate
        gets NaN in every entry, as in the reference."""
        return self.encoder_engine().encode(x)

    @staticmethod
    def reparameterize(mu: torch.Tensor, logvar: torch.Tensor) -> torch.Tensor:
        """mu + eps * std with std = exp(0.5 * logvar) and eps = randn_like(std) (the reference's draw)."""
        std = torch.exp(0.5 * logvar)
        return mu + torch.randn_like(std) * std

    @torch.no_grad()
    def forward(self, x: torch.Tensor):
        """Reference SimplePointNetVAE.forward: (decode(reparameterize(mu, logvar)), mu, logvar)."""
        mu, logvar = self.encode(x)
        return self.decode(self.reparameterize(mu, logvar)), mu, logvar

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location="cpu", **overrides):
        """Lightning `.ckpt` dict parsed without Lightning (reference call site train_point_ldm.py:43,190); `precision=` may be
        passed as an override."""
        return _vae_from_checkpoint(cls, checkpoint_path, map_location, overrides, strict=True)


class FoldingLayer(nn.Module):
    """Parameter container mirroring reference networks.py:386-412 (Conv1d, ReLU, Conv1d)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.layer = nn.Sequential(nn.Conv1d(in_channels, out_channels, 1), nn.ReLU(), nn.Conv1d(out_channels, out_channels, 1))


class FoldingDecoder(nn.Module):
    """Parameter container mirroring reference networks.py:1449-1482; `grid` is a plain attribute there too."""

    def __init__(self, latent_dim, num_points):
        super().__init__()
        if latent_dim != 256:
            raise NotImplementedError("the B200 folding kernels are specialised for latent_dim = 256 (the reference default)")
        self.num_points, self.latent_dim = num_points, latent_dim
        self.grid = folding_grid()
        self.fold1 = nn.Sequential(FoldingLayer(latent_dim + 2, 512), FoldingLayer(512, 512), FoldingLayer(512, 3))
        self.fold2 = nn.Sequential(FoldingLayer(latent_dim + 3, 512), FoldingLayer(512, 512), FoldingLayer(512, 3))
        self.upsample = nn.Linear(1024, num_points)


def folding_grid() -> torch.Tensor:
    """Reference networks.py:1463-1467: 32 x 32 grid on [-1, 1]^2 ('ij' meshgrid) as [2, 1024]."""
    r = torch.linspace(-1, 1, 32)
    xc, yc = torch.meshgrid(r, r, indexing="ij")
    return torch.stack([xc, yc], dim=-1).view(-1, 2).transpose(0, 1).contiguous()


class PointNetVAE(nn.Module):
    """Decoder half of reference networks.py:1512-1589 (`decode` = FoldingDecoder).  The PointNet++ encoder
    (set abstraction + FPS, networks.py:182-366, 1414-1447) is off the sampling path (SURVEY C12/C13) and is not
    mirrored: load a reference checkpoint with `load_state_dict(sd, strict=False)`."""

    def __init__(self, num_points=2048, latent_dim=256, lr=1e-4, beta=1e-1):
        super().__init__()
        self.hparams = _HParams(num_points=num_points, latent_dim=latent_dim, lr=lr, beta=beta)
        self.decoder = FoldingDecoder(latent_dim, num_points)

    def decode(self, z):
        """Reference networks.py:1579-1589 (`FoldingDecoder.forward`, :1484-1509) on the library's folding kernels."""
        return _own_decoder_engine(self, self.decoder.upsample.out_features).decode(z)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location="cpu", **overrides):
        """Lightning `.ckpt` dict parsed without Lightning; the PointNet++ encoder keys are ignored (off the sampling path)."""
        return _vae_from_checkpoint(cls, checkpoint_path, map_location, overrides, strict=False)


def _vae_from_checkpoint(cls, checkpoint_path, map_location, overrides, strict):
    import inspect
    ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
    hp = dict(ckpt.get("hyper_parameters", {}))
    hp.update(overrides)
    allowed = set(inspect.signature(cls.__init__).parameters) - {"self"}
    vae = cls(**{k: v for k, v in hp.items() if k in allowed})
    vae.load_state_dict(ckpt["state_dict"], strict=strict)
    return vae


def _own_decoder_engine(vae, num_points):
    """Decoder-only library handle of a standalone point VAE (built from its own state_dict, rebuilt when the weights change)."""
    dev = next(vae.parameters()).device
    if dev.type != "cuda":
        raise _lib.PcdError("VAE is on %s: the B200 decoder has no CPU fallback; call .to('cuda')" % dev)
    key = (dev, tuple(p._version for p in vae.parameters()))
    if getattr(vae, "_dec_engine", None) is None or vae._dec_key != key:
        if getattr(vae, "_dec_engine", None) is not None:
            vae._dec_engine.close()
        sd = {"vae." + k: v for k, v in vae.state_dict().items()}
        object.__setattr__(vae, "_dec_engine", LatentEngine(sd, num_points, dev))
        object.__setattr__(vae, "_dec_key", key)
    return vae._dec_engine


def _is_folding_vae(vae) -> bool:
    try:
        d = vae.decoder
        return (isinstance(d.fold1, nn.Sequential) and isinstance(d.fold2, nn.Sequential) and isinstance(d.upsample, nn.Linear)
                and d.upsample.in_features == 1024 and d.fold1[0].layer[0].in_channels == 258
                and d.fold2[0].layer[0].in_channels == 259)
    except (AttributeError, IndexError, TypeError):
        return False


def _is_simple_point_vae(vae) -> bool:
    try:
        return (isinstance(vae.decoder, nn.Sequential) and isinstance(vae.decoder[0], nn.Linear)
                and isinstance(vae.output_layer, nn.Linear) and vae.decoder[0].in_features == 256
                and vae.decoder[0].out_features == 256 and vae.decoder[2].out_features == 512
                and vae.output_layer.in_features == vae.output_layer.out_features)
    except (AttributeError, IndexError, TypeError):
        return False


class LatentEngine:
    """Owns the opaque pcd_latent handle."""

    def __init__(self, state_dict, num_points: int, device: torch.device):
        if device.type != "cuda":
            raise _lib.PcdError("the B200 latent path needs a CUDA device; there is no CPU fallback")
        items = [(k, v) for k, v in state_dict.items() if k.startswith("model.") or k.startswith("vae.decoder.")
                 or k.startswith("vae.output_layer.")]
        if any(k.startswith("vae.decoder.fold1.") for k, _ in items):
            items.append(("vae.decoder.grid", folding_grid()))     # not a parameter in the reference (networks.py:1467)
        keep, arr = [], (_lib._NamedTensor * len(items))()
        for i, (k, v) in enumerate(items):
            t = v.detach().to(device="cpu", dtype=torch.float32).contiguous()
            keep.append(t)
            arr[i].name, arr[i].data, arr[i].dtype, arr[i].ndim = k.encode(), t.data_ptr(), 0, t.dim()
            for d in range(t.dim()):
                arr[i].shape[d] = t.shape[d]
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.lib().pcd_latent_create(arr, len(items), num_points, idx, C.byref(h)))
        self._h, self.device, self.num_points = h, device, num_points

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pcd_latent_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def forward(self, z, t):
        _lib._require_cuda(z, "z")
        z = z.to(torch.float32).contiguous()
        t = t.to(device=z.device, dtype=torch.float32).contiguous()
        eps = torch.empty_like(z)
        _lib.check(_lib.lib().pcd_latent_forward(self._h, z.data_ptr(), t.data_ptr(), eps.data_ptr(), z.shape[0],
                                                 _lib.stream_ptr(z.device)))
        return eps

    def sample_(self, sched, z, noise=None, seed=0, sample_offset=0):
        _lib._require_cuda(z, "z")
        assert z.dtype == torch.float32 and z.is_contiguous() and z.shape[1] == 256
        sched = sched.to(device="cpu", dtype=torch.float32).contiguous()
        S, B = sched.shape[0], z.shape[0]
        rows = 1 if sched.dim() == 2 else sched.shape[1]      # [S, 8] shared by the batch, or [S, B, 8] one row per sample
        assert rows in (1, B)
        nptr = None
        if noise is not None:
            _lib._require_cuda(noise, "noise")
            assert noise.dtype == torch.float32 and noise.is_contiguous() and tuple(noise.shape) == (S - 1, B, 256)
            nptr = noise.data_ptr()
        _lib.check(_lib.lib().pcd_latent_sample_rows(self._h, sched.data_ptr(), S, rows, z.data_ptr(), nptr, seed, sample_offset, B,
                                                     _lib.stream_ptr(z.device)))
        return z

    def decode(self, z):
        _lib._require_cuda(z, "z")
        z = z.to(torch.float32).contiguous()
        out = torch.empty(z.shape[0], self.num_points, 3, device=z.device, dtype=torch.float32)
        _lib.check(_lib.lib().pcd_vae_decode(self._h, z.data_ptr(), out.data_ptr(), z.shape[0], _lib.stream_ptr(z.device)))
        return out


class PointEncoderEngine:
    """Owns the opaque pcd_point_encoder handle built from the encoder half of a SimplePointNetVAE state_dict (`encoder.*`,
    `fc_mu.*`, `fc_logvar.*`, with or without the `vae.` prefix, so the reference's own module encodes from its `state_dict()`).
    Only hidden_dim = 512 and latent_dim = 256 (the reference defaults) are supported."""

    def __init__(self, state_dict, device: torch.device, precision: str = "bf16x3"):
        if device.type != "cuda":
            raise _lib.PcdError("the B200 point encoder needs a CUDA device; there is no CPU fallback")
        if precision not in ("bf16", "bf16x3", "f16", "f16mix"):
            raise ValueError("precision must be 'bf16', 'bf16x3', 'f16' or 'f16mix' (fp16 hi+lo planes)")
        items = []
        for k, v in state_dict.items():
            k = k[4:] if k.startswith("vae.") else k
            if k.startswith(("encoder.", "fc_mu.", "fc_logvar.")) and not k.endswith("num_batches_tracked"):
                items.append(("vae." + k, v))
        keep, arr = [], (_lib._NamedTensor * max(len(items), 1))()
        for i, (k, v) in enumerate(items):
            t = v.detach().to(device="cpu", dtype=torch.float32).contiguous()
            keep.append(t)
            arr[i].name, arr[i].data, arr[i].dtype, arr[i].ndim = k.encode(), t.data_ptr(), 0, min(t.dim(), 4)
            for d in range(min(t.dim(), 4)):
                arr[i].shape[d] = t.shape[d]
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.lib().pcd_point_encoder_create(arr, len(items), _lib.PRECISION[precision], idx, C.byref(h)))
        self._h, self.device, self.precision = h, device, precision
        self.latent_dim = 256

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pcd_point_encoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _clouds(x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3 or x.shape[2] != 3:
            raise ValueError("x must be [B, N, 3], got %s" % (tuple(x.shape),))
        _lib._require_cuda(x, "x")
        return x.to(torch.float32).contiguous()

    def encode(self, x: torch.Tensor):
        """x [B, N, 3] -> (mu, logvar), each [B, 256] fp32 on x's device."""
        x = self._clouds(x)
        B, N, _ = x.shape
        mu = torch.empty(B, self.latent_dim, device=x.device, dtype=torch.float32)
        logvar = torch.empty_like(mu)
        _lib.check(_lib.lib().pcd_point_encode(self._h, x.data_ptr(), mu.data_ptr(), logvar.data_ptr(), B, N, _lib.stream_ptr(x.device)))
        return mu, logvar

    def tap(self, x: torch.Tensor, index: int) -> torch.Tensor:
        """Parity hook on the host: index 0..11 = the activation after encoder.<index // 3>.conv<index % 3 + 1> (+ BatchNorm +
        ReLU) as [B, C, N] (the reference's channels-first layout); 12 = the pooled [B, 512]; 13 = encoder.7's output [B, 256]."""
        x = self._clouds(x)
        B, N, _ = x.shape
        if index == 12:
            out = torch.empty(B, 512, dtype=torch.float32)
        elif index == 13:
            out = torch.empty(B, 256, dtype=torch.float32)
        else:
            out = torch.empty(B, N, (64, 128, 256, 512)[min(max(index, 0), 11) // 3], dtype=torch.float32)
        _lib.check(_lib.lib().pcd_point_encoder_tap(self._h, x.data_ptr(), B, N, index, out.data_ptr(), out.numel(),
                                                    _lib.stream_ptr(x.device)))
        return out if index >= 12 else out.transpose(1, 2).contiguous()

    def profile(self, x: torch.Tensor):
        """[(name, ms, useful FLOPs)] of one eager encode, CUDA-event timed per launch group."""
        x = self._clouds(x)
        B, N, _ = x.shape
        cap, stride = 32, 48
        ms, fl = (C.c_float * cap)(), (C.c_double * cap)()
        names, n = C.create_string_buffer(cap * stride), C.c_int32(0)
        mu = torch.empty(B, self.latent_dim, device=x.device, dtype=torch.float32)
        logvar = torch.empty_like(mu)
        _lib.check(_lib.lib().pcd_point_encoder_profile(self._h, x.data_ptr(), mu.data_ptr(), logvar.data_ptr(), B, N, ms, fl, names,
                                                        stride, cap, C.byref(n), _lib.stream_ptr(x.device)))
        return [(names.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode(), float(ms[i]), float(fl[i])) for i in range(n.value)]


def latent_philox_normal(seed, sample_offset, step, B, D, device):
    out = torch.empty(B, D, device=device, dtype=torch.float32)
    _lib.check(_lib.lib().pcd_latent_philox_normal(seed, sample_offset, step, out.data_ptr(), B, D, _lib.stream_ptr(out.device)))
    return out


def voxel_tensor_to_point_clouds(voxel_grid: torch.Tensor, threshold: float = 0.5):
    """Reference utils.py:511-539 (ragged output) -- GPU stream compaction, see voxel.py."""
    return _voxel.voxel_tensor_to_point_clouds(voxel_grid, threshold)


class LatentDiffusion(nn.Module):
    """Reference diffusion.py:361-707 sampling API: `sample(num_samples, num_steps=1000, threshold=0.4)`
    (DDIM), `sample2` (DDPM), `sample3(num_samples, z=None, start_t=None, num_steps=1000, threshold=0.4)`."""

    def __init__(self, vae, latent_dim=256, dim=512, time_dim=256, lr=1e-4, noise_schedule="cosine", is_voxel_based=True):
        super().__init__()
        self.hparams = _HParams(latent_dim=latent_dim, dim=dim, time_dim=time_dim, lr=lr, noise_schedule=noise_schedule,
                                is_voxel_based=is_voxel_based)
        self.vae = vae
        for p in self.vae.parameters():
            p.requires_grad = False
        self.model = SimpleLatentUNetPointNet(latent_dim, dim, time_dim)
        self.lr, self.noise_schedule = lr, noise_schedule
        self.cosine_min_signal_rate, self.cosine_max_signal_rate = 0.02, 0.95
        self.linear_min_rate, self.linear_max_rate = 0.0001, 0.02
        self.diffusion_schedule = (self.offset_cosine_diffusion_schedule if noise_schedule == "cosine"
                                   else self.linear_diffusion_schedule)
        for m in self.model.modules():   # reference :391-408 (VAE is skipped)
            if isinstance(m, nn.Linear):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                nn.init.constant_(m.bias, 0)
        self._engine = None
        self._engine_key = None

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location="cpu", *, vae, strict=True, **overrides):
        """Lightning-style checkpoint of the reference's LatentDiffusion (call sites train_point_ldm.py:106,222:
        `LatentDiffusion.load_from_checkpoint(path, vae=vae, is_voxel_based=...)`), parsed without Lightning.  `vae` is passed by
        the caller because the reference excludes it from the saved hyper-parameters (`save_hyperparameters(ignore=['vae'])`,
        diffusion.py:375); the checkpoint's `state_dict` still carries the frozen `vae.*` tensors next to `model.*` and they are
        loaded into it.  Keyword overrides (e.g. is_voxel_based=) win over the stored hyper-parameters, as in Lightning."""
        ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
        hp = dict(ckpt.get("hyper_parameters", {}))
        hp.update(overrides)
        allowed = ("latent_dim", "dim", "time_dim", "lr", "noise_schedule", "is_voxel_based")
        model = cls(vae, **{k: v for k, v in hp.items() if k in allowed})
        sd = ckpt["state_dict"]
        if not strict or not any(k.startswith("vae.") for k in sd):
            res = model.load_state_dict(sd, strict=False)
            bad = [k for k in res.missing_keys if k.startswith("model.")] + list(res.unexpected_keys if strict else [])
            if bad:
                raise RuntimeError(f"LatentDiffusion checkpoint does not match: {bad[:5]}")
        else:
            # a decoder-only VAE container (PointNetVAE here) does not mirror the encoder: its keys may be absent from the module
            own = set(model.state_dict())
            extra = [k for k in sd if k not in own and not k.startswith("vae.")]
            if extra:
                raise RuntimeError(f"unexpected keys in LatentDiffusion checkpoint: {extra[:5]}")
            res = model.load_state_dict({k: v for k, v in sd.items() if k in own}, strict=False)
            missing = [k for k in res.missing_keys if k.startswith("model.")]
            if missing:
                raise RuntimeError(f"missing keys in LatentDiffusion checkpoint: {missing[:5]}")
        return model

    @property
    def device(self):
        return next(self.model.parameters()).device

    def add_noise(self, z_0, t):
        """Reference diffusion.py:490-504."""
        noise = torch.randn_like(z_0)
        noise_rates, signal_rates = self.diffusion_schedule(t)
        z_t = signal_rates.view(-1, 1) * z_0 + noise_rates.view(-1, 1) * noise
        return z_t, noise, noise_rates, signal_rates

    def offset_cosine_diffusion_schedule(self, diffusion_times):
        """Reference diffusion.py:539-556 (same as the point model's)."""
        a0 = torch.acos(torch.tensor(self.cosine_max_signal_rate, device=diffusion_times.device))
        a1 = torch.acos(torch.tensor(self.cosine_min_signal_rate, device=diffusion_times.device))
        ang = a0 + diffusion_times * (a1 - a0)
        return torch.sin(ang), torch.cos(ang)

    def linear_diffusion_schedule(self, diffusion_times):
        betas = self.linear_min_rate + diffusion_times.clone() * (self.linear_max_rate - self.linear_min_rate)
        alpha_bars = torch.cumprod(1 - betas, dim=0)
        return 1 - alpha_bars, alpha_bars

    def remove_noise(self, z_t, predicted_noise, noise_rates, signal_rates):
        """Reference diffusion.py:506-520."""
        return (z_t - noise_rates.view(-1, 1) * predicted_noise) / signal_rates.view(-1, 1)

    def engine(self) -> LatentEngine:
        dev = self.device
        if dev.type != "cuda":
            raise _lib.PcdError("model is on %s: the B200 latent path has no CPU fallback; call .to('cuda')" % dev)
        fused = self._fused_decoder()
        key = (dev, fused, tuple(p._version for p in self.parameters()))
        if self._engine is None or key != self._engine_key:
            if self._engine is not None:
                self._engine.close()
            sd = {k: v for k, v in self.state_dict().items() if k.startswith("model.") or fused}
            npts = 0
            if fused:
                npts = self.vae.decoder.upsample.out_features if _is_folding_vae(self.vae) else self.vae.output_layer.out_features // 3
            self._engine = LatentEngine(sd, npts, dev)
            self._engine_key = key
        return self._engine

    def _fused_decoder(self) -> bool:
        """True when the VAE's decoder runs in the library: SimplePointNetVAE (networks.py:1144-1154) or
        PointNetVAE's FoldingDecoder (networks.py:1449-1509), both point based."""
        return (_is_simple_point_vae(self.vae) or _is_folding_vae(self.vae)) and not self.hparams.is_voxel_based

    def _table_batch(self, batch: int) -> int:
        # the cosine schedule is elementwise in t: one row per step serves the whole batch; the reference's 'linear' schedule
        # cumprods over the BATCH axis (diffusion.py:553-569), so every sample of a batch gets its own rates: one row per sample
        return 1 if self.noise_schedule == "cosine" else batch

    def _decode(self, z0, threshold):
        eng = self.engine()
        if self._fused_decoder():
            return eng.decode(z0)
        if self.hparams.is_voxel_based and _voxel.is_vae3d_large(self.vae):
            # the reference's default configuration: VAE3DLarge.decode + voxel_tensor_to_point_clouds (diffusion.py:609-612)
            x0 = self._vae3d_engine().decode(z0)
        else:
            x0 = self.vae.decode(z0)        # any other user-supplied decoder module
        if self.hparams.is_voxel_based:
            return voxel_tensor_to_point_clouds(x0, threshold=threshold)
        return x0

    def _vae3d_engine(self):
        """The voxel decoder handle: the VAE's own engine when it is our container, else one built from the module's state_dict
        (e.g. the reference's own VAE3DLarge instance)."""
        if isinstance(self.vae, _voxel.VAE3DLarge):
            return self.vae.engine()
        key = (self.device, tuple(p._version for p in self.vae.parameters()), tuple(b._version for b in self.vae.buffers()))
        if getattr(self, "_v3d", None) is None or self._v3d_key != key:
            if getattr(self, "_v3d", None) is not None:
                self._v3d.close()
            self._v3d = _voxel.Vae3dEngine(self.vae.state_dict(), self.device, getattr(self.vae, "precision", _voxel.DEFAULT_PRECISION))
            self._v3d_key = key
        return self._v3d

    def _start(self, num_samples, z_T):
        if z_T is None:
            return torch.randn(num_samples, self.hparams.latent_dim, device=self.device)
        return z_T.to(device=self.device, dtype=torch.float32).clone().contiguous()

    @torch.no_grad()
    def sample(self, num_samples, num_steps=1000, threshold=0.4, *, z_T: Optional[torch.Tensor] = None, sample_offset=0,
               return_latent=False):
        """DDIM in latent space (reference diffusion.py:619-653).  For a point-based VAE the reference
        crashes (`point_clouds` unassigned, :650-653); the defined behaviour here mirrors sample2's else
        branch (:611-614): return vae.decode(z_0)."""
        self.eval()
        z = self.engine().sample_(build_ddim_table(self.diffusion_schedule, num_steps, self._table_batch(num_samples)),
                                  self._start(num_samples, z_T), sample_offset=sample_offset)
        return z if return_latent else self._decode(z, threshold)

    @torch.no_grad()
    def sample2(self, num_samples, num_steps=1000, threshold=0.4, *, z_T=None, noise=None, seed=0, sample_offset=0,
                return_latent=False):
        """Pure DDPM in latent space (reference diffusion.py:575-616)."""
        self.eval()
        if noise is not None:
            noise = noise.to(device=self.device, dtype=torch.float32).contiguous()
        z = self.engine().sample_(build_ddpm_table(self.diffusion_schedule, num_steps, self._table_batch(num_samples)), self._start(num_samples, z_T), noise=noise, seed=seed,
                                  sample_offset=sample_offset)
        return z if return_latent else self._decode(z, threshold)

    @torch.no_grad()
    def sample3(self, num_samples, z=None, start_t=None, num_steps=1000, threshold=0.4, *, return_latent=False):
        """DDIM from a given latent / start time (reference diffusion.py:655-707)."""
        self.eval()
        start = 1.0 if (z is None or start_t is None) else float(start_t.reshape(-1)[0])
        z = self.engine().sample_(build_ddim3_table(self.diffusion_schedule, start, num_steps), self._start(num_samples, z))
        return z if return_latent else self._decode(z, threshold)
