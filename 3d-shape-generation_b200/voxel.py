"""Voxel VAE encoding and decoding on the B200 path (SURVEY 8(f) rank 4): the reference's DEFAULT latent-diffusion configuration
(`LatentDiffusion(vae=VAE3DLarge(...), is_voxel_based=True)`, diffusion.py:362, train_point_ldm.py:161-222).

* `VAE3DLarge` / `ResidualBlock3D` are parameter containers with the reference's exact `state_dict` keys
  (networks.py:471-505, 2208-2264); `decode` (networks.py:2327-2339) runs in the CUDA library (`pcd_vae3d_decode`:
  implicit-GEMM 3-D convolutions on the tcgen05 kernel), and so does `encode` (`pcd_vae3d_encode`: the same kernels plus
  stride-2 convolutions, learned 1x1 shortcuts, a CUDA-core first layer and fp32 heads).  Training is out of scope.
* `voxel_tensor_to_point_clouds` (utils.py:511-539) is an ordered stream compaction on the GPU
  (`pcd_voxel_count` + `pcd_voxel_points`), bit-identical to the reference's `torch.where` path.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib

DEFAULT_PRECISION = "bf16x3"


class _HParams(dict):
    __getattr__ = dict.__getitem__


class ResidualBlock3D(nn.Module):
    """Parameter container mirroring reference networks.py:471-486."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv1 = nn.Conv3d(in_channels, out_channels, kernel_size=3, padding=1)
        self.bn1 = nn.BatchNorm3d(out_channels)
        self.conv2 = nn.Conv3d(out_channels, out_channels, kernel_size=3, padding=1)
        self.bn2 = nn.BatchNorm3d(out_channels)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = nn.Conv3d(in_channels, out_channels, kernel_size=1) if in_channels != out_channels else None


class VAE3DLarge(nn.Module):
    """Parameter container mirroring reference networks.py:2208-2264 (same constructor signature, same state_dict keys, so
    `load_state_dict(strict=True)` works in both directions).  `encode(x)`, `decode(z)` and
    `forward(x)` run on the B200 kernels (inference: eval-mode BatchNorm, no autograd); training is out of scope."""

    def __init__(self, input_shape=(32, 32, 32), latent_dim=256, lr=1e-4, kl_warmup_epochs=10, kl_warmup_max_beta=0.1,
                 kl_annealing_epochs=100, *, precision: str = DEFAULT_PRECISION):
        super().__init__()
        if tuple(input_shape) != (32, 32, 32):
            raise NotImplementedError("the B200 voxel decoder is specialised for 32^3 grids (the reference default)")
        self.hparams = _HParams(input_shape=input_shape, latent_dim=latent_dim, lr=lr, kl_warmup_epochs=kl_warmup_epochs,
                                kl_warmup_max_beta=kl_warmup_max_beta, kl_annealing_epochs=kl_annealing_epochs)
        self.precision = precision
        self.encoder = nn.Sequential(
            nn.Conv3d(1, 32, kernel_size=3, stride=1, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(32, 64),
            nn.Conv3d(64, 64, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(64, 128),
            nn.Conv3d(128, 128, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(128, 256),
            nn.Conv3d(256, 256, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(256, 512),
            nn.Conv3d(512, 512, kernel_size=4, stride=1, padding=0), nn.ReLU(inplace=True), nn.Flatten())
        self.fc_mu = nn.Linear(512, latent_dim)
        self.fc_logvar = nn.Linear(512, latent_dim)
        self.decoder_input = nn.Linear(latent_dim, 512 * 4 * 4 * 4)
        self.decoder = nn.Sequential(
            nn.ConvTranspose3d(512, 256, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(256, 256),
            nn.ConvTranspose3d(256, 128, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(128, 128),
            nn.ConvTranspose3d(128, 64, kernel_size=4, stride=2, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(64, 64),
            nn.Conv3d(64, 32, kernel_size=3, padding=1), nn.ReLU(inplace=True), ResidualBlock3D(32, 32),
            nn.Conv3d(32, 1, kernel_size=3, padding=1), nn.Sigmoid())
        self._engine = None
        self._engine_key = None
        self._enc_engine = None
        self._enc_engine_key = None

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location="cpu", **overrides):
        """Lightning-style `.ckpt` dict parsed without Lightning (reference call sites test_point_ldm.py:157,
        train_point_ldm.py:43,190)."""
        ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
        hp = dict(ckpt.get("hyper_parameters", {}))
        hp.update(overrides)
        allowed = ("input_shape", "latent_dim", "lr", "kl_warmup_epochs", "kl_warmup_max_beta", "kl_annealing_epochs", "precision")
        vae = cls(**{k: v for k, v in hp.items() if k in allowed})
        vae.load_state_dict(ckpt["state_dict"], strict=True)
        return vae

    @property
    def device(self):
        return self.decoder_input.weight.device

    def _key(self, what):
        dev = self.device
        if dev.type != "cuda":
            raise _lib.PcdError("VAE3DLarge is on %s: the B200 voxel %s has no CPU fallback; call .to('cuda')" % (dev, what))
        return (dev, self.precision, tuple(p._version for p in self.parameters()), tuple(b._version for b in self.buffers()))

    def engine(self) -> "Vae3dEngine":
        dev = self.device
        key = self._key("decoder")
        if self._engine is None or key != self._engine_key:
            if self._engine is not None:
                self._engine.close()
            self._engine = Vae3dEngine(self.state_dict(), dev, self.precision)
            self._engine_key = key
        return self._engine

    @torch.no_grad()
    def decode(self, z: torch.Tensor) -> torch.Tensor:
        """Reference networks.py:2327-2339: z [B, latent] -> voxel probabilities [B, 1, 32, 32, 32] (eval-mode BatchNorm)."""
        return self.engine().decode(z)

    def encoder_engine(self) -> "Vae3dEncoderEngine":
        key = self._key("encoder")
        if self._enc_engine is None or key != self._enc_engine_key:
            if self._enc_engine is not None:
                self._enc_engine.close()
            self._enc_engine = Vae3dEncoderEngine(self.state_dict(), self.device, self.precision)
            self._enc_engine_key = key
        return self._enc_engine

    @torch.no_grad()
    def encode(self, x: torch.Tensor):
        """Reference VAE3DLarge.encode: occupancy x [B, 1, 32, 32, 32] -> (mu, logvar), each [B, latent] (eval-mode BatchNorm)."""
        return self.encoder_engine().encode(x)

    @staticmethod
    def reparameterize(mu: torch.Tensor, logvar: torch.Tensor) -> torch.Tensor:
        """mu + eps * std with std = exp(0.5 * logvar) and eps = randn_like(std) (the reference's draw)."""
        std = torch.exp(0.5 * logvar)
        return mu + torch.randn_like(std) * std

    @torch.no_grad()
    def forward(self, x: torch.Tensor):
        """Reference VAE3DLarge.forward: (decode(reparameterize(mu, logvar)), mu, logvar)."""
        mu, logvar = self.encode(x)
        return self.decode(self.reparameterize(mu, logvar)), mu, logvar


def is_vae3d_large(vae) -> bool:
    """True for a module with VAE3DLarge's decoder layout (ours or the reference's own class)."""
    try:
        d = vae.decoder
        return (isinstance(vae.decoder_input, nn.Linear) and vae.decoder_input.out_features == 512 * 64
                and isinstance(d[0], nn.ConvTranspose3d) and d[0].in_channels == 512 and isinstance(d[12], nn.Conv3d)
                and d[12].out_channels == 1 and len(d) == 14)
    except (AttributeError, IndexError, TypeError):
        return False


class Vae3dEngine:
    """Owns the opaque pcd_vae3d handle built from the decoder half of a VAE3DLarge state_dict (keys with or without the
    `vae.` prefix LatentDiffusion.state_dict() adds)."""

    def __init__(self, state_dict, device: torch.device, precision: str = DEFAULT_PRECISION):
        if device.type != "cuda":
            raise _lib.PcdError("the B200 voxel decoder needs a CUDA device; there is no CPU fallback")
        if precision not in ("bf16", "bf16x3", "f16", "f16mix"):
            raise ValueError("precision must be 'bf16', 'bf16x3', 'f16' or 'f16mix' (fp16 hi+lo planes)")
        items = []
        for k, v in state_dict.items():
            k = k[4:] if k.startswith("vae.") else k
            if (k.startswith("decoder_input.") or k.startswith("decoder.")) and not k.endswith("num_batches_tracked"):
                items.append(("vae." + k, v))
        keep, arr = [], (_lib._NamedTensor * len(items))()
        for i, (k, v) in enumerate(items):
            t = v.detach().to(device="cpu", dtype=torch.float32).contiguous()
            keep.append(t)
            arr[i].name, arr[i].data, arr[i].dtype, arr[i].ndim = k.encode(), t.data_ptr(), 0, min(t.dim(), 4)
            shape = list(t.shape)
            if len(shape) > 4:      # conv weights are 5-D: fold the kernel axes (pcd_named_tensor carries 4 dims)
                shape = shape[:3] + [int(torch.tensor(shape[3:]).prod())]
            for d, n in enumerate(shape):
                arr[i].shape[d] = n
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.lib().pcd_vae3d_create(arr, len(items), _lib.PRECISION[precision], idx, C.byref(h)))
        self._h, self.device, self.precision = h, device, precision
        self.latent_dim = int(state_dict[[k for k in state_dict if k.endswith("decoder_input.weight")][0]].shape[1])

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pcd_vae3d_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        _lib._require_cuda(z, "z")
        z = z.to(torch.float32).contiguous()
        assert z.dim() == 2 and z.shape[1] == self.latent_dim, "z must be [B, latent_dim]"
        out = torch.empty(z.shape[0], 1, 32, 32, 32, device=z.device, dtype=torch.float32)
        _lib.check(_lib.lib().pcd_vae3d_decode(self._h, z.data_ptr(), out.data_ptr(), z.shape[0], _lib.stream_ptr(z.device)))
        return out

    TAP_SHAPES = {-1: (4, 512), 0: (8, 256), 2: (8, 256), 3: (16, 128), 5: (16, 128), 6: (32, 64), 8: (32, 64), 9: (32, 32),
                  11: (32, 32)}

    def tap(self, z: torch.Tensor, seq_index: int) -> torch.Tensor:
        """Parity hook: activation after nn.Sequential index `seq_index` (-1 = decoder_input) as [B, C, D, H, W] on the host."""
        _lib._require_cuda(z, "z")
        z = z.to(torch.float32).contiguous()
        G, Cn = self.TAP_SHAPES[seq_index]
        out = torch.empty(z.shape[0], G, G, G, Cn, dtype=torch.float32)
        _lib.check(_lib.lib().pcd_vae3d_tap(self._h, z.data_ptr(), z.shape[0], seq_index, out.data_ptr(), out.numel(),
                                            _lib.stream_ptr(z.device)))
        return out.permute(0, 4, 1, 2, 3).contiguous()

    def profile(self, z: torch.Tensor):
        """[(name, ms, algorithmic FLOPs)] of one eager decode, CUDA-event timed per launch."""
        _lib._require_cuda(z, "z")
        z = z.to(torch.float32).contiguous()
        cap, stride = 64, 48
        ms, fl = (C.c_float * cap)(), (C.c_double * cap)()
        names, n = C.create_string_buffer(cap * stride), C.c_int32(0)
        vox = torch.empty(z.shape[0], 1, 32, 32, 32, device=z.device, dtype=torch.float32)
        _lib.check(_lib.lib().pcd_vae3d_profile(self._h, z.data_ptr(), vox.data_ptr(), z.shape[0], ms, fl, names, stride, cap,
                                                C.byref(n), _lib.stream_ptr(z.device)))
        return [(names.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode(), float(ms[i]), float(fl[i])) for i in range(n.value)]


class Vae3dEncoderEngine:
    """Owns the opaque pcd_vae3d_encoder handle built from the encoder half of a VAE3DLarge state_dict (`encoder.*`,
    `fc_mu.*`, `fc_logvar.*`, with or without the `vae.` prefix)."""

    TAP_SHAPES = {0: (32, 32), 2: (32, 64), 3: (16, 64), 5: (16, 128), 6: (8, 128), 8: (8, 256), 9: (4, 256), 11: (4, 512)}

    def __init__(self, state_dict, device: torch.device, precision: str = DEFAULT_PRECISION):
        if device.type != "cuda":
            raise _lib.PcdError("the B200 voxel encoder needs a CUDA device; there is no CPU fallback")
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
            shape = list(t.shape)
            if len(shape) > 4:      # conv weights are 5-D: fold the kernel axes (pcd_named_tensor carries 4 dims)
                shape = shape[:3] + [int(torch.tensor(shape[3:]).prod())]
            for d, n in enumerate(shape):
                arr[i].shape[d] = n
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.lib().pcd_vae3d_encoder_create(arr, len(items), _lib.PRECISION[precision], idx, C.byref(h)))
        self._h, self.device, self.precision = h, device, precision
        self.latent_dim = int(state_dict[[k for k in state_dict if k.endswith("fc_mu.weight")][0]].shape[0])

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pcd_vae3d_encoder_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _grid(x: torch.Tensor) -> torch.Tensor:
        _lib._require_cuda(x, "x")
        if x.dim() != 5 or tuple(x.shape[1:]) != (1, 32, 32, 32):
            raise ValueError("x must be [B, 1, 32, 32, 32], got %s" % (tuple(x.shape),))
        return x.to(torch.float32).contiguous()

    def encode(self, x: torch.Tensor):
        x = self._grid(x)
        B = x.shape[0]
        mu = torch.empty(B, self.latent_dim, device=x.device, dtype=torch.float32)
        logvar = torch.empty_like(mu)
        _lib.check(_lib.lib().pcd_vae3d_encode(self._h, x.data_ptr(), mu.data_ptr(), logvar.data_ptr(), B, _lib.stream_ptr(x.device)))
        return mu, logvar

    def tap(self, x: torch.Tensor, seq_index: int) -> torch.Tensor:
        """Parity hook: activation after encoder index `seq_index` as [B, C, D, H, W] on the host ([B, 512] for 12)."""
        x = self._grid(x)
        B = x.shape[0]
        if seq_index == 12:
            out = torch.empty(B, 512, dtype=torch.float32)
        else:
            G, Cn = self.TAP_SHAPES.get(seq_index, (1, 1))
            out = torch.empty(B, G, G, G, Cn, dtype=torch.float32)
        _lib.check(_lib.lib().pcd_vae3d_encoder_tap(self._h, x.data_ptr(), B, seq_index, out.data_ptr(), out.numel(),
                                                    _lib.stream_ptr(x.device)))
        return out if seq_index == 12 else out.permute(0, 4, 1, 2, 3).contiguous()

    def profile(self, x: torch.Tensor):
        """[(name, ms, algorithmic FLOPs)] of one eager encode, CUDA-event timed per launch."""
        x = self._grid(x)
        B = x.shape[0]
        cap, stride = 64, 48
        ms, fl = (C.c_float * cap)(), (C.c_double * cap)()
        names, n = C.create_string_buffer(cap * stride), C.c_int32(0)
        mu = torch.empty(B, self.latent_dim, device=x.device, dtype=torch.float32)
        logvar = torch.empty_like(mu)
        _lib.check(_lib.lib().pcd_vae3d_encoder_profile(self._h, x.data_ptr(), mu.data_ptr(), logvar.data_ptr(), B, ms, fl, names,
                                                        stride, cap, C.byref(n), _lib.stream_ptr(x.device)))
        return [(names.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode(), float(ms[i]), float(fl[i])) for i in range(n.value)]


def voxel_tensor_to_point_clouds(voxel_grid: torch.Tensor, threshold: float = 0.5):
    """Reference utils.py:511-539 on the GPU: per sample the voxels above `threshold` in torch.where order as (x, y, z)
    points in [-1, 1].  Returns a list of [n_i, 3] tensors (views of one packed buffer; empty samples give [0, 3])."""
    _lib._require_cuda(voxel_grid, "voxel_grid")
    assert voxel_grid.dim() == 5 and voxel_grid.shape[1] == 1, "voxel_grid must be [B, 1, D, H, W]"
    v = voxel_grid.to(torch.float32).contiguous()
    B, _, D, H, W = v.shape
    counts = torch.empty(B, device=v.device, dtype=torch.int32)
    s = _lib.stream_ptr(v.device)
    _lib.check(_lib.lib().pcd_voxel_count(v.data_ptr(), B, D, H, W, float(threshold), counts.data_ptr(), s))
    ends = torch.cumsum(counts.to(torch.int64), 0)
    offsets = (ends - counts).contiguous()
    ends_host = ends.cpu().tolist()           # ragged output: the sizes have to reach the host (as torch.where does)
    total = ends_host[-1] if B > 0 else 0
    pts = torch.empty(max(total, 1), 3, device=v.device, dtype=torch.float32)
    if total > 0:
        _lib.check(_lib.lib().pcd_voxel_points(v.data_ptr(), B, D, H, W, float(threshold), offsets.data_ptr(), pts.data_ptr(), s))
    out, lo = [], 0
    for hi in ends_host:
        out.append(pts[lo:hi])
        lo = hi
    return out
