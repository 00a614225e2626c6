"""CPU: the voxel-VAE encoder oracle (VAE3DLarge.encode) -- the stride-2 identity the kernels rely on, the state_dict layout,
the no-CPU-fallback rule and, where the reference tree is mounted, the reference's own encode / forward."""
import pytest
import torch
import torch.nn.functional as F

import pcd_b200
from oracle import pointdiff_oracle as O
from oracle import ref_shim
import vae3d_encoder_oracle as E


def _full_checkpoint():
    sd = O.make_synthetic_vae3d_decoder_checkpoint()
    sd.update(E.make_synthetic_vae3d_encoder_checkpoint())
    return {k[4:]: t for k, t in sd.items()}


def test_strided_conv_parity_decomposition():
    """Conv3d(k=4, s=2, p=1): output o reads input 2o - 1 + k.  Written as input 2j + p, the taps are (k, p, j - o) =
    (0, 1, -1), (1, 0, 0), (2, 1, 0), (3, 0, +1): a sum over the 8 input-parity sub-grids (each the size of the output grid)
    of 2 x 2 x 2 taps each -- 64 (parity, tap) pairs, no zero MACs, out-of-range shifts = zero padding."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 5, 8, 8, 8, generator=g, dtype=torch.float64)
    w = torch.randn(7, 5, 4, 4, 4, generator=g, dtype=torch.float64)
    ref = F.conv3d(x, w, stride=2, padding=1)
    PJ = {0: (1, -1), 1: (0, 0), 2: (1, 0), 3: (0, 1)}           # k -> (parity, shift)
    out = torch.zeros_like(ref)
    pairs = 0
    for kd in range(4):
        for kh in range(4):
            for kw in range(4):
                (pd, sd), (ph, sh), (pw, sw) = PJ[kd], PJ[kh], PJ[kw]
                sub = F.pad(x[:, :, pd::2, ph::2, pw::2], (1, 1, 1, 1, 1, 1))        # parity sub-grid, zero border
                sl = sub[:, :, 1 + sd:5 + sd, 1 + sh:5 + sh, 1 + sw:5 + sw]
                out += torch.einsum("bidhw,oi->bodhw", sl, w[:, :, kd, kh, kw])
                pairs += 1
    assert pairs == 64
    assert torch.allclose(out, ref, atol=1e-12)


def test_encoder_spec_matches_container_and_full_checkpoint_loads_strictly():
    v = pcd_b200.VAE3DLarge()
    sd = v.state_dict()
    spec = E.vae3d_encoder_state_dict_spec(prefix="vae")
    for k, shape, _ in spec:
        assert tuple(sd[k[4:]].shape) == tuple(shape), k
    enc_keys = {k for k in sd if k.startswith(("encoder.", "fc_mu.", "fc_logvar."))}
    assert enc_keys == {k[4:] for k, _, _ in spec}
    v.load_state_dict(_full_checkpoint(), strict=True)


def test_encode_on_cpu_raises():
    v = pcd_b200.VAE3DLarge()
    v.load_state_dict(_full_checkpoint(), strict=True)
    x = torch.zeros(1, 1, 32, 32, 32)
    with pytest.raises(pcd_b200.PcdError):                # no CPU fallback
        v.encode(x)
    with pytest.raises(pcd_b200.PcdError):
        v(x)


def test_reparameterize_draws_like_the_reference():
    mu, logvar = torch.randn(3, 8), torch.randn(3, 8)
    torch.manual_seed(5)
    got = pcd_b200.VAE3DLarge.reparameterize(mu, logvar)
    torch.manual_seed(5)
    std = torch.exp(0.5 * logvar)
    assert torch.equal(got, mu + torch.randn_like(std) * std)


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference tree not mounted")
def test_encoder_oracle_vs_reference_module():
    _, rn, _ = ref_shim.load_reference()
    ref = rn.VAE3DLarge()
    full = _full_checkpoint()
    ref.load_state_dict(full, strict=True)
    ref.eval()
    sd = {"vae." + k: t for k, t in full.items()}
    g = torch.Generator().manual_seed(9)
    x = (torch.rand(2, 1, 32, 32, 32, generator=g) < 0.3).float()
    with torch.no_grad():
        mu, logvar = ref.encode(x)
        want_mu, want_lv = E.vae3d_encode(sd, x)
        assert torch.equal(mu, want_mu) and torch.equal(logvar, want_lv)
        torch.manual_seed(3)
        recon, fmu, flv = ref(x)
        torch.manual_seed(3)
        std = torch.exp(0.5 * want_lv)
        z = want_mu + torch.randn_like(std) * std
    assert torch.equal(fmu, want_mu) and torch.equal(flv, want_lv)
    assert torch.equal(recon, O.vae3d_decode(sd, z))
