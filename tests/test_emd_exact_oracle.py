"""CPU: the SciPy restatement of the exact EMD (reference metrics.py:49-92, `earth_mover_distance_cpu`; tests/exact_emd_scipy.py)
against the known answer and, where the reference tree is mounted, against the reference itself; `evaluate_sets(metric="emd")`
with an injected CPU matrix function."""
import pytest
import torch

import exact_emd_scipy as S
import pcd_b200
from oracle import pointdiff_oracle as O
from oracle import ref_shim

KNOWN = 44.30706787109375   # SciPy on the cube-normalised units.py inputs: 132.9212028820274 / 3, rounded to float32


def _clouds(seed, B, N, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, N, 3, generator=g) * torch.rand(B, 1, 3, generator=g) + shift


def test_known_answer_units_inputs(golden):
    x, y = golden["cd.units.x"], golden["cd.units.y"]          # seed-0 randn(1,994,3) vs randn(1,948,3)
    got = S.exact_emd(x, y)
    assert got.dtype == torch.float32 and float(got) == KNOWN
    assert float(S.exact_emd(x[0], y[0])) == KNOWN              # [N, 3] promotion


def test_ragged_batch_is_the_mean_over_pairs():
    x, y = _clouds(1, 3, 40), _clouds(2, 3, 25, 0.3)
    per, assign = S.exact_emd(x, y, per_pair=True, return_assignment=True)
    alone = torch.stack([S.exact_emd(x[b], y[b], per_pair=True)[0] for b in range(3)])
    assert torch.equal(per, alone)
    assert float(S.exact_emd(x, y)) == float(per.mean().float())
    assert assign.shape == (3, 40) and int((assign >= 0).sum()) == 3 * 25
    for b in range(3):
        m = assign[b][assign[b] >= 0]
        assert m.unique().numel() == m.numel()


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference tree not mounted")
def test_oracle_vs_reference_cpu_emd():
    _, _, rm = ref_shim.load_reference()
    torch.manual_seed(0)
    x, y = torch.randn(1, 994, 3), torch.randn(1, 948, 3)
    assert float(rm.earth_mover_distance_cpu(x, y)) == pytest.approx(float(S.exact_emd(x, y)), rel=1e-6)
    xb, yb = _clouds(3, 4, 60), _clouds(4, 4, 50, 0.2)
    assert float(rm.earth_mover_distance_cpu(xb, yb)) == pytest.approx(float(S.exact_emd(xb, yb)), rel=1e-6)


def _oracle_emd_matrix(A, B, scale):
    ii = torch.arange(A.shape[0]).repeat_interleave(B.shape[0])
    jj = torch.arange(B.shape[0]).repeat(A.shape[0])
    return (S.exact_emd(A[ii], B[jj], per_pair=True) * scale).float().view(A.shape[0], B.shape[0])


def test_evaluate_sets_emd_with_injected_matrix():
    G, R = _clouds(5, 7, 32), _clouds(6, 6, 32, 0.1)
    want = O.set_metrics_from_matrices(_oracle_emd_matrix(G, R, 1.0), _oracle_emd_matrix(G, G, 1.0), _oracle_emd_matrix(R, R, 1.0))
    for tile in (None, 3):
        got = pcd_b200.evaluate_sets(G, R, metric="emd", matrix_fn=_oracle_emd_matrix, tile=tile)
        assert set(got) == {"mmd_emd", "cov_emd", "1nna_emd"}
        assert got["cov_emd"] == want["cov_cd"]
        assert got["mmd_emd"] == pytest.approx(want["mmd_cd"], rel=1e-6)
        assert got["1nna_emd"] == pytest.approx(want["1nna_cd"], abs=1e-6)
    with pytest.raises(ValueError):
        pcd_b200.evaluate_sets(G, R, metric="l2", matrix_fn=_oracle_emd_matrix)
