"""CPU pinning (`-m "not gpu"`) of oracle/kmeans.py against vectors produced by EXECUTING the reference's Triton
flash-k-means and its GPU identify_dynamic_map on a B200 (tests/golden/make_golden_gpu.py -> kmeans_golden.npz).
Sizes: the small / mid cases (the full-size cases are consumed by the `-m gpu` tests)."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "golden"))
from gen_inputs import checksum, dm_inputs, kmeans_inputs, load_kmeans_golden  # noqa: E402

from oracle import kmeans as ok  # noqa: E402

GK = load_kmeans_golden(HERE / "golden")
pytestmark = pytest.mark.skipif(GK is None, reason="kmeans_golden*.npz not generated yet")


def from_bits(a):
    return torch.from_numpy(a.copy()).view(torch.bfloat16)


def _have(name):
    return GK is not None and f"km_{name}_in" in GK


def _case(name):
    if not _have(name):
        pytest.skip(f"golden case {name} not generated yet")
    seed, B, N, D, K, clustered, csum = GK[f"km_{name}_in"]
    x, init = kmeans_inputs(seed, int(B), int(N), int(D), int(K), int(clustered))
    assert abs(checksum(x, init) - csum) <= 1e-6 * abs(csum), "seeded inputs differ from the generator's"
    return x, init, int(K)


@pytest.mark.parametrize("name", ["small", "mid"])
def test_oracle_assign_matches_reference_triton(name):
    x, init, K = _case(name)
    lab, margin = ok.euclid_assign(x, init, ok.row_sqnorm(x))
    ref = torch.from_numpy(GK[f"km_{name}_labels"].astype(np.int64))
    safe = margin > ok.assign_margin_threshold(init)
    assert safe.float().mean() > 0.6
    assert torch.equal(lab[safe], ref[safe])
    assert (lab != ref).float().mean() < 0.04


@pytest.mark.parametrize("name", ["small", "mid"])
def test_oracle_update_matches_reference_triton(name):
    x, init, K = _case(name)
    ref_lab = torch.from_numpy(GK[f"km_{name}_labels"].astype(np.int64))
    c_new, counts = ok.centroid_update(x, ref_lab, init)
    assert torch.equal(counts, torch.from_numpy(GK[f"km_{name}_counts"]))
    ref_c = from_bits(GK[f"km_{name}_cnew"])
    torch.testing.assert_close(c_new.float(), ref_c.float(), rtol=2 ** -7, atol=1e-6)
    assert (c_new != ref_c).float().mean() < 0.02


@pytest.mark.parametrize("name", ["small", "mid", "sep"])
@pytest.mark.parametrize("iters", [2, 8])
def test_oracle_lloyd_loop_matches_reference(name, iters):
    x, init, K = _case(name)
    lab, cen, sizes, nit = ok.batch_kmeans_euclid(x, K, iters, init_centroids=init)
    assert nit == int(GK[f"km_{name}_run{iters}_nit"])
    D = x.shape[-1]
    inertia = (x.float() - torch.gather(cen.float(), 1, lab[..., None].expand(-1, -1, D))).pow(2).sum(-1).mean(dim=1)
    np.testing.assert_allclose(inertia.numpy(), GK[f"km_{name}_run{iters}_inertia"], rtol=1e-3)
    ref_lab = torch.from_numpy(GK[f"km_{name}_run{iters}_labels"].astype(np.int64))
    # Lloyd trajectories amplify the label noise of near-tie points (several centroids compete inside one blob):
    # quality (inertia, above) is the parity statement, label agreement a sanity bound
    assert (lab == ref_lab).float().mean() > (0.999 if name == "sep" else (0.85 if iters == 2 else 0.75))
    if name == "sep":  # well-conditioned run: same labels, same centroids
        torch.testing.assert_close(cen.float(), from_bits(GK[f"km_{name}_run{iters}_cent"]).float(), rtol=2 ** -6, atol=1e-3)


def test_oracle_early_exit_matches_reference():
    seed, B, N, D, K, clustered, csum = GK["km_early_in"]
    x, init = kmeans_inputs(seed, int(B), int(N), int(D), int(K), True)
    lab, cen, sizes, nit = ok.batch_kmeans_euclid(x, int(K), 10, tol=1e9, init_centroids=init)
    assert nit == int(GK["km_early_nit"]) == 1
    assert torch.equal(cen, from_bits(GK["km_early_cent"]))
    ref_lab = torch.from_numpy(GK["km_early_labels"].astype(np.int64))
    assert (lab != ref_lab).float().mean() < 0.04


@pytest.mark.parametrize("name", ["small", "hy"])
def test_oracle_dynamic_map_matches_reference_gpu(name):
    """identify_dynamic_map executed by the reference ON THE GPU (cuBLAS bf16 scores, CUDA sort, torch's CUDA cumsum =
    bf16 Sklansky scan) vs the oracle with cumsum_like_torch_cuda: identical maps (800 x 1000 at the HunyuanVideo
    shape).  A tolerance of a few rows is left for cuBLAS summation-order effects on other inputs."""
    H, QC, KC, D = (int(v) for v in GK[f"dm_{name}_dims"])
    qc, kc, ks, qs = dm_inputs()[name]
    ref = torch.from_numpy(np.unpackbits(GK[f"dm_{name}_map"])[: H * QC * KC].reshape(1, H, QC, KC).astype(bool))
    mine = ok.identify_dynamic_map(qc, kc, qs, ks, 0.9, 0.1)
    diff = mine != ref
    rows = diff.any(-1)
    assert rows.float().mean() < 0.01, rows.float().mean()
    assert diff.sum(-1).max() <= 2
    probs = ok.weighted_softmax(torch.matmul(qc, kc.transpose(-2, -1)) / (D ** 0.5), ks.unsqueeze(-2).float()).float()
    for b, h, i in zip(*torch.nonzero(rows, as_tuple=True)):
        vals = probs[b, h, i][diff[b, h, i]]
        assert (vals.max() - vals.min()) <= 2 ** -5 * vals.max() + 1e-12


def test_cuda_scan_emulation_differs_from_fp32_running_sum():
    """The point of cumsum_like_torch_cuda: on sorted probabilities near p = 0.9 the bf16 Sklansky scan stays below an
    fp32-accumulated cumsum, so more clusters survive the cut (what the reference does on the GPU)."""
    qc, kc, ks, qs = dm_inputs()["hy"]
    a = ok.identify_dynamic_map(qc, kc, qs, ks, 0.9, 0.1, cumsum="cuda")
    b = ok.identify_dynamic_map(qc, kc, qs, ks, 0.9, 0.1, cumsum="cpu")
    assert (a.sum(-1) >= b.sum(-1)).float().mean() > 0.7 and a.sum() > 1.02 * b.sum()
    assert ok.cuda_scan_log_threads(24 * 400, 1000) == 4 and ok.cuda_scan_log_threads(400, 1000) == 5
