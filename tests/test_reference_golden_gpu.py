"""GPU parity against vectors produced by EXECUTING THE REFERENCE (no restated oracle in between):

  tests/golden/svg1_golden.npz    real processors' bf16 sample_mse (HY / Wan / Cog), run on CPU in the build container
  tests/golden/kmeans_golden.npz  the reference's Triton flash-k-means, GPU identify_dynamic_map, Triton permutation and
                                  FlashInfer variable-block launcher, run ON A B200 (tests/golden/make_golden_gpu.py)

Integer outputs are compared exactly wherever the arithmetic is well-conditioned: a point whose best and second-best
centroid distances are closer than the fp32 / bf16 evaluation noise can legitimately land on either side in two
different kernels (the reference's own autotuned Triton tiles change the summation order from run to run); such
points are excluded by an fp32 margin test and counted."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "golden"))
from gen_inputs import checksum, dm_inputs, kmeans_inputs, load_kmeans_golden, smse_inputs  # noqa: E402

BIG = ("hyq", "hyk", "wank")  # stored subsampled: every 4th token of the Lloyd-loop labels, every 4th centroid

G1 = np.load(HERE / "golden" / "svg1_golden.npz")
GK = load_kmeans_golden(HERE / "golden")
needs_km = pytest.mark.skipif(GK is None, reason="tests/golden/kmeans_golden*.npz not generated yet")


def from_bits(a, dtype=torch.bfloat16):
    return torch.from_numpy(a.copy()).view(dtype)


# ------------------------------------------------------------------------------------------------ sample_mse
@pytest.mark.parametrize("case", ["hy0", "hy1", "wan0", "wan1", "cog0", "cog1", "cog2", "cog3"])
def test_sample_mse_matches_reference_processor(cuda, case):
    """svgb_sample_mse (analytic masks, fp32 softmax) vs <Model>_SVGAttn_Processor.sample_mse (materialised masks,
    bf16 eager torch): MSE within the reference's own bf16 noise, identical best_mask_idx wherever decided."""
    from svgb200.models import cog, hyvideo, wan

    seed, cfg, H, S, D, csum = G1[f"smse_{case}_in"]
    q, k, v = smse_inputs(seed, int(cfg), int(H), int(S), int(D))
    assert abs(checksum(q, k, v) - csum) <= 1e-6 * abs(csum)
    rows = torch.from_numpy(G1[f"smse_{case}_rows"])
    ref = torch.from_numpy(G1[f"smse_{case}_mses"])
    fam = case[:-1]
    if fam == "hy":
        core_obj = hyvideo.SVG1Core(16, 3, 200, num_sampled_rows=24, sample_mse_max_row=500)
        core_obj.smse_layout = 0
    elif fam == "wan":
        core_obj = wan.SVG1Core(0, 4, 150, num_sampled_rows=24, sample_mse_max_row=600)
        core_obj.smse_layout = 1
    else:
        core_obj = cog.CogSVG1Core.__new__(cog.CogSVG1Core)
        cog.SVG1Core.__init__(core_obj, 30, 3, 200, num_sampled_rows=24, sample_mse_max_row=630)
    got = core_obj.sample_mse(q.to(cuda), k.to(cuda), v.to(cuda), sampled_rows=rows).float().cpu()
    nan_ref = torch.isnan(ref)
    assert torch.equal(torch.isnan(got), nan_ref)  # Cog: sampled text rows -> NaN temporal MSE (cog/utils.py:76-86)
    ok = ~nan_ref
    torch.testing.assert_close(got[ok], ref[ok], rtol=6e-2, atol=1e-5)
    best_ref = torch.from_numpy(G1[f"smse_{case}_best"])
    decided = ((ref[0] - ref[1]).abs() > 0.1 * torch.maximum(ref[0], ref[1])) | nan_ref.any(0)
    assert torch.equal(torch.argmin(got, dim=0)[decided], best_ref[decided])


# ------------------------------------------------------------------------------------------------ flash k-means
def _km_case(name):
    if f"km_{name}_in" not in GK:
        pytest.skip(f"golden case {name} not generated yet")
    seed, B, N, D, K, clustered, csum = GK[f"km_{name}_in"]
    x, init = kmeans_inputs(seed, int(B), int(N), int(D), int(K), int(clustered))
    assert abs(checksum(x, init) - csum) <= 1e-6 * abs(csum), "seeded inputs differ from the generator's"
    return x, init, int(K)


def _margin(x, c, chunk=8192):
    """fp32 (best, second best) squared-distance gap per point, on the GPU (test plumbing)."""
    out = []
    for b in range(x.shape[0]):
        cf = c[b].float()
        csq = (cf * cf).sum(-1)
        for s in range(0, x.shape[1], chunk):
            xf = x[b, s:s + chunk].float()
            d = (xf * xf).sum(-1, keepdim=True) + csq[None] - 2 * xf @ cf.T
            t = torch.topk(d, 2, dim=-1, largest=False).values
            out.append(t[:, 1] - t[:, 0])
    return torch.cat(out).view(x.shape[0], -1)


@needs_km
@pytest.mark.parametrize("name", ["small", "mid", "hyq", "hyk", "wank", "sep"])
def test_kmeans_assign_matches_reference_triton(cuda, name):
    """euclid_assign_triton (svg/kmeans_utils.py:562-625) run on a B200 vs svgb_kmeans_assign, incl. the HunyuanVideo
    sizes N=118 800 with K=400 / K=1000."""
    from svgb200 import kmeans_utils as ku

    x, init, K = _km_case(name)
    xd, cd = x.to(cuda), init.to(cuda)
    x_sq = (xd ** 2).sum(dim=-1)
    lab = ku.euclid_assign_triton(xd, cd, x_sq)
    ref = torch.from_numpy(GK[f"km_{name}_labels"].astype(np.int64)).to(cuda)
    assert lab.dtype == torch.int64 and lab.shape == ref.shape
    from oracle.kmeans import assign_margin_threshold

    # the reference's own ||c||^2 term is only good to ~2 bf16 ulps (oracle/kmeans.py docstring): exact elsewhere
    safe = _margin(xd, cd) > assign_margin_threshold(init)
    assert safe.float().mean() > 0.5, safe.float().mean()
    bad_safe = (lab[safe] != ref[safe]).float().mean().item()
    assert bad_safe <= 1e-4, bad_safe  # exact; at N = 118 800 x K = 1000 a handful of 6-sigma points may slip through
    assert (lab != ref).float().mean() < 0.05
    # every choice (ours and the reference's) is a near-minimiser: inertia agrees
    def inertia(l):
        return (xd.float() - torch.gather(cd.float(), 1, l[..., None].expand(-1, -1, xd.shape[-1]))).pow(2).sum(-1).mean()
    torch.testing.assert_close(inertia(lab), inertia(ref), rtol=1e-3, atol=0)


@needs_km
@pytest.mark.parametrize("name", ["small", "mid", "hyq", "hyk", "wank", "sep"])
def test_kmeans_update_matches_reference_triton(cuda, name):
    """triton_centroid_update_sorted_euclid (:375-421; fp32 atomics, order not defined) given the REFERENCE's labels:
    counts exact, centroids equal up to one 16-bit ulp of summation-order noise, empty clusters keep the old one."""
    from svgb200 import kmeans_utils as ku

    x, init, K = _km_case(name)
    ref_lab = torch.from_numpy(GK[f"km_{name}_labels"].astype(np.int64))
    c_new, counts = ku.triton_centroid_update_sorted_euclid(x.to(cuda), ref_lab.to(cuda), init.to(cuda))
    assert torch.equal(counts.cpu(), torch.from_numpy(GK[f"km_{name}_counts"]))
    ref_c = from_bits(GK[f"km_{name}_cnew"])
    mine_c = c_new.cpu()[:, ::4] if name in BIG else c_new.cpu()
    torch.testing.assert_close(mine_c.float(), ref_c.float(), rtol=2 ** -7, atol=1e-6)
    assert (mine_c != ref_c).float().mean() < 0.02
    empty = torch.from_numpy(GK[f"km_{name}_counts"]) == 0
    assert torch.equal(c_new.cpu()[empty], init[empty])


@needs_km
@pytest.mark.parametrize("name", ["small", "mid", "hyq", "hyk", "wank", "sep"])
@pytest.mark.parametrize("iters", [2, 8])
def test_kmeans_run_matches_reference_loop(cuda, name, iters):
    """batch_kmeans_Euclid (:684-733) from the same initial centroids: same iteration count, inertia of the returned
    (labels, centroids) pair within 1e-3, label agreement, and the return convention (labels of the LAST assignment,
    centroids = the updated ones)."""
    from svgb200 import kmeans_utils as ku

    x, init, K = _km_case(name)
    xd = x.to(cuda)
    lab, cen, sizes, nit = ku.batch_kmeans_Euclid(xd, K, max_iters=iters, init_centroids=init.to(cuda))
    assert int(nit) == int(GK[f"km_{name}_run{iters}_nit"])
    D = x.shape[-1]
    inertia = (xd.float() - torch.gather(cen.float(), 1, lab[..., None].expand(-1, -1, D))).pow(2).sum(-1).mean(dim=1)
    np.testing.assert_allclose(inertia.cpu().numpy(), GK[f"km_{name}_run{iters}_inertia"], rtol=1e-3)
    assert int(sizes.sum()) == x.shape[0] * x.shape[1]
    ref_sizes = torch.from_numpy(GK[f"km_{name}_run{iters}_sizes"]).long()
    well_conditioned = name == "sep"
    moved = (sizes.cpu().long() - ref_sizes).abs().sum().item()
    # K > number of blobs (several centroids compete inside one blob): Lloyd amplifies near-tie label noise, the
    # partition of a blob between its centroids drifts while the quality (inertia, above) stays the same
    assert moved <= (0.002 if well_conditioned else 0.6) * x.shape[0] * x.shape[1], moved
    if f"km_{name}_run{iters}_labels" not in GK:
        return  # full-size cases keep labels / centroids of the 2-iteration run only
    stride = 4 if name in BIG else 1
    ref_lab = torch.from_numpy(GK[f"km_{name}_run{iters}_labels"].astype(np.int64))
    agree = (lab.cpu()[:, ::stride] == ref_lab).float().mean().item()
    assert agree > (0.999 if well_conditioned else 0.5), agree
    if well_conditioned:  # same labels -> same centroids up to fp32 summation order
        ref_c = from_bits(GK[f"km_{name}_run{iters}_cent"]).float()
        torch.testing.assert_close(cen.cpu().float()[:, ::stride], ref_c, rtol=2 ** -6, atol=1e-3)


@needs_km
def test_kmeans_early_exit_matches_reference(cuda):
    """tol so large that the loop breaks after the first iteration (:723): the reference returns the INITIAL centroids
    with the labels assigned against them, n_iter = 1."""
    from svgb200 import kmeans_utils as ku

    seed, B, N, D, K, clustered, csum = GK["km_early_in"]
    x, init = kmeans_inputs(seed, int(B), int(N), int(D), int(K), True)
    lab, cen, sizes, nit = ku.batch_kmeans_Euclid(x.to(cuda), int(K), max_iters=10, tol=1e9, init_centroids=init.to(cuda))
    assert int(nit) == int(GK["km_early_nit"]) == 1
    assert torch.equal(cen.cpu(), from_bits(GK["km_early_cent"])) and torch.equal(cen.cpu(), init)
    ref_lab = torch.from_numpy(GK["km_early_labels"].astype(np.int64))
    assert (lab.cpu() != ref_lab).float().mean() < 0.04


# ------------------------------------------------------------------------------------------------ dynamic map
@needs_km
@pytest.mark.parametrize("name", ["hy", "small"])
def test_dynamic_map_matches_reference_gpu(cuda, name):
    """identify_dynamic_map (:864-896) executed on the GPU (cuBLAS bf16 scores, CUDA sort / bf16 cumsum) vs
    svgb_dynamic_map at QC=400 / KC=1000.  Rows may differ only where the bf16 rounding of a probability or of the
    running sum sits on a boundary (different fp32 summation order) or where torch's unstable sort broke a tie at the
    cut differently; every such difference must be a near-tie of the probability values involved."""
    from svgb200 import kmeans_utils as ku

    from oracle import kmeans as ok

    H, QC, KC, D = (int(v) for v in GK[f"dm_{name}_dims"])
    qc, kc, ks, qs = dm_inputs()[name]
    csum = float(GK[f"dm_{name}_in"][0])
    assert abs(checksum(qc, kc, ks.float(), qs.float()) - csum) <= 1e-6 * abs(csum), "seeded inputs differ"
    ref = torch.from_numpy(np.unpackbits(GK[f"dm_{name}_map"])[: H * QC * KC].reshape(1, H, QC, KC).astype(bool))
    # probabilities only serve to show that disputed entries are near-ties: the oracle's (CPU bf16) are close enough
    probs = ok.weighted_softmax(torch.matmul(qc, kc.transpose(-2, -1)) / (D ** 0.5), ks.unsqueeze(-2).float()).float()
    got = ku.identify_dynamic_map(qc.to(cuda), kc.to(cuda), qs.to(cuda), ks.to(cuda), 0.9, 0.1).cpu()
    assert got.shape == ref.shape and got.dtype == torch.bool
    diff = got != ref
    rows_diff = diff.any(-1)
    # exact since the kernel reproduces torch's CUDA bf16 scan; a few rows are left for fp32 summation-order effects
    # in the bf16-rounded scores (cuBLAS vs our dot products)
    assert rows_diff.float().mean() < 0.03, rows_diff.float().mean()
    assert diff.sum(-1).max() <= 4
    for b, h, i in zip(*torch.nonzero(rows_diff, as_tuple=True)):
        p = probs[b, h, i]
        vals = p[diff[b, h, i]]
        # the disputed clusters all sit at the cut: their probabilities are within 2 bf16 ulps of each other
        assert (vals.max() - vals.min()) <= 2 ** -5 * vals.max() + 1e-12
    # kept mass is the same up to the disputed entries
    kept_g, kept_r = (probs * got).sum(-1), (probs * ref).sum(-1)
    torch.testing.assert_close(kept_g, kept_r, rtol=0, atol=0.02)


# ------------------------------------------------------------------------------------------------ permutation
@needs_km
def test_permutation_matches_reference_triton(cuda):
    """permute_tensor_by_labels_triton (svg/kernels/triton/permute.py:82-128): torch.argsort on CUDA is not stable, so
    indices are compared cluster-wise; ours is the stable one.  The gathered tensor must be bit-identical per cluster
    as a multiset, the inverse permutation an exact round trip."""
    from svgb200 import permute as pm

    g = torch.Generator().manual_seed(int(GK["pm_seed"]))
    x = torch.randn(1, 2, 3000, 64, generator=g).bfloat16()
    labels = torch.randint(0, 37, (2, 3000), generator=g)
    xp, idx = pm.permute_tensor_by_labels_triton(x.to(cuda), labels.to(cuda), dim=2)
    assert idx.dtype == torch.int32
    ref_idx = torch.from_numpy(GK["pm_idx"]).long()
    mine = idx.cpu().long()
    assert torch.equal(torch.gather(labels, 1, mine), torch.gather(labels, 1, ref_idx))  # same cluster order
    for h in range(2):
        lab_sorted = labels[h][mine[h]]
        bounds = torch.nonzero(torch.diff(lab_sorted, prepend=torch.tensor([-1]))).flatten().tolist() + [3000]
        for a, b in zip(bounds[:-1], bounds[1:]):
            assert torch.equal(torch.sort(mine[h, a:b]).values, torch.sort(ref_idx[h, a:b]).values)
            assert torch.equal(mine[h, a:b], torch.sort(mine[h, a:b]).values)  # stable = ascending inside a cluster
    assert bool(GK["pm_roundtrip_equal"])  # the reference's own round trip on the B200
    assert torch.equal(pm.apply_inverse_permutation_triton(xp, idx, dim=2).cpu(), x)
    assert torch.equal(xp.cpu()[0, 0], x[0, 0][mine[0]])


# ------------------------------------------------------------------------------------------------ live sparse kernel
@needs_km
def test_varblock_attention_matches_reference_flashinfer(cuda):
    """dynamic_block_sparse_fwd_flashinfer (svg/kmeans_utils.py:1319-1392, the reference's LIVE SVG2 kernel) output,
    recorded on a B200, vs svgb_attn_fwd on the same inputs; tolerance of the reference's own test
    (test_sparse_attn_dyn_blk_wan.py:133: atol = rtol = 1e-2)."""
    if "fi_o" not in GK:
        pytest.skip("FlashInfer golden unavailable: " + str(GK["fi_error"]))
    from svgb200 import kmeans_utils as ku

    B, H, S, D, QC, KC = (int(v) for v in GK["fi_dims"])
    g = torch.Generator().manual_seed(int(GK["fi_seed"]))
    q, k, v = (torch.randn(B, H, S, D, generator=g).bfloat16() for _ in range(3))
    assert abs(checksum(q, k, v) - float(GK["fi_checksum"])) <= 1e-6 * abs(float(GK["fi_checksum"]))
    m, qs, ks = torch.from_numpy(GK["fi_map"]), torch.from_numpy(GK["fi_qs"]), torch.from_numpy(GK["fi_ks"])
    o = ku.dynamic_block_sparse_fwd_flashinfer(q.to(cuda), k.to(cuda), v.to(cuda), m.to(cuda), qs.to(cuda), ks.to(cuda),
                                               is_cpu=False)
    st = int(GK["fi_o_row_stride"])  # every 4th query row is stored
    torch.testing.assert_close(o.float().cpu()[:, :, ::st], from_bits(GK["fi_o"]).float(), rtol=1e-2, atol=1e-2)
