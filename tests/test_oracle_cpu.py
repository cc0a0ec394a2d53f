"""CPU pinning of the oracle (`-m "not gpu"`):
  1. against golden vectors generated from the real reference (tests/golden/make_golden.py ->
     reference_golden.npz) — runs anywhere;
  2. against the reference's own functions imported live, when a checkout is named by SVGB200_REFERENCE
     (skipped otherwise; 1. pins the same functions);
  3. BASELINE config[0]: 1 head, S=1024, fixed spatial block mask, naive torch attention on CPU.
"""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "golden"))
from ref_import import import_kmeans_utils, import_placement, reference_available  # noqa: E402

from oracle import attention as oa  # noqa: E402
from oracle import kmeans as ok  # noqa: E402
from oracle import layout as ol  # noqa: E402

G = np.load(HERE / "golden" / "reference_golden.npz")


def T(name):
    return torch.from_numpy(G[name])


def test_varblock_attention_matches_reference_golden():
    o = oa.dynamic_block_sparse_fwd(T("vb_q"), T("vb_k"), T("vb_v"), T("vb_map"), T("vb_qs"), T("vb_ks"))
    torch.testing.assert_close(o, T("vb_o"), rtol=1e-5, atol=1e-6)
    assert torch.all(o[0, 0, int(G["vb_qs"][0, 0, 0]): int(G["vb_qs"][0, 0, :2].sum())] == 0)  # fully masked q-block


def test_dynamic_map_matches_reference_golden_up_to_ties():
    qc, kc = T("dm_qc").bfloat16(), T("dm_kc").bfloat16()
    # this golden was produced by the reference running on the CPU: torch's CPU cumsum (fp32 running sum, rounded per
    # element).  The GPU semantics (bf16 Sklansky scan) is pinned by tests/test_golden_kmeans_cpu.py.
    mine = ok.identify_dynamic_map(qc, kc, T("dm_qs"), T("dm_ks"), 0.9, 0.1, cumsum="cpu")
    ref = T("dm_map")
    probs = T("dm_probs")
    assert torch.equal(mine.sum(-1), ref.sum(-1))  # same number of kept clusters per row
    diff = mine != ref
    for b, h, i in zip(*torch.nonzero(diff.any(-1), as_tuple=True)):
        vals = probs[b, h, i][diff[b, h, i]]
        assert len(set(vals.tolist())) == 1, "differences must be ties of one probability value at the cut"
    torch.testing.assert_close(ok.density_calculation(ref, T("dm_qs"), T("dm_ks")), T("dm_density"), rtol=1e-6, atol=0)


def test_permutation_matches_reference_golden():
    x, labels = T("pm_x"), T("pm_labels")
    perm = ol.stable_argsort_labels(labels[0].numpy())
    xp = ol.permute_gather(x[0], perm)
    # the reference's argsort is unstable: compare cluster-wise multisets + exact inverse round trip
    ref_idx = G["pm_idx"][0]
    for h in range(2):
        assert np.array_equal(labels[0, h].numpy()[perm[h]], labels[0, h].numpy()[ref_idx[h]])
    assert torch.equal(ol.permute_scatter(xp, perm), x[0])
    assert torch.equal(T("pm_xr"), x)
    assert torch.equal(ol.permute_gather(x[0], ref_idx), T("pm_xp")[0])


@pytest.mark.parametrize("name,text_first", [("hy", False), ("cog", True)])
def test_placement_matches_reference_golden(name, text_first):
    ctx, F, P = (int(x) for x in G[f"pl_{name}_dims"])
    q, best = T(f"pl_{name}_q"), G[f"pl_{name}_best"]
    cfg, H, S, D = q.shape
    out = ol.head_placement(q.view(cfg * H, S, D), best.reshape(-1), ctx, F, P, text_first=text_first)
    assert torch.equal(out.view(cfg, H, S, D), T(f"pl_{name}_qo"))
    back = ol.head_placement(out, best.reshape(-1), ctx, F, P, text_first=text_first, inverse=True)
    assert torch.equal(back.view(cfg, H, S, D), T(f"pl_{name}_back"))
    assert torch.equal(back.view(cfg, H, S, D), q)


def test_mask_mods_match_reference_golden():
    qi = torch.arange(0, 700).view(-1, 1)
    ki = torch.arange(0, 700).view(1, -1)
    assert np.array_equal(oa.wan_mask_mod(5, 140, 1.3)(qi, ki).numpy(), G["mm_wan"])
    assert np.array_equal(oa.cog_mask_mod(30, 5, 134, 1.2)(qi, ki).numpy(), G["mm_cog"])
    assert np.array_equal(oa.cog_mask_mod(30, 5, 134, 1.2, attn_sink=True)(qi, ki).numpy(), G["mm_cog_sink"])
    # the engine's parametrisation of the same masks
    assert np.array_equal(oa.generic_mask_fn(2, 140, 0, oa.wan_band_width(1.3, 140))(qi, ki).numpy(), G["mm_wan"])
    assert np.array_equal(oa.generic_mask_fn(3, 30, 30, oa.hy_band_width(1.2, 134))(qi, ki).numpy(), G["mm_cog"])
    np.testing.assert_allclose([oa.sparsity_to_width(0.3, 0, 21, 3600), oa.sparsity_to_width(0.25, 256, 33, 3600),
                                oa.sparsity_to_width(0.25, 226, 11, 4080)], G["s2w"], rtol=1e-12)


def test_hy_mask_generic_parametrisation_equals_mask_mod():
    """hyvideo/utils.py cannot be imported (diffusers); the oracle restates it and the engine's
    (mode, m0, m1, m2) form must be the same function."""
    ctx, plen, F, P, mul = 40, 17, 4, 150, 1.3
    S = ctx + F * P
    qi = torch.arange(S).view(-1, 1)
    ki = torch.arange(S).view(1, -1)
    a = oa.hy_mask_mod(ctx, plen, F, P, mul)(qi, ki)
    b = oa.generic_mask_fn(1, F * P, F * P + plen, oa.hy_band_width(mul, P))(qi, ki)
    assert torch.equal(a, b)
    assert a[F * P + plen:, : F * P + plen].sum() == 0 and a[F * P + plen:, F * P + plen:].all()


def test_baseline_config0_plumbing():
    """BASELINE.json configs[0]: 1 head, S=1024, fixed spatial block mask (F=8, P=128, mul=1), naive
    torch attention on CPU.  Two independent formulations of the oracle must agree."""
    g = torch.Generator().manual_seed(0)
    S, H, D = 1024, 1, 128
    q, k, v = (torch.randn(S, H, D, generator=g) for _ in range(3))
    bmask, bsz = oa.ref_gen_spatial_mask(8, 128, 1)
    em = oa.gen_mask_block2element(bmask, bsz, 0)
    o1 = oa.ref_torch_attn_impl(q, k, v, em)
    keep = torch.from_numpy(bmask >= 0)
    sz = torch.full((1, 1, 8), 128)
    o2 = oa.dynamic_block_sparse_fwd(q.permute(1, 0, 2)[None], k.permute(1, 0, 2)[None], v.permute(1, 0, 2)[None],
                                     keep[None, None], sz, sz)
    torch.testing.assert_close(o1.permute(1, 0, 2)[None], o2, rtol=1e-5, atol=1e-6)
    assert abs(em.float().mean().item() - (3 * 8 - 2 + 6) / 64) < 1e-6  # band + first-frame column


def test_profiling_masks_match_literal_construction():
    """oracle.profiling_mask_rows (analytic) == the reference's literal block painting + reshape/permute
    (hyvideo/utils.py:47-93, wan/utils.py:63-110) on a size where the S x S mask is affordable."""
    import math

    for layout, ctx, F, P in (("hy", 16, 3, 200), ("wan", 0, 4, 150)):
        V, S = F * P, ctx + F * P
        thres = (P * (1.5 if layout == "hy" else 2)) // 128
        pix = torch.zeros(V, V, dtype=torch.bool)
        if layout == "wan":
            pix[:, :P] = True
        nb = math.ceil(V / 128)
        for i in range(nb):
            for j in range(nb):
                if abs(i - j) < thres:
                    pix[i * 128:(i + 1) * 128, j * 128:(j + 1) * 128] = True
        for name in ("spatial", "temporal"):
            m = pix if name == "spatial" else pix.reshape(P, F, P, F).permute(1, 0, 3, 2).reshape(V, V)
            full = torch.zeros(S, S, dtype=torch.bool)
            full[:V, :V] = m
            if layout == "hy":
                full[V:, :] = True
                full[:, V:] = True
            rows = list(range(0, S, 7))
            got = oa.profiling_mask_rows(name, rows, layout, ctx, F, P)
            assert torch.equal(got, full[rows]), (layout, name)


@pytest.mark.skipif(not reference_available(), reason="reference not importable (no SVGB200_REFERENCE, no baseline/_ref)")
def test_live_reference_functions():
    ku = import_kmeans_utils()
    g = torch.Generator().manual_seed(5)
    B, H, S, D = 1, 2, 64, 16
    q, k, v = (torch.randn(B, H, S, D, generator=g) for _ in range(3))
    qs = torch.tensor([[[10, 0, 30, 24], [64, 0, 0, 0]]])
    ks = torch.tensor([[[5, 5, 40, 14, 0], [0, 0, 0, 60, 4]]])
    m = torch.rand(B, H, 4, 5, generator=g) > 0.4
    torch.testing.assert_close(oa.dynamic_block_sparse_fwd(q, k, v, m, qs, ks),
                               ku.dynamic_block_sparse_fwd_torch(q, k, v, m, qs, ks), rtol=1e-5, atol=1e-6)
    pl = import_placement("hyvideo")
    ctx, F, P = 5, 4, 9
    x = torch.randn(2, 3, ctx + F * P, 8, generator=g)
    best = torch.randint(0, 2, (2, 3), generator=g)
    qo, _, _ = pl.ref_hunyuan_sparse_head_placement(x.clone(), x.clone(), x.clone(), best, ctx, F, P)
    assert torch.equal(ol.head_placement(x.view(6, -1, 8), best.view(-1).numpy(), ctx, F, P).view_as(x), qo)
