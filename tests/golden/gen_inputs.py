"""Seeded input generators shared by the golden-vector scripts and the tests that consume the vectors, so that large
random inputs are stored as (seed, checksum) instead of raw tensors.  torch's CPU generator is bit-reproducible for a
given torch build (the GPU box runs the same image); every consumer checks the stored checksum first."""
import numpy as np
import torch


def smse_inputs(seed, cfg, H, S, D):
    """q, k, v bf16 [cfg,H,S,D]; head 0 gets strongly local structure so that the two profiling masks differ."""
    g = torch.Generator().manual_seed(int(seed))
    q, k, v = (torch.randn(cfg, H, S, D, generator=g).bfloat16() for _ in range(3))
    k[:, 0] = k[:, 0] * 0.2 + q[:, 0]
    return q, k, v


def checksum(*ts):
    return float(sum(t.double().sum().item() + (t.double() ** 2).sum().item() for t in ts))


def kmeans_inputs(seed, B, N, D, K, clustered=True):
    """x bf16 [B,N,D] (mixture of K/4 well-separated blobs + noise when `clustered`), init centroids = rows of x.
    clustered == 2: exactly K well-separated blobs, init = blob centres + small noise (a well-conditioned Lloyd run:
    every point keeps a large margin, so two correct implementations must agree on the labels, not just on inertia)."""
    g = torch.Generator().manual_seed(int(seed))
    if int(clustered) == 2:
        centers = torch.randn(B, K, D, generator=g) * 2.0
        which = torch.randint(0, K, (B, N), generator=g)
        x = (torch.gather(centers, 1, which[..., None].expand(-1, -1, D)) + 0.5 * torch.randn(B, N, D, generator=g)).bfloat16()
        init = (centers + 0.3 * torch.randn(B, K, D, generator=g)).bfloat16()
        return x, init
    if clustered:
        nb = max(2, K // 4)
        centers = torch.randn(B, nb, D, generator=g) * 2.0
        which = torch.randint(0, nb, (B, N), generator=g)
        x = torch.gather(centers, 1, which[..., None].expand(-1, -1, D)) + torch.randn(B, N, D, generator=g)
    else:
        x = torch.randn(B, N, D, generator=g)
    x = x.bfloat16()
    idx = torch.randint(0, N, (B, K), generator=g)
    init = torch.gather(x, 1, idx[..., None].expand(-1, -1, D)).contiguous()
    return x, init


def structured_qkv(seed, H, F, P, ctx, D, text_first=False, scale=1.5):
    """q, k, v bf16 [1,H,S,D] whose heads clearly prefer one profiling mask: even heads attend inside their own FRAME
    (spatial heads), odd heads to the same PATCH position across frames (temporal heads), so that best_mask_idx does
    not hinge on bf16-vs-fp32 noise in sample_mse."""
    g = torch.Generator().manual_seed(int(seed))
    V, S = F * P, ctx + F * P
    q, k, v = (torch.randn(1, H, S, D, generator=g) * 0.5 for _ in range(3))
    v = v * 2
    tok = torch.arange(V)
    frame, patch = tok // P, tok % P
    lo = ctx if text_first else 0
    for h in range(H):
        emb = torch.randn(max(F, P), D, generator=g) * scale
        idx = frame if h % 2 == 0 else patch
        q[0, h, lo:lo + V] += emb[idx]
        k[0, h, lo:lo + V] += emb[idx]
    return q.bfloat16(), k.bfloat16(), v.bfloat16()


KM_FULLSIZE = ("hyq", "hyk", "wank")  # k-means cases at the HunyuanVideo / Wan token counts
KM_GOLDEN = ("kmeans_golden.npz", "kmeans_golden_fullsize.npz")  # two files so that neither exceeds 1 MB


def split_kmeans_golden(out):
    """{name: array} -> the two dicts stored as KM_GOLDEN: the full-size cases go to the second file."""
    full = {k: v for k, v in out.items() if k.startswith("km_") and k.split("_")[1] in KM_FULLSIZE}
    return {k: v for k, v in out.items() if k not in full}, full


def load_kmeans_golden(golden_dir):
    """Both KM_GOLDEN files merged into one {name: array} dict, or None when they have not been generated."""
    paths = [golden_dir / n for n in KM_GOLDEN]
    if not all(p.exists() for p in paths):
        return None
    out = {}
    for p in paths:
        with np.load(p) as z:
            out.update({k: z[k] for k in z.files})
    return out


DM_CASES = {"hy": (2, 400, 1000, 128), "small": (3, 12, 40, 64)}


def dm_inputs():
    """Inputs of the GPU identify_dynamic_map goldens: {name: (qc, kc bf16 [1,H,*,D], k_sizes, q_sizes int32)}, drawn in
    this order from one generator (seed 41)."""
    g = torch.Generator().manual_seed(41)
    out = {}
    for name, (H, QC, KC, D) in DM_CASES.items():
        qc = (torch.randn(1, H, QC, D, generator=g) * 1.5).bfloat16()
        kc = (torch.randn(1, H, KC, D, generator=g) * 1.5).bfloat16()
        ks = torch.randint(0, 300, (1, H, KC), generator=g, dtype=torch.int32)
        qs = torch.randint(1, 300, (1, H, QC), generator=g, dtype=torch.int32)
        out[name] = (qc, kc, ks, qs)
    return out
