"""Golden vectors that need a GPU: the reference's Triton flash-k-means, its GPU identify_dynamic_map, its Triton
permutation and its FlashInfer variable-block launcher, EXECUTED ON A B200 from the unmodified reference
(baseline/_ref, installed by tools/install_reference.py; /root/reference does not exist on the GPU box).

    gpurun -- python tests/golden/make_golden_gpu.py     ->  gpurun_out/kmeans_golden.npz  (copied to tests/golden/)

Functions executed (reference file:line, all in svg/kmeans_utils.py unless noted):
  euclid_assign_triton                   :562-625  (_euclid_assign_kernel :464-554, autotuned)
  triton_centroid_update_sorted_euclid   :375-421  (_centroid_update_chunk_kernel :258-322, fp32 atomics)
  batch_kmeans_Euclid                    :684-733
  identify_dynamic_map                   :864-896  (cuBLAS bf16 matmul, CUDA sort / cumsum)
  dynamic_block_sparse_fwd_flashinfer    :1319-1392
  svg/kernels/triton/permute.py:82-170   permute_tensor_by_labels_triton, apply_inverse_permutation_triton

Inputs are stored as (seed, checksum) — tests/golden/gen_inputs.py regenerates them bit-exactly on the CPU.
"""
import sys
import time
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parents[1]
sys.path.insert(0, str(HERE))
import ref_import as R  # noqa: E402
from gen_inputs import DM_CASES, KM_GOLDEN, checksum, dm_inputs, kmeans_inputs, split_kmeans_golden  # noqa: E402

BIG = ("hyq", "hyk", "wank")  # full-size cases: big arrays are stored subsampled (every 4th token / centroid)


def bits(t):
    return t.detach().contiguous().cpu().view(torch.int16).numpy()


def main():
    assert torch.cuda.is_available()
    dev = torch.device("cuda:0")
    ku = R.import_kmeans_utils()
    print("reference from", R.reference_root(), flush=True)
    out = {"torch": np.array(torch.__version__), "gpu": np.array(torch.cuda.get_device_name(0))}

    # ---- assign / update / Lloyd loop
    # name: (seed, B, N, D, K, clustered)
    cases = {"small": (21, 2, 6000, 64, 50, True), "mid": (22, 2, 5000, 128, 300, True),
             "hyq": (23, 1, 118800, 128, 400, True), "hyk": (24, 1, 118800, 128, 1000, True),
             "wank": (25, 1, 75600, 128, 1000, False), "sep": (26, 2, 8000, 64, 40, 2)}
    for name, (seed, B, N, D, K, clustered) in cases.items():
        t0 = time.time()
        x, init = kmeans_inputs(seed, B, N, D, K, clustered)
        out[f"km_{name}_in"] = np.array([seed, B, N, D, K, int(clustered), checksum(x, init)], dtype=np.float64)
        xd, cd = x.to(dev), init.to(dev)
        x_sq = (xd ** 2).sum(dim=-1)  # bf16, as batch_kmeans_Euclid computes it (:704)
        labels = ku.euclid_assign_triton(xd, cd, x_sq)
        out[f"km_{name}_labels"] = labels.cpu().numpy().astype(np.int16)
        c_new, counts = ku.triton_centroid_update_sorted_euclid(xd, labels, cd)
        out[f"km_{name}_cnew"] = bits(c_new)[:, ::4].copy() if name in BIG else bits(c_new)
        out[f"km_{name}_counts"] = counts.cpu().numpy().astype(np.int32)
        for iters in (2, 8):
            lab, cen, sizes, nit = ku.batch_kmeans_Euclid(xd, K, max_iters=iters, init_centroids=cd)
            if name not in BIG:
                out[f"km_{name}_run{iters}_labels"] = lab.cpu().numpy().astype(np.int16)
                out[f"km_{name}_run{iters}_cent"] = bits(cen)
            elif iters == 2:
                out[f"km_{name}_run{iters}_labels"] = lab.cpu().numpy().astype(np.int16)[:, ::4].copy()
                out[f"km_{name}_run{iters}_cent"] = bits(cen)[:, ::4].copy()
            out[f"km_{name}_run{iters}_sizes"] = sizes.cpu().numpy().astype(np.int32)
            out[f"km_{name}_run{iters}_nit"] = np.array(nit)
            # inertia of the returned (labels, centroids) pair in fp32: what "same quality" is measured by
            d = (xd.float() - torch.gather(cen.float(), 1, lab[..., None].expand(-1, -1, D).long())).pow(2).sum(-1)
            out[f"km_{name}_run{iters}_inertia"] = d.mean(dim=1).cpu().numpy()
        torch.cuda.synchronize()
        print(name, "done in %.1fs" % (time.time() - t0), flush=True)

    # early-exit control flow: tol large enough to stop after the first iteration (:723)
    x, init = kmeans_inputs(31, 2, 4000, 64, 32, True)
    xd, cd = x.to(dev), init.to(dev)
    lab, cen, sizes, nit = ku.batch_kmeans_Euclid(xd, 32, max_iters=10, tol=1e9, init_centroids=cd)
    out["km_early_in"] = np.array([31, 2, 4000, 64, 32, 1, checksum(x, init)], dtype=np.float64)
    out["km_early_labels"] = lab.cpu().numpy().astype(np.int16)
    out["km_early_cent"] = bits(cen)
    out["km_early_nit"] = np.array(nit)

    # ---- identify_dynamic_map on the GPU at the HunyuanVideo shape (inputs: gen_inputs.dm_inputs, stored as checksums)
    out["km_big_label_stride"], out["km_big_cent_stride"] = np.array(4), np.array(4)
    for name, (qc, kc, ks, qs) in dm_inputs().items():
        H, QC, KC, D = DM_CASES[name]
        dm = ku.identify_dynamic_map(qc.to(dev), kc.to(dev), qs.to(dev), ks.to(dev), 0.9, 0.1)
        out[f"dm_{name}_in"] = np.array([checksum(qc, kc, ks.float(), qs.float())])
        out[f"dm_{name}_map"] = np.packbits(dm.cpu().numpy())
        out[f"dm_{name}_dims"] = np.array([H, QC, KC, D])
        if name != "hy":
            probs = ku.weighted_softmax(torch.matmul(qc.to(dev), kc.to(dev).transpose(-2, -1)) / (D ** 0.5),
                                        ks.to(dev).unsqueeze(-2).float())
            out[f"dm_{name}_probs"] = bits(probs)

    # ---- Triton permutation (argsort is unstable: the test compares cluster-wise) + inverse
    perm_mod = __import__('importlib').import_module("svg.kernels.triton.permute")
    g = torch.Generator().manual_seed(42)
    x = torch.randn(1, 2, 3000, 64, generator=g).bfloat16()
    labels = torch.randint(0, 37, (2, 3000), generator=g)
    xp, idx = perm_mod.permute_tensor_by_labels_triton(x.to(dev), labels.to(dev), dim=2)
    xr = perm_mod.apply_inverse_permutation_triton(xp, idx, dim=2)
    out.update(pm_seed=np.array(42), pm_idx=idx.cpu().numpy().astype(np.int32),
               pm_gather_equal=np.array(bool(torch.equal(xp.cpu()[0, 0], x[0, 0][idx.cpu().long()[0]]))),
               pm_roundtrip_equal=np.array(bool(torch.equal(xr.cpu(), x))))

    # ---- the live sparse kernel: FlashInfer variable-block launcher, small shape, bf16
    try:
        g = torch.Generator().manual_seed(43)
        B, H, S, D, QC, KC = 1, 2, 2048, 128, 10, 50
        q, k, v = (torch.randn(B, H, S, D, generator=g).bfloat16() for _ in range(3))

        def part(n):
            cuts = torch.sort(torch.randperm(S - 1, generator=g)[: n - 1] + 1)[0]
            return torch.diff(torch.cat([torch.tensor([0]), cuts, torch.tensor([S])])).int()
        qs = torch.stack([part(QC) for _ in range(H)])[None]
        ks = torch.stack([part(KC) for _ in range(H)])[None]
        m = torch.rand(B, H, QC, KC, generator=g) < 0.4
        m[..., 0] = True
        o, how = R.reference_flashinfer_varblock(q.to(dev), k.to(dev), v.to(dev), m.to(dev), qs.to(dev), ks.to(dev))
        out["fi_how"] = np.array(how)
        out.update(fi_seed=np.array(43), fi_dims=np.array([B, H, S, D, QC, KC]), fi_qs=qs.numpy(), fi_ks=ks.numpy(),
                   fi_map=m.numpy(), fi_o=bits(o).reshape(B, H, S, D)[:, :, ::4].copy(),
                   fi_o_row_stride=np.array(4), fi_checksum=np.array(checksum(q, k, v)))
    except Exception as e:  # noqa: BLE001  (FlashInfer JIT may be unavailable offline)
        out["fi_error"] = np.array(repr(e)[:300])
        print("flashinfer golden skipped:", repr(e)[:300])

    dst = ROOT / "gpurun_out"
    dst.mkdir(exist_ok=True)
    for name, part in zip(KM_GOLDEN, split_kmeans_golden(out)):
        np.savez_compressed(dst / name, **part)
        print("wrote", dst / name)


if __name__ == "__main__":
    main()
