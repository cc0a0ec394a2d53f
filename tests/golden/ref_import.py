"""Import helpers for the UNMODIFIED reference.

The reference is not part of this repository.  Two places can hold it: a Sparse-VideoGen checkout named by the
environment variable SVGB200_REFERENCE and the git-ignored install `baseline/_ref` (written by
tools/install_reference.py), which is how the reference's Triton / FlashInfer code is executed on a B200 for
golden vectors and for bench.py's `ref_gpu` section.  Without either, the tests that import it skip.  Nothing in
the product package imports this module.

Packages the reference imports at module scope but that this image lacks are replaced by inert stubs — none of
them is touched by the functions we execute:
  cuvs (svg/kmeans_utils.py:6), diffusers (svg/models/*/attention.py:7-8, hyvideo/utils.py:8),
  matplotlib (svg/kernels/ops/attention_ops_wan.py:6), termcolor, IPython.
"""
import importlib
import os
import sys
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
CANDIDATES = [p for p in (os.environ.get("SVGB200_REFERENCE"), str(ROOT / "baseline" / "_ref")) if p]


def reference_root():
    for c in CANDIDATES:
        if os.path.isdir(os.path.join(c, "svg")):
            return c
    return None


def reference_available() -> bool:
    return reference_root() is not None


def _mod(name, **attrs):
    if name in sys.modules:
        m = sys.modules[name]
    else:
        m = types.ModuleType(name)
        m.__path__ = []  # behaves as a package for `import a.b.c`
        sys.modules[name] = m
        if "." in name:
            parent, child = name.rsplit(".", 1)
            setattr(_mod(parent), child, m)
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def install_stubs():
    """Inert stand-ins for the import-time dependencies this image lacks."""
    def _missing(*a, **k):
        raise RuntimeError("stubbed third-party function called")

    def have(name):
        try:
            importlib.import_module(name)
            return True
        except Exception:  # noqa: BLE001
            return False

    if not have("cuvs"):
        _mod("cuvs.cluster.kmeans", KMeansParams=object, fit=_missing)
    if not have("diffusers"):
        class Attention:  # the processors only use it as a type annotation / attribute bag
            pass

        class RMSNorm:
            pass

        _mod("diffusers.models.attention", Attention=Attention)
        _mod("diffusers.models.attention_processor", Attention=Attention)
        _mod("diffusers.models.embeddings", apply_rotary_emb=_missing)
        _mod("diffusers.models.normalization", RMSNorm=RMSNorm)
        _mod("diffusers.pipelines.hunyuan_video.pipeline_hunyuan_video",
             DEFAULT_PROMPT_TEMPLATE={"template": "", "crop_start": 0})
    if not have("matplotlib"):
        _mod("matplotlib.pyplot")
    if not have("termcolor"):
        _mod("termcolor", colored=lambda s, *a, **k: s)
    if not have("IPython"):
        _mod("IPython", embed=_missing)


def _path():
    root = reference_root()
    if root is None:
        raise ImportError("the reference is neither named by SVGB200_REFERENCE nor installed in baseline/_ref "
                          "(python tools/install_reference.py)")
    if root not in sys.path:
        sys.path.insert(0, root)
    install_stubs()
    return root


def import_kmeans_utils():
    _path()
    import svg.kmeans_utils as ku

    return ku


def import_placement(model="hyvideo"):
    _path()
    return importlib.import_module(f"svg.models.{model}.placement")


def import_model_module(model, name):
    """svg.models.<model>.<name> (attention / utils / placement) with the stubs in place."""
    _path()
    return importlib.import_module(f"svg.models.{model}.{name}")


def import_ops(name="attention_ops"):
    _path()
    return importlib.import_module(f"svg.kernels.ops.{name}")


def import_kernel_test(name):
    """svg/kernels/test/<name>.py does `from ops.attention_ops import ...` (it is run from svg/kernels)."""
    root = _path()
    kdir = os.path.join(root, "svg", "kernels")
    if kdir not in sys.path:
        sys.path.insert(0, kdir)
    tdir = os.path.join(kdir, "test")
    if tdir not in sys.path:
        sys.path.insert(0, tdir)
    return importlib.import_module(name)


def reference_flashinfer_varblock(q, k, v, block_mask_map, block_row_sz, block_col_sz):
    """The reference's live SVG2 attention call, svg.kmeans_utils.dynamic_block_sparse_fwd_flashinfer(..., is_cpu=False)
    (svg/kmeans_utils.py:1319-1392).

    The reference pins FlashInfer 0.2.10 + assets/patches/modifications.patch and resets two PRIVATE wrapper buffers
    (`_vector_sparse_indices_buffer` / `_vector_sparse_indptr_buffer`, :1361-1366) that FlashInfer 0.6.x (this image)
    no longer has, so the unmodified function raises AttributeError here.  In that case the same public-API sequence
    is run without that one call: 512 MB float workspace, VariableBlockSparseAttentionWrapper(backend="auto"),
    plan(block_mask_map, block_row_sz, block_col_sz, ...), run(q, k, v) — allocation, plan and run per call exactly
    as the reference does every attention call.  Returns (o [B,H,S,D], how)."""
    ku = import_kmeans_utils()
    try:
        return ku.dynamic_block_sparse_fwd_flashinfer(q, k, v, block_mask_map, block_row_sz, block_col_sz,
                                                      is_cpu=False), "reference function, unmodified"
    except AttributeError:
        pass
    import flashinfer
    import torch

    B, H, S, D = q.shape
    qc_num, kc_num = block_row_sz.shape[-1], block_col_sz.shape[-1]
    float_workspace_buffer = torch.empty(128 * 1024 * 1024, device=q.device)
    wrapper = flashinfer.sparse.VariableBlockSparseAttentionWrapper(float_workspace_buffer, backend="auto")
    wrapper.plan(block_mask_map=block_mask_map.reshape(B * H, qc_num, kc_num),
                 block_row_sz=block_row_sz.reshape(B * H, qc_num), block_col_sz=block_col_sz.reshape(B * H, kc_num),
                 num_qo_heads=B * H, num_kv_heads=B * H, head_dim=D, q_data_type=q.dtype, kv_data_type=k.dtype)
    o = wrapper.run(q.reshape(B * H, S, D), k.reshape(B * H, S, D), v.reshape(B * H, S, D))
    return o.reshape(B, H, S, D), "reference call sequence on FlashInfer 0.6.x (private-buffer reset skipped)"
