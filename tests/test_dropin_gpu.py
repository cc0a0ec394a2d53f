"""The drop-in, proven against the REAL reference processors.

The unmodified reference is imported (tests/golden/ref_import.py: a checkout named by SVGB200_REFERENCE or the
git-ignored install baseline/_ref; `diffusers` / `cuvs` replaced by inert stubs),
`svgb200.patch.install(module)` swaps the operator names the reference resolves as module globals, and the
reference's OWN `attention_core_logic` runs on the GPU:

  svg/models/hyvideo/attention.py:473-524   Hunyuan_SVGAttn_Processor2_0      (SVG1)
  svg/models/hyvideo/attention.py:714-804   Hunyuan_SAPAttn_Processor2_0      (SVG2, prompt / padding blocks, dense varlen)
  svg/models/wan/attention.py:284-328,499-559   WanAttn_SVGAttn_Processor2_0 / WanAttn_SAPAttn_Processor
  svg/models/cog/attention.py:164-196       CogVideoX_SparseAttn_Processor2_0

Its output is compared with the CPU oracle.  The signature test (no GPU needed) fails when a reference call site and
a mirrored operator drift apart.  Everything here is skipped when the reference is not importable."""
import inspect
import sys
from pathlib import Path

import pytest
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE / "golden"))
import ref_import as R  # noqa: E402
from gen_inputs import structured_qkv  # noqa: E402

needs_ref = pytest.mark.skipif(not R.reference_available(), reason="reference not importable (no SVGB200_REFERENCE, no baseline/_ref)")


def _positional(fn):
    return [p.name for p in inspect.signature(fn).parameters.values()
            if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]


@needs_ref
def test_mirrored_operator_signatures_match_reference():
    """Every name patch.install() replaces must accept the reference's positional arguments in the same order."""
    from svgb200 import patch

    ku = R.import_kmeans_utils()
    perm = __import__("importlib").import_module("svg.kernels.triton.permute")
    places = {m: R.import_placement(m) for m in ("hyvideo", "wan", "cosmos", "cog")}
    checked = 0
    for name, mine in patch._NAMES.items():
        ref = None
        for mod in (ku, perm, *places.values()):
            if hasattr(mod, name):
                ref = getattr(mod, name)
                break
        assert ref is not None, f"{name}: not found in the reference"
        ref_fn = inspect.unwrap(ref)
        a, b = _positional(ref_fn), _positional(mine)
        assert b[: len(a)] == a, (name, a, b)  # same leading positional names; ours may add optional trailing ones
        checked += 1
    assert checked == len(patch._NAMES)
    for model, cls_name in (("hyvideo", "Hunyuan_SVGAttn_Processor2_0"), ("wan", "WanAttn_SVGAttn_Processor2_0"),
                            ("cog", "CogVideoX_SparseAttn_Processor2_0")):
        A = R.import_model_module(model, "attention")
        ours = {"hyvideo": "hyvideo", "wan": "wan", "cog": "cog"}[model]
        mine = getattr(__import__(f"svgb200.models.{ours}", fromlist=["x"]), "prepare_flexattention")
        a = _positional(A.prepare_flexattention)
        assert _positional(mine)[: len(a)] == a, model  # trailing extras of ours must be optional
        assert hasattr(getattr(A, cls_name), "attention_core_logic")
    hy = R.import_model_module("hyvideo", "attention")
    assert _positional(patch.flashinfer_varlen_func) == _positional(hy.flashinfer_varlen_func)


# -------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _redraw_rows(seed, high, n):
    torch.manual_seed(seed)
    return torch.randint(low=0, high=high, size=(n,))


def _svg1_oracle(q, k, v, rows, layout, ctx, plen, F, P, sparsity, text_first=False):
    from oracle import attention as oa
    from oracle import layout as ol

    if layout == "cog":
        masks = [oa.profiling_mask_rows_cog(mn, rows, ctx, F, P) for mn in ("spatial", "temporal")]
    else:
        masks = [oa.profiling_mask_rows(mn, rows, layout, ctx, F, P) for mn in ("spatial", "temporal")]
    mses = oa.sample_mse(q, k, v, rows, masks)
    best = torch.argmin(mses.bfloat16(), dim=0).view(-1)
    mul = oa.sparsity_to_width(sparsity, ctx, F, P)
    mod = {"hy": lambda: oa.hy_mask_mod(ctx, plen, F, P, mul), "wan": lambda: oa.wan_mask_mod(F, P, mul),
           "cog": lambda: oa.cog_mask_mod(ctx, F, P, mul)}[layout]()
    qp, kp, vp = (ol.head_placement(t[0], best.numpy(), ctx, F, P, text_first=text_first) for t in (q, k, v))
    ref = ol.head_placement(oa.masked_attention_bhsd(qp, kp, vp, mod).bfloat16(), best.numpy(), ctx, F, P,
                            text_first=text_first, inverse=True)
    return ref.float(), mses, best


@gpu
@needs_ref
@pytest.mark.parametrize("own_sample_mse", [True, False])
def test_hunyuan_svg1_processor_runs_on_svgb200(cuda, own_sample_mse):
    """Hunyuan_SVGAttn_Processor2_0.attention_core_logic (hyvideo/attention.py:473-524) with svgb200 installed.
    own_sample_mse=False keeps the REFERENCE's eager sample_mse on its materialised profiling masks, so the test also
    checks our analytic masks against the reference's get_attention_mask on the GPU path."""
    from svgb200 import patch

    A = R.import_model_module("hyvideo", "attention")
    U = R.import_model_module("hyvideo", "utils")
    ref_smse = vars(A.Hunyuan_SVGAttn_Processor2_0).get("_ref_sample_mse") or A.Hunyuan_SVGAttn_Processor2_0.sample_mse
    A.Hunyuan_SVGAttn_Processor2_0._ref_sample_mse = ref_smse
    done = patch.install(A)
    assert {"hunyuan_sparse_head_placement", "flex_attention", "prepare_flexattention"} <= set(done)
    cls = A.Hunyuan_SVGAttn_Processor2_0
    if not own_sample_mse:
        cls.sample_mse = ref_smse
    H, F, P, ctx, plen, D, sparsity = 3, 4, 200, 48, 20, 128, 0.4
    S = ctx + F * P
    cls.context_length, cls.prompt_length, cls.num_frame, cls.frame_size = ctx, plen, F, P
    cls.num_sampled_rows, cls.sample_mse_max_row = 24, 500
    cls.first_layers_fp, cls.first_times_fp = 0, 900
    if not own_sample_mse:
        cls.attention_masks = [U.get_attention_mask(n, 500, ctx, F, P, device="cpu") for n in ("spatial", "temporal")]
    w = U.sparsity_to_width(sparsity, ctx, F, P)
    cls.block_mask = A.prepare_flexattention(1, H, D, torch.bfloat16, cuda, ctx, plen, F, P, diag_width=w, multiplier=w)
    q, k, v = structured_qkv(0, H, F, P, ctx, D)  # heads with a clear spatial / temporal preference
    proc = cls(layer_idx=0)
    cu = torch.tensor([0, F * P + plen, S], dtype=torch.int32, device=cuda)
    torch.manual_seed(123)
    o = proc.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([100.0]), 0, (cu, cu, S, S))
    rows = _redraw_rows(123, 500, 24)
    ref, _, _ = _svg1_oracle(q, k, v, rows, "hy", ctx, plen, F, P, sparsity)
    torch.testing.assert_close(o.float().cpu()[0], ref, rtol=3e-2, atol=2e-2)
    # dense branch of the same processor: flash_attn_varlen_func call site (:452-470) -> our dense varlen plan
    od = proc.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([950.0]), 0, (cu, cu, S, S))
    from oracle import attention as oa

    seg_mask = lambda qi, ki: ((qi < F * P + plen) & (ki < F * P + plen)) | ((qi >= F * P + plen) & (ki >= F * P + plen))  # noqa: E731
    torch.testing.assert_close(od.float().cpu()[0], oa.masked_attention_bhsd(q[0], k[0], v[0], seg_mask), rtol=3e-2, atol=2e-2)


class _Spy:
    def __init__(self, fn):
        self.fn, self.calls = fn, []

    def __call__(self, *a, **k):
        r = self.fn(*a, **k)
        self.calls.append((a, k, r))
        return r


def _sap_oracle_check(o, q, k, v, spies, S, V, ctx, plen):
    """masked attention under the element mask implied by the integers the patched operators produced."""
    H, D = q.shape[1], q.shape[-1]
    dyn = spies["identify_dynamic_map"].calls[-1][2][0].cpu()           # [H, QC, KC]
    km = spies["batch_kmeans_Euclid"].calls
    (ql, _, qs, _), (kl, _, ks, _) = km[-2][2], km[-1][2]
    ql, kl, qs, ks = ql.cpu(), kl.cpu(), qs.cpu(), ks.cpu()
    assert int(qs.sum(1)[0]) == V and int(ks.sum(1)[0]) == V
    for h in range(H):
        allowed = torch.zeros(S, S, dtype=torch.bool)
        allowed[:V, :V] = dyn[h][ql[h]][:, kl[h]]
        if ctx:
            R_ = V + plen
            allowed[:R_, V:R_] = True      # prompt columns for every real row   (hyvideo/attention.py:681-684)
            allowed[V:R_, :R_] = True      # prompt rows see everything real
            allowed[R_:, R_:] = True       # padding attends padding only
        s = (q[0, h].float() @ k[0, h].float().T) * D ** -0.5
        w = torch.nan_to_num(torch.softmax(s.masked_fill(~allowed, float("-inf")), -1), nan=0.0)
        torch.testing.assert_close(o[0, h], w @ v[0, h].float(), rtol=3e-2, atol=2e-2)


@gpu
@needs_ref
def test_hunyuan_sap_processor_runs_on_svgb200(cuda):
    """Hunyuan_SAPAttn_Processor2_0.attention_core_logic (hyvideo/attention.py:714-804): reference control flow
    (prepare_video_part, kmeans state machine, dynamic_map_post_processing, logging) + svgb200 operators."""
    import json
    import tempfile

    from svgb200 import patch

    A = R.import_model_module("hyvideo", "attention")
    patch.install(A)
    spies = {n: _Spy(getattr(A, n)) for n in ("identify_dynamic_map", "batch_kmeans_Euclid")}
    for n, s in spies.items():
        setattr(A, n, s)
    cls = A.Hunyuan_SAPAttn_Processor2_0
    H, F, P, ctx, plen, D = 2, 4, 256, 64, 20, 128
    V, S = F * P, ctx + F * P
    cls.context_length, cls.prompt_length, cls.num_frame, cls.frame_size = ctx, plen, F, P
    cls.num_q_centroids, cls.num_k_centroids, cls.top_p_kmeans, cls.min_kc_ratio = 8, 16, 0.9, 0.1
    cls.kmeans_iter_init, cls.kmeans_iter_step, cls.zero_step_kmeans_init = 3, 1, True
    cls.first_layers_fp, cls.first_times_fp = 0, 900
    cls.centroids_init, cls.q_centroids, cls.k_centroids = {}, {}, {}
    log = tempfile.NamedTemporaryFile(suffix=".jsonl", delete=False).name
    cls.logging_file = log
    g = torch.Generator().manual_seed(1)
    q, k, v = (torch.randn(1, H, S, D, generator=g).to(torch.bfloat16) for _ in range(3))
    proc = cls(layer_idx=0)
    cu = torch.tensor([0, V + plen, S], dtype=torch.int32, device=cuda)
    cu_max = (cu, cu, S, S)
    # dense step first: zero_step_kmeans_init warms the centroids up (:739-743), attention through flashinfer_varlen_func
    od = proc.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([950.0]), 0, cu_max)
    from oracle import attention as oa

    seg_mask = lambda qi, ki: ((qi < V + plen) & (ki < V + plen)) | ((qi >= V + plen) & (ki >= V + plen))  # noqa: E731
    torch.testing.assert_close(od.float().cpu()[0], oa.masked_attention_bhsd(q[0], k[0], v[0], seg_mask), rtol=3e-2, atol=2e-2)
    assert cls.centroids_init.get(0) is True and len(spies["batch_kmeans_Euclid"].calls) == 2
    # sparse steps: warm-started k-means (kmeans_step), reference post-processing, our kernels
    for step in range(2):
        o = proc.attention_core_logic(q.to(cuda).clone(), k.to(cuda).clone(), v.to(cuda).clone(), torch.tensor([100.0]), 0,
                                      cu_max).float().cpu()
        assert spies["batch_kmeans_Euclid"].calls[-1][1].get("init_centroids") is not None
        _sap_oracle_check(o, q, k, v, spies, S, V, ctx, plen)
    lines = [json.loads(x) for x in open(log)]
    assert len(lines) == 2 and set(lines[0]) == {"timestep", "layer", "avg_density", "density"}
    assert len(lines[0]["density"][0]) == H and 0 < lines[0]["avg_density"] <= 1
    cls.logging_file = None


@gpu
@needs_ref
def test_wan_processors_run_on_svgb200(cuda):
    """WanAttn_SAPAttn_Processor / WanAttn_SVGAttn_Processor2_0 (wan/attention.py:499-559, 284-328)."""
    from svgb200 import patch

    A = R.import_model_module("wan", "attention")
    U = R.import_model_module("wan", "utils")
    patch.install(A)
    spies = {n: _Spy(getattr(A, n)) for n in ("identify_dynamic_map", "batch_kmeans_Euclid")}
    for n, s in spies.items():
        setattr(A, n, s)
    H, F, P, D = 3, 4, 300, 128
    S = F * P
    g = torch.Generator().manual_seed(2)
    q, k, v = (torch.randn(1, H, S, D, generator=g).to(torch.bfloat16) for _ in range(3))
    # SVG2
    cls = A.WanAttn_SAPAttn_Processor
    cls.context_length, cls.num_frame, cls.frame_size = 0, F, P
    cls.num_q_centroids, cls.num_k_centroids, cls.top_p_kmeans, cls.min_kc_ratio = 6, 20, 0.8, 0.1
    cls.kmeans_iter_init, cls.kmeans_iter_step = 4, 1
    cls.first_layers_fp, cls.first_times_fp = 0, 900
    proc = cls(layer_idx=0)
    for step in range(2):
        o = proc.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([100.0])).float().cpu()
        _sap_oracle_check(o, q, k, v, spies, S, S, 0, 0)
    assert proc.centroids_init is True
    # SVG1
    cls1 = A.WanAttn_SVGAttn_Processor2_0
    sparsity = 0.4
    cls1.context_length, cls1.num_frame, cls1.frame_size = 0, F, P
    cls1.num_sampled_rows, cls1.sample_mse_max_row = 24, 600
    w = U.sparsity_to_width(sparsity, 0, F, P)
    cls1.block_mask = A.prepare_flexattention(1, H, D, torch.bfloat16, cuda, 0, 0, F, P, diag_width=w, multiplier=w)
    p1 = cls1(layer_idx=0)
    q, k, v = structured_qkv(2, H, F, P, 0, D)
    torch.manual_seed(77)
    o1 = p1.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([100.0])).float().cpu()
    rows = _redraw_rows(77, 600, 24)
    ref, _, _ = _svg1_oracle(q, k, v, rows, "wan", 0, 0, F, P, sparsity)
    torch.testing.assert_close(o1[0], ref, rtol=3e-2, atol=2e-2)


@gpu
@needs_ref
def test_cog_processor_runs_on_svgb200(cuda):
    """CogVideoX_SparseAttn_Processor2_0.attention_core_logic (cog/attention.py:164-196), text first."""
    from svgb200 import patch

    A = R.import_model_module("cog", "attention")
    U = R.import_model_module("cog", "utils")
    done = patch.install(A)
    assert {"sparse_head_placement", "hidden_states_placement", "flex_attention", "prepare_flexattention"} <= set(done)
    cls = A.CogVideoX_SparseAttn_Processor2_0
    H, F, P, ctx, D, sparsity = 3, 5, 200, 34, 64, 0.45
    S = ctx + F * P
    cls.context_length, cls.num_frame, cls.frame_size = ctx, F, P
    cls.num_sampled_rows, cls.first_layers_fp, cls.first_times_fp = 24, 0, 0.0
    w = U.sparsity_to_width(sparsity, ctx, F, P)
    cls.block_mask = A.prepare_flexattention(1, H, D, torch.bfloat16, cuda, ctx, F, P, diag_width=w, multiplier=w)
    q, k, v = structured_qkv(3, H, F, P, ctx, D, text_first=True)
    proc = cls(layer_idx=5)
    for seed in (5, 6, 7):
        torch.manual_seed(seed)
        o = proc.attention_core_logic(q.to(cuda), k.to(cuda), v.to(cuda), torch.tensor([500.0])).float().cpu()
        rows = _redraw_rows(seed, S, 24)
        ref, mses, best = _svg1_oracle(q, k, v, rows, "cog", ctx, 0, F, P, sparsity, text_first=True)
        if bool((rows < ctx).any()):
            assert (best == 1).all()
        torch.testing.assert_close(o[0], ref, rtol=3e-2, atol=2e-2)
