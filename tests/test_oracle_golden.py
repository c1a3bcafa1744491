"""CPU: the oracle restatement against the committed reference outputs (tests/golden/*.npz, written by
oracle/make_golden.py from the UNMODIFIED reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import rules
from oracle import cpu as ocpu
from oracle import vit as ovit


def T(a):
    return torch.from_numpy(np.asarray(a))


def test_rules_match_reference_layer_classes(golden_dir):
    g = np.load(os.path.join(golden_dir, "rules.npz"))
    # bit-exact: the closed forms are the same fp32 operations in the same order
    assert torch.equal(rules.linear_relprop(T(g["lin_x"]), T(g["lin_w"]), T(g["lin_r"])), T(g["lin_out"]))
    oa, ob = rules.add_relprop(T(g["add_a"]), T(g["add_b"]), T(g["add_r"]))
    assert torch.equal(oa, T(g["add_oa"])) and torch.equal(ob, T(g["add_ob"]))
    assert torch.equal(rules.clone_relprop(T(g["clone_x"]), (T(g["clone_r1"]), T(g["clone_r2"]))), T(g["clone_out"]))
    op, ov = rules.matmul_av_relprop(T(g["av_p"]), T(g["av_v"]), T(g["av_r"]))
    assert torch.equal(op, T(g["av_op"])) and torch.equal(ov, T(g["av_ov"]))
    oq, ok = rules.matmul_qk_relprop(T(g["qk_q"]), T(g["qk_k"]), T(g["qk_r"]))
    assert torch.equal(oq, T(g["qk_oq"])) and torch.equal(ok, T(g["qk_ok"]))
    assert torch.equal(rules.index_select_relprop(T(g["isel_x"]), T(g["isel_r"])), T(g["isel_out"]))
    assert torch.equal(rules.safe_divide(T(g["sd_a"]), T(g["sd_b"])), T(g["sd_out"]))


def _tiny_params(g, dtype):
    return {k[len("param."):]: T(g[k]).to(dtype) for k in g.files if k.startswith("param.")}


@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("f64", torch.float64)])
def test_vit_tiny_matches_reference(golden_dir, tag, dtype):
    g = np.load(os.path.join(golden_dir, "vit_tiny.npz"))
    params = _tiny_params(g, dtype)
    heads = int(g["heads"])
    x = T(g["x"]).to(dtype)
    for s in range(x.shape[0]):
        for sl in (0, 1):
            out, idx, taps = ovit.explain(params, x[s:s + 1], heads, start_layer=sl, return_taps=True)
            ref = T(g["%s.s%d.map.sl%d" % (tag, s, sl)])
            assert torch.equal(out, ref), "map differs from the reference (sample %d start_layer %d)" % (s, sl)
        assert torch.equal(taps["logits"], T(g["%s.s%d.logits" % (tag, s)]))
        out0, _, taps = ovit.explain(params, x[s:s + 1], heads, start_layer=0, return_taps=True)
        for l in range(3):
            assert torch.equal(taps["grads"][l], T(g["%s.s%d.grad.%d" % (tag, s, l)]))
            assert torch.equal(taps["cams"][l], T(g["%s.s%d.cam.%d" % (tag, s, l)]))
    out, idx = ovit.explain(params, x[0:1], heads, index=3)
    assert torch.equal(out, T(g["%s.s0.map.index3" % tag]))


@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("f64", torch.float64)])
def test_vit_tiny_other_methods_match_reference(golden_dir, tag, dtype):
    """Every other ``method`` branch of VisionTransformer.relprop (rollout, full, last_layer, ...), incl. the
    first-layer z^B rule, is bit-equal to the unmodified reference."""
    g = np.load(os.path.join(golden_dir, "vit_tiny_methods.npz"))
    params, heads = ovit.init_params("vit_tiny_test", seed=int(g["param_seed"]), rand_affine=True)
    params = {k: v.to(dtype) for k, v in params.items()}
    x = T(g["x"]).to(dtype)
    for s in range(x.shape[0]):
        for key in [k for k in g.files if k.startswith("%s.s%d." % (tag, s))]:
            method, suffix = key.split(".")[2:4]
            kw = {"is_ablation": True} if suffix == "ablation" else {"start_layer": int(suffix[2:])}
            out, _ = ovit.explain_method(params, x[s:s + 1], heads, method, **kw)
            ref = T(g[key]).reshape(out.shape)
            assert torch.equal(out, ref), key
    # a batch is a set of independent B=1 explanations for these branches as well
    out, _ = ovit.explain_method(params, x, heads, "full")
    for s in range(x.shape[0]):
        one, _ = ovit.explain_method(params, x[s:s + 1], heads, "full")
        assert torch.allclose(out[s], one[0], rtol=1e-4 if dtype == torch.float32 else 1e-10, atol=0)


def test_vit_tiny_batched_equals_per_sample(golden_dir):
    """A batch is a set of independent B=1 explanations (per-sample reductions)."""
    g = np.load(os.path.join(golden_dir, "vit_tiny.npz"))
    params = _tiny_params(g, torch.float64)
    x = T(g["x"]).double()
    both, _ = ovit.explain(params, x, int(g["heads"]))
    for s in range(x.shape[0]):
        one, _ = ovit.explain(params, x[s:s + 1], int(g["heads"]))
        assert torch.allclose(both[s:s + 1], one, rtol=1e-9, atol=1e-15)


def test_vit_base_matches_reference(golden_dir):
    """ViT-B/16: oracle (fp32) on regenerated weights/inputs vs the stored reference maps.  The weights are
    regenerated from a seed; the stored checksums guard against RNG drift between machines."""
    g = np.load(os.path.join(golden_dir, "vit_base.npz"))
    params, heads = ovit.init_params("vit_base_patch16_224", seed=int(g["param_seed"]))
    wsum = sum(v.double().sum().item() for v in params.values())
    xs = torch.randn(int(g["n"]), 3, 224, 224, generator=torch.Generator().manual_seed(int(g["x_seed"])))
    if abs(wsum - float(g["w_checksum"])) > 1e-6 * abs(float(g["w_checksum"])) or \
            not np.allclose(xs.double().sum(dim=(1, 2, 3)).numpy(), g["x_checksum"], rtol=1e-9):
        pytest.skip("seeded weights/inputs do not reproduce on this machine")
    ocpu.set_torch_threads()
    s = 1                                   # one sample keeps the CPU suite short
    out, idx = ovit.explain(params, xs[s:s + 1], heads)
    assert int(idx) == int(g["f32.index"][s]) == int(g["f64.index"][s])
    ref32, ref64 = g["f32.maps"][s], g["f64.maps"][s]
    # same fp32 formulas; thread count / BLAS blocking may differ from the generating run, so compare at the
    # reference's own fp32-vs-fp64 noise level (SURVEY.md §8c) rather than bit-exactly
    noise = np.abs(ref32 - ref64).max()
    assert np.abs(out[0].numpy() - ref64).max() <= max(1e-4, 50 * noise)
    assert np.abs(out[0].numpy() - ref32).max() <= 1e-4


def test_oracle_bit_equal_to_live_reference(golden_dir):
    """Map and per-block taps bit-equal to those the reference computed live on the tiny model under a second weight
    seed (``vit_tiny_seed9.npz``)."""
    g = np.load(os.path.join(golden_dir, "vit_tiny_seed9.npz"))
    params, heads = ovit.init_params("vit_tiny_test", seed=int(g["param_seed"]), rand_affine=True)
    out, idx, taps = ovit.explain(params, T(g["x"]), heads, return_taps=True)
    assert torch.equal(out, T(g["map"]))
    for l in range(3):
        assert torch.equal(taps["cams"][l], T(g["cam.%d" % l]))
        assert torch.equal(taps["grads"][l], T(g["grad.%d" % l]))


@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("f64", torch.float64)])
def test_bert_tiny_matches_reference(golden_dir, tag, dtype):
    """BERT oracle vs the reference's Generator.generate_LRP (incl. a padded sequence: -10000 mask path)."""
    from oracle import bert as obert
    g = np.load(os.path.join(golden_dir, "bert_tiny.npz"))
    params = {k[len("param."):]: T(g[k]).to(dtype) for k in g.files if k.startswith("param.")}
    heads = int(g["heads"])
    ids, mask = T(g["ids"]), T(g["mask"])
    for s in range(2):
        for sl in (0, 1, 2):
            out, idx, taps = obert.explain(params, ids[s:s + 1], mask[s:s + 1], heads, start_layer=sl, return_taps=True)
            assert torch.equal(out, T(g["%s.s%d.map.sl%d" % (tag, s, sl)]))
            if sl == 0:
                assert torch.equal(taps["logits"], T(g["%s.s%d.logits" % (tag, s)]))
                for l in range(3):
                    assert torch.equal(taps["grads"][l], T(g["%s.s%d.grad.%d" % (tag, s, l)]))
                    assert torch.equal(taps["cams"][l], T(g["%s.s%d.cam.%d" % (tag, s, l)]))
    out, _ = obert.explain(params, ids[0:1], mask[0:1], heads, index=0, start_layer=0)
    assert torch.equal(out, T(g["%s.s0.map.index0" % tag]))
    # padded tokens receive exactly zero relevance (SURVEY.md §8c invariant)
    out, _ = obert.explain(params, ids[1:2], mask[1:2], heads, start_layer=0)
    assert float(out[0, 18:].abs().max()) == 0.0


def _same(a, b):
    """bit-equal including the NaN pattern (an all-zero GradCAM map min-max-normalises to NaN in the reference too)."""
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(nan=0.), b.nan_to_num(nan=0.))


def test_vit_baselines_match_reference(golden_dir):
    """Baselines.generate_rollout / generate_cam_attn (ViT_explanation_generator.py:45-83) on the ViT_new model."""
    g = np.load(os.path.join(golden_dir, "vit_baselines.npz"))
    params, heads = ovit.init_params("vit_tiny_test", seed=int(g["param_seed"]), rand_affine=True, img=112)
    x = T(g["x"])
    eps = float(g["norm_eps"])
    for s in range(x.shape[0]):
        for sl in (0, 1):
            out = ovit.baseline_rollout(params, x[s:s + 1], heads, start_layer=sl, norm_eps=eps)
            assert torch.equal(out, T(g["f32.s%d.rollout.sl%d" % (s, sl)]))
        for tag, idx in (("argmax", None), ("index3", 3), ("index7", 7)):
            out, _ = ovit.baseline_cam_attn(params, x[s:s + 1], heads, index=idx, norm_eps=eps)
            assert _same(out[0], T(g["f32.s%d.cam_attn.%s" % (s, tag)])), (s, tag)


def test_bert_generators_match_reference(golden_dir):
    """generate_LRP_last_layer / full_lrp / attn_last_layer / rollout / attn_gradcam (ExplanationGenerator.py:61-155)."""
    from oracle import bert as obert
    g = np.load(os.path.join(golden_dir, "bert_generators.npz"))
    params, heads = obert.init_params(seed=int(g["param_seed"]), vocab=100, max_pos=32, dim=64, depth=3, heads=4,
                                      inter=128, rand_affine=True)
    ids, mask = T(g["ids"]), T(g["mask"])
    seen = 0
    for key in [k for k in g.files if k.startswith("f32.")]:
        _, s, which, tag = key.split(".")
        s = int(s[1:])
        kw = {"start_layer": int(tag[2:])} if tag.startswith("sl") else ({} if tag == "argmax" else {"index": int(tag[5:])})
        out = obert.generate(params, ids[s:s + 1], mask[s:s + 1], heads, which, **kw)
        assert _same(out, T(g[key])), key
        seen += 1
    assert seen == 28


@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("f64", torch.float64)])
def test_vit_orig_lrp_variant_matches_reference(golden_dir, tag, dtype):
    """The ``layers_lrp`` rule library (``modules/layers_lrp.py``: Linear with separate denominators, Add without ratio
    normalisation) behind ``baselines/ViT/ViT_orig_LRP.py``: oracle (``variant="lrp"``) bit-equal to the stored outputs
    of the UNMODIFIED reference for method = grad / full / last_layer / rollout."""
    g = np.load(os.path.join(golden_dir, "vit_orig_lrp.npz"))
    params, heads = ovit.init_params("vit_tiny_test", seed=int(g["param_seed"]), rand_affine=True)
    p = {k: v.to(dtype) for k, v in params.items()}
    xs = T(g["x"]).to(dtype)
    keys = [k for k in g.files if k.startswith(tag + ".")]
    assert len(keys) == 12
    for key in keys:
        s, method, sl = int(key.split(".")[1][1:]), key.split(".")[2], int(key.split(".")[3][2:])
        out, _ = ovit.explain_method(p, xs[s:s + 1], heads, method, start_layer=sl, variant="lrp")
        assert torch.equal(out, T(g[key]).reshape(out.shape)), key
    # the two rules on their own, against closed forms written out independently here
    x, w, r = torch.randn(5, 7, dtype=dtype), torch.randn(4, 7, dtype=dtype), torch.rand(5, 4, dtype=dtype)
    z1, z2 = x.clamp(min=0) @ w.clamp(min=0).t(), x.clamp(max=0) @ w.clamp(max=0).t()
    want = x.clamp(min=0) * (rules.safe_divide(r, z1) @ w.clamp(min=0)) + x.clamp(max=0) * (rules.safe_divide(r, z2) @ w.clamp(max=0))
    assert torch.equal(rules.linear_relprop_lrp(x, w, r), want)
    a, b = rules.add_relprop_simple(x, 2 * x + 1, x)
    assert torch.allclose(a + b, x * ((3 * x + 1) != 0))                  # conservation without any re-normalisation
