"""Import and run the UNMODIFIED reference on CPU (TEST INFRASTRUCTURE, authoring container only).

``/root/reference`` does not exist on the GPU box; there the harness imports the
byte-for-byte mirror of the hot-path files that ``oracle/fetch_ref.py`` leaves in
``oracle/_ref`` (git-ignored).  It is used by ``oracle/make_golden.py`` (fixture
generation) and by ``bench.py``'s ``cpu_baseline`` leg / ``--impl reference`` arm.

Shims (SURVEY.md §8c) — each one works around an incompatibility of the
reference with this container, none changes the arithmetic:
 1. ``sys.path.insert(0, REF)`` so ``modules.*`` / ``baselines.*`` import.
 2. the hard-coded ``.cuda()`` on the one-hot (``ViT_explanation_generator.py:35``,
    ``ExplanationGenerator.py:40``) is neutralised when no GPU is present.
 BERT additionally:
 3. stub ``gensim`` (imported at ``BERT_rationale_benchmark/models/model_utils.py:5``).
 4. ``BertPreTrainedModel.init_weights`` -> guarded ``post_init`` (transformers 5.x).
 5. ``get_extended_attention_mask`` -> transformers 3.5.1 arithmetic ``(1-mask)*-10000``.
 6. ``get_head_mask`` -> ``[None]*n``.
 7. ``BertConfig(return_dict=False)``.
"""
import contextlib
import os
import sys
import types

import torch

def _find_ref():
    """``/root/reference`` in the authoring container; on the GPU box the byte-for-byte mirror of the hot-path files
    that ``oracle/fetch_ref.py`` leaves in ``oracle/_ref`` (git-ignored, shipped with the snapshot)."""
    for c in (os.environ.get("TE_REFERENCE_PATH"), "/root/reference",
              os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")):
        if c and os.path.isdir(os.path.join(c, "baselines", "ViT")):
            return c
    return os.environ.get("TE_REFERENCE_PATH", "/root/reference")


REF = _find_ref()


def available():
    return os.path.isdir(os.path.join(REF, "baselines", "ViT"))


def is_mirror():
    return os.path.basename(REF.rstrip("/")) == "_ref"


@contextlib.contextmanager
def _cpu_cuda_shim():
    """Make ``Tensor.cuda()`` a no-op while the reference runs: the harness always runs the reference ON THE HOST CORES
    (it is the CPU arm), also on a GPU box, where the hard-coded ``.cuda()`` on the one-hot
    (``ViT_explanation_generator.py:35``) would otherwise mix a CUDA tensor into a CPU model."""
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.Tensor.cuda = orig


_TOP = ("modules", "baselines", "BERT_explainability", "BERT_rationale_benchmark")
_REF_MODS = {}


def _is_ref_name(k):
    return any(k == t or k.startswith(t + ".") for t in _TOP)


@contextlib.contextmanager
def _ref_imports():
    """Import the reference's top-level packages (``modules``, ``baselines`` ...) even when the product's
    ``install_aliases()`` has registered its own modules under the same names: swap sys.modules entries in,
    run, swap back."""
    if not available():
        raise RuntimeError("reference not present at %s" % REF)
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if _is_ref_name(k)}
    sys.modules.update(_REF_MODS)
    sys.path.insert(0, REF)
    try:
        yield
    finally:
        sys.path.remove(REF)
        for k in list(sys.modules):
            if _is_ref_name(k):
                _REF_MODS[k] = sys.modules.pop(k)
        sys.modules.update(saved)


def _ensure_path():
    if not available():
        raise RuntimeError("reference not present at %s" % REF)


def vit_module():
    with _ref_imports():
        import baselines.ViT.ViT_LRP as m          # noqa: E402  (the reference's own module)
    return m


def build_vit(name="vit_base_patch16_224", seed=0, dtype=torch.float32, state_dict=None, **kwargs):
    """Reference model, its own constructor init under ``torch.manual_seed(seed)``
    (or a supplied state_dict), eval mode."""
    m = vit_module()
    torch.manual_seed(seed)
    if name == "custom":
        model = m.VisionTransformer(**kwargs)
    else:
        model = getattr(m, name)(pretrained=False, **kwargs)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    return model.to(dtype).eval()


def build_vit_orig_lrp(state_dict=None, dtype=torch.float32, **kwargs):
    """The reference's ``layers_lrp`` baseline model (``baselines/ViT/ViT_orig_LRP.py``: same architecture as ``ViT_LRP``
    on the rule library of ``modules/layers_lrp.py``)."""
    _ensure_path()
    with _ref_imports():
        import baselines.ViT.ViT_orig_LRP as m
    model = m.VisionTransformer(**kwargs)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    return model.to(dtype).eval()


def vit_generate_lrp(model, x, index=None, start_layer=0, method="transformer_attribution", taps=False):
    """``LRP(model).generate_LRP`` of the reference, B=1, on CPU.  Returns a dict."""
    with _ref_imports():
        from baselines.ViT.ViT_explanation_generator import LRP
    assert x.shape[0] == 1, "the reference path is only correct at B=1 (SURVEY.md §0-6)"
    with _cpu_cuda_shim():
        if x.dtype == torch.float64:
            out = _generate_lrp_any_dtype(model, x, index, start_layer, method)
        else:
            out = LRP(model).generate_LRP(x, index=index, method=method, start_layer=start_layer)
    res = {"map": out.detach()}
    if taps:
        res["grads"] = [b.attn.get_attn_gradients().detach() for b in model.blocks]
        res["cams"] = [b.attn.get_attn_cam().detach() for b in model.blocks]
        res["attn"] = [b.attn.get_attn().detach() for b in model.blocks]
    return res


def _generate_lrp_any_dtype(model, x, index, start_layer, method, is_ablation=False):
    """``generate_LRP`` (``ViT_explanation_generator.py:25-41``) with the one-hot built in the
    model's dtype — the reference hard-codes float32 numpy there, which cannot multiply an
    fp64 output.  Every model/relprop call is still the reference's own code."""
    import numpy as np
    output = model(x)
    if index is None:
        index = np.argmax(output.cpu().data.numpy(), axis=-1)
    one_hot = np.zeros((1, output.size()[-1]), dtype=np.float64)
    one_hot[0, index] = 1
    oh = torch.from_numpy(one_hot).to(x.dtype)
    loss = torch.sum(oh * output)
    model.zero_grad()
    loss.backward(retain_graph=True)
    return model.relprop(oh.clone(), method=method, is_ablation=is_ablation, start_layer=start_layer, alpha=1)


def build_vit_new(name="vit_base_patch16_224", state_dict=None, dtype=torch.float32, **kwargs):
    """The hook-free reference ViT (``baselines/ViT/ViT_new.py``) that ``Baselines`` explains."""
    _ensure_path()
    with _ref_imports():
        import baselines.ViT.ViT_new as m
    if name == "custom":
        model = m.VisionTransformer(**kwargs)
    else:
        model = getattr(m, name)(pretrained=False, **kwargs)
    if state_dict is not None:
        model.load_state_dict(state_dict)
    return model.to(dtype).eval()


def vit_baselines(model, x, which, **kw):
    """``Baselines(model).generate_cam_attn / generate_rollout`` (``ViT_explanation_generator.py:45-83``), B=1, CPU."""
    with _ref_imports():
        from baselines.ViT.ViT_explanation_generator import Baselines
    assert x.shape[0] == 1
    with _cpu_cuda_shim():
        out = getattr(Baselines(model), "generate_" + which)(x, **kw)
    return out.detach()


def bert_generate(model, input_ids, attention_mask, which, **kw):
    """The comparison generators of the reference ``Generator`` (``ExplanationGenerator.py:61-155``), B=1, CPU, fp32."""
    _prepare_bert_imports()
    assert input_ids.shape[0] == 1
    with _ref_imports():
        from BERT_explainability.modules.BERT.ExplanationGenerator import Generator
        with _cpu_cuda_shim():
            out = getattr(Generator(model), "generate_" + which)(input_ids, attention_mask, **kw)
    return out.detach()


def vit_logits(model, x):
    with torch.enable_grad():
        return model(x).detach()


# ----------------------------------------------------------------------------------------------
# BERT
# ----------------------------------------------------------------------------------------------
_BERT_READY = False


def _prepare_bert_imports():
    global _BERT_READY
    if _BERT_READY:
        return
    _ensure_path()
    if "gensim" not in sys.modules:                                   # shim 3
        g = types.ModuleType("gensim")
        gm = types.ModuleType("gensim.models")
        gm.KeyedVectors = type("KeyedVectors", (), {})
        g.models = gm
        sys.modules["gensim"] = g
        sys.modules["gensim.models"] = gm
    import transformers
    from transformers import BertPreTrainedModel

    def init_weights(self):                                           # shim 4
        if getattr(self, "_te_in_init", False):
            return
        self._te_in_init = True
        try:
            self.post_init()
        finally:
            self._te_in_init = False

    BertPreTrainedModel.init_weights = init_weights

    def get_extended_attention_mask(self, attention_mask, input_shape=None, device=None, *a, **k):  # shim 5
        return (1.0 - attention_mask[:, None, None, :].to(torch.get_default_dtype())) * -10000.0

    def get_head_mask(self, head_mask, num_hidden_layers, *a, **k):  # shim 6
        return [None] * num_hidden_layers

    BertPreTrainedModel.get_extended_attention_mask = get_extended_attention_mask
    BertPreTrainedModel.get_head_mask = get_head_mask
    _BERT_READY = True


def build_bert(seed=0, dtype=torch.float32, state_dict=None, **cfg_over):
    _prepare_bert_imports()
    from transformers import BertConfig
    with _ref_imports():          # transformers 5.x looks the model class's module up in sys.modules at construction
        from BERT_explainability.modules.BERT.BertForSequenceClassification import BertForSequenceClassification
        cfg = BertConfig(num_labels=2, return_dict=False, **cfg_over)     # shim 7
        torch.manual_seed(seed)
        model = BertForSequenceClassification(cfg)
        if state_dict is not None:
            model.load_state_dict(state_dict, strict=False)
        model = model.to(dtype).eval()
    return model


def bert_generate_lrp(model, input_ids, attention_mask, index=None, start_layer=11, taps=False):
    _prepare_bert_imports()
    assert input_ids.shape[0] == 1
    with _ref_imports():
        from BERT_explainability.modules.BERT.ExplanationGenerator import Generator
        with _cpu_cuda_shim():
            if next(model.parameters()).dtype == torch.float64:
                out = _bert_generate_lrp_any_dtype(Generator, model, input_ids, attention_mask, index, start_layer)
            else:
                out = Generator(model).generate_LRP(input_ids, attention_mask, index=index, start_layer=start_layer)
    res = {"map": out.detach()}
    if taps:
        layers = model.bert.encoder.layer
        res["grads"] = [l.attention.self.get_attn_gradients().detach() for l in layers]
        res["cams"] = [l.attention.self.get_attn_cam().detach() for l in layers]
        res["attn"] = [l.attention.self.get_attn().detach() for l in layers]
    return res


def _bert_generate_lrp_any_dtype(Generator, model, input_ids, attention_mask, index, start_layer):
    """``Generator.generate_LRP`` (``ExplanationGenerator.py:28-59``) with the one-hot built in the model dtype
    (the reference hard-codes float32 numpy); model / relprop / rollout calls are the reference's own code."""
    import numpy as np
    import sys as _sys
    mod = _sys.modules[Generator.__module__]
    output = model(input_ids=input_ids, attention_mask=attention_mask)[0]
    if index is None:
        index = np.argmax(output.cpu().data.numpy(), axis=-1)
    one_hot = np.zeros((1, output.size()[-1]), dtype=np.float64)
    one_hot[0, index] = 1
    oh = torch.from_numpy(one_hot).to(output.dtype)
    loss = torch.sum(oh * output)
    model.zero_grad()
    loss.backward(retain_graph=True)
    model.relprop(oh.clone(), alpha=1)
    cams = []
    for blk in model.bert.encoder.layer:
        grad = blk.attention.self.get_attn_gradients()
        cam = blk.attention.self.get_attn_cam()
        cam = cam[0].reshape(-1, cam.shape[-1], cam.shape[-1])
        grad = grad[0].reshape(-1, grad.shape[-1], grad.shape[-1])
        cam = (grad * cam).clamp(min=0).mean(dim=0)
        cams.append(cam.unsqueeze(0))
    rollout = mod.compute_rollout_attention(cams, start_layer=start_layer)
    rollout[:, 0, 0] = rollout[:, 0].min()
    return rollout[:, 0]


def bert_logits(model, input_ids, attention_mask):
    with _ref_imports():
        with torch.enable_grad():
            return model(input_ids=input_ids, attention_mask=attention_mask)[0].detach()
