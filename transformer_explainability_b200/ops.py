"""Stand-alone LRP rules and rollout on CUDA tensors (thin wrappers over the C ABI).

Each function is the CUDA counterpart of one ``relprop`` of the reference's
``modules/layers_ours.py`` (alpha=1); see ``include/te_b200.h`` for the citations.
All inputs must be contiguous fp32 CUDA tensors; there is no CPU path.
"""
import torch

from . import _lib
from ._lib import check, ptr


import functools


def _stream():
    return _lib.ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _on_device(fn):
    """Run the op with the device of its first CUDA tensor argument current: the C library launches on the current
    device and the stream handed to it must belong to that device (a model on a non-current GPU otherwise fails with
    an invalid resource handle)."""
    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        dev = None
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, (list, tuple)) and a and torch.is_tensor(a[0]):
                a = a[0]
            if torch.is_tensor(a) and a.is_cuda:
                dev = a.device
                break
        if dev is None:
            raise ValueError("te_b200 ops need CUDA tensors (no CPU fallback)")
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapped


def _req(*ts):
    dev = None
    for t in ts:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError("te_b200 ops need contiguous fp32 CUDA tensors (no CPU fallback)")
        if dev is not None and t.device != dev:
            raise ValueError("te_b200 ops: all tensors of one call must live on the same device")
        dev = t.device


def _same_shape(what, *ts):
    ts = [t for t in ts if t is not None]
    for t in ts[1:]:
        if t.shape != ts[0].shape:
            raise ValueError("%s: shape mismatch %s vs %s" % (what, tuple(ts[0].shape), tuple(t.shape)))


def _workspace(nbytes, device):
    return torch.empty((nbytes + 255) // 256 * 64, dtype=torch.float32, device=device)   # 256-byte multiple


@_on_device
def linear_forward(x, w, bias=None, tensor_cores=False, f16_split=False):
    """y = x W^T + b.  tensor_cores: fp32-grade 3xTF32 split on tcgen05 (shapes that do not qualify fall back);
    f16_split (with tensor_cores): the row-scaled fp16 (hi, lo) split on tcgen05 kind::f16 (TE_FLAG_LINEAR_F16_SPLIT)."""
    _req(x, w, bias)
    if w.dim() != 2 or x.shape[-1] != w.shape[1] or (bias is not None and bias.numel() != w.shape[0]):
        raise ValueError("linear_forward: x [...,in], w [out,in], bias [out] expected")
    rows = x.numel() // x.shape[-1]
    y = torch.empty(*x.shape[:-1], w.shape[0], device=x.device, dtype=torch.float32)
    nscratch = 16 * w.numel() + ((x.numel() + 63) // 64 * 64 + rows * ((x.shape[-1] + 127) // 128) if f16_split else 0)
    scratch = torch.empty(nscratch, device=x.device, dtype=torch.float32) if tensor_cores else None
    flags = (_lib.FLAG_LINEAR_TENSOR_CORES if tensor_cores else 0) | (_lib.FLAG_LINEAR_F16_SPLIT if f16_split else 0)
    check(_lib.load().te_linear_forward_ex(ptr(x), ptr(w), ptr(bias), ptr(y), ptr(scratch), rows, x.shape[-1], w.shape[0],
                                           flags, _stream()),
          "te_linear_forward_ex")
    return y


@_on_device
def f16_block_split(x):
    """The block-scaled fp16 (hi, lo) operand format of the fp16-split forward Linear: x [rows, cols] fp32 ->
    (hi, lo) fp16 [rows, cols], scale_inv fp32 [rows, ceil(cols / 128)]  (see include/te_b200.h: te_f16_block_split)."""
    _req(x)
    if x.dim() != 2 or x.shape[1] % 4 != 0:
        raise ValueError("f16_block_split: x [rows, cols] with cols % 4 == 0 expected")
    rows, cols = x.shape
    buf = torch.empty(2, rows, cols, device=x.device, dtype=torch.float16)
    scale = torch.empty(rows, (cols + 127) // 128, device=x.device, dtype=torch.float32)
    check(_lib.load().te_f16_block_split(ptr(x), rows, cols, ptr(buf[0]), ptr(buf[1]), ptr(scale), _stream()), "te_f16_block_split")
    return buf[0], buf[1], scale


@_on_device
def linear_backward(dy, w, tensor_cores=False):
    """dx = dy W  (activation gradient of a Linear; no dW on this path)."""
    _req(dy, w)
    if w.dim() != 2 or dy.shape[-1] != w.shape[0]:
        raise ValueError("linear_backward: dy [...,out], w [out,in] expected")
    rows = dy.numel() // dy.shape[-1]
    dx = torch.empty(*dy.shape[:-1], w.shape[1], device=dy.device, dtype=torch.float32)
    scratch = torch.empty(16 * w.numel(), device=dy.device, dtype=torch.float32) if tensor_cores else None
    check(_lib.load().te_linear_backward_ex(ptr(dy), ptr(w), ptr(dx), ptr(scratch), rows, w.shape[1], w.shape[0],
                                            _lib.FLAG_LINEAR_TENSOR_CORES if tensor_cores else 0, _stream()),
          "te_linear_backward_ex")
    return dx


@_on_device
def linear_backward_f16(dy, w):
    """dx = dy W as a single-pass fp16 GEMM (block-scaled fp16 gradient, row-scaled fp16 weights; TE_FLAG_BACKWARD_F16)."""
    _req(dy, w)
    if w.dim() != 2 or dy.shape[-1] != w.shape[0]:
        raise ValueError("linear_backward_f16: dy [...,out], w [out,in] expected")
    rows = dy.numel() // dy.shape[-1]
    dx = torch.empty(*dy.shape[:-1], w.shape[1], device=dy.device, dtype=torch.float32)
    n = 16 * w.numel() + (dy.numel() // 2 + 63) // 64 * 64 + rows * ((w.shape[0] + 127) // 128)
    scratch = torch.empty(n, device=dy.device, dtype=torch.float32)
    check(_lib.load().te_linear_backward_ex(ptr(dy), ptr(w), ptr(dx), ptr(scratch), rows, w.shape[1], w.shape[0],
                                            _lib.FLAG_LINEAR_TENSOR_CORES | _lib.FLAG_BACKWARD_F16, _stream()),
          "te_linear_backward_ex")
    return dx


@_on_device
def linear_backward_tf32(dy, w):
    """dx = dy W as a single-pass TF32 GEMM on the persistent CTA-pair kernel (what TE_FLAG_BACKWARD_TF32 selects)."""
    _req(dy, w)
    if w.dim() != 2 or dy.shape[-1] != w.shape[0]:
        raise ValueError("linear_backward_tf32: dy [...,out], w [out,in] expected")
    rows = dy.numel() // dy.shape[-1]
    dx = torch.empty(*dy.shape[:-1], w.shape[1], device=dy.device, dtype=torch.float32)
    scratch = torch.empty(16 * w.numel(), device=dy.device, dtype=torch.float32)
    check(_lib.load().te_linear_backward_ex(ptr(dy), ptr(w), ptr(dx), ptr(scratch), rows, w.shape[1], w.shape[0],
                                            _lib.FLAG_LINEAR_TENSOR_CORES | _lib.FLAG_BACKWARD_TF32, _stream()),
          "te_linear_backward_ex")
    return dx


_ATTN_EPI = {"store": _lib.ATTN_STORE, "mul": _lib.ATTN_MUL, "sd": _lib.ATTN_SD, "softmax": _lib.ATTN_SOFTMAX}


def _packed_rows(t, what):
    """Row stride of a 2-D fp32 CUDA view with unit column stride (e.g. a column slice of a packed activation)."""
    if t.dim() != 2 or t.dtype != torch.float32 or not t.is_cuda or t.stride(1) != 1:
        raise ValueError("%s: 2-D fp32 CUDA view with unit column stride expected" % what)
    return t.stride(0)


@_on_device
def attention_nn(a, b, batch, heads, epi="store", e=None, out=None, alpha=1.0, flags=0):
    """TEST ONLY (kernel unit tests; the engines call the same dispatch internally).  The N x N attention contraction
    ``out[b,h,i,j] = epi(alpha * sum_d a[b*n+i, h*dh+d] * b[b*n+j, h*dh+d])`` (see include/te_b200.h: te_attention_nn).
    a, b: [batch*n, heads*dh] views with unit column stride (head slices of a packed qkv buffer, addressed in place);
    out, e: contiguous [batch, heads, n, ld_out] (out allocated with ld_out = round_up(n, 4) when None);
    epi: "store" | "mul" | "sd" | "softmax"; flags: 0 (fp32 SIMT) or FLAG_ATTN_TENSOR_CORES [| FLAG_RELPROP_TF32]."""
    lda, ldb = _packed_rows(a, "attention_nn a"), _packed_rows(b, "attention_nn b")
    if a.shape != b.shape or a.shape[0] % batch or a.shape[1] % heads:
        raise ValueError("attention_nn: a, b [batch*n, heads*dh] expected")
    n, dh = a.shape[0] // batch, a.shape[1] // heads
    if out is None:
        out = torch.empty(batch, heads, n, (n + 3) // 4 * 4, device=a.device, dtype=torch.float32)
    _req(out, e)
    if out.dim() != 4 or tuple(out.shape[:3]) != (batch, heads, n) or (e is not None and e.shape != out.shape):
        raise ValueError("attention_nn: out / e [batch, heads, n, ld_out] expected")
    check(_lib.load().te_attention_nn(ptr(a), lda, ptr(b), ldb, batch, heads, n, dh, ptr(e), ptr(out), out.shape[3], alpha,
                                      _ATTN_EPI[epi], flags, _stream()), "te_attention_nn")
    return out


@_on_device
def attention_nk(amap, x, heads, transpose=False, epi="store", e=None, out=None, alpha=1.0, flags=0):
    """TEST ONLY (kernel unit tests; the engines call the same dispatch internally).  The token-reduced N x d contraction
    ``out[b*n+m, h*dh+c] = epi(alpha * sum_k A_h[m,k] * x[b*n+k, h*dh+c])`` with A_h = amap[b,h] or its transpose
    (see include/te_b200.h: te_attention_nk).  amap: contiguous [batch, heads, n, np] (pad columns finite);
    x, out, e: [batch*n, heads*dh] views with unit column stride (out, e share one row stride; out allocated packed when
    None); epi: "store" | "mul"; flags: 0 (fp32 SIMT) or FLAG_ATTN_TENSOR_CORES [| FLAG_RELPROP_TF32]."""
    _req(amap)
    ldx = _packed_rows(x, "attention_nk x")
    if amap.dim() != 4 or amap.shape[1] != heads or x.shape[0] != amap.shape[0] * amap.shape[2] or x.shape[1] % heads:
        raise ValueError("attention_nk: amap [batch, heads, n, np], x [batch*n, heads*dh] expected")
    batch, n, np_ = amap.shape[0], amap.shape[2], amap.shape[3]
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.float32)
    ld_out = _packed_rows(out, "attention_nk out")
    if out.shape != x.shape or (e is not None and (e.shape != x.shape or _packed_rows(e, "attention_nk e") != ld_out)):
        raise ValueError("attention_nk: out / e [batch*n, heads*dh] with one row stride expected")
    check(_lib.load().te_attention_nk(ptr(amap), np_, int(transpose), ptr(x), ldx, batch, heads, n, x.shape[1] // heads,
                                      ptr(e), ptr(out), ld_out, alpha, _ATTN_EPI[epi], flags, _stream()), "te_attention_nk")
    return out


@_on_device
def linear_relprop(x, w, r, tensor_cores=False, y=None, bias=None, bf16=False, variant="ours", r_f16=False):
    """``Linear.relprop`` (layers_ours.py:207-230): x [...,in], w [out,in], r [...,out] -> [...,in].
    y / bias: the layer's saved forward output (and bias) — lets the tensor-core path form the denominator in one pass.
    variant="lrp": the rule of ``modules/layers_lrp.py:187-210`` (separate denominators; fp32 SIMT)."""
    _req(x, w, r, y, bias)
    if (w.dim() != 2 or x.shape[-1] != w.shape[1] or r.shape[-1] != w.shape[0] or r.shape[:-1] != x.shape[:-1]
            or (y is not None and y.shape != r.shape) or (bias is not None and bias.numel() != w.shape[0])):
        raise ValueError("linear_relprop: x [...,in], w [out,in], r / y [...,out], bias [out] expected")
    rows = x.numel() // x.shape[-1]
    out = torch.empty_like(x)
    nscratch = rows * w.shape[0]
    if tensor_cores:
        nscratch = (nscratch + 63) // 64 * 64 + 16 * w.numel() + x.numel()
    scratch = torch.empty(nscratch, device=x.device, dtype=torch.float32)
    flags = _lib.FLAG_ZPLUS_TENSOR_CORES if tensor_cores else 0
    if r_f16:
        flags |= _lib.FLAG_ZPLUS_R_F16
    if bf16 == "s1":
        flags |= _lib.FLAG_ZPLUS_S1_BF16              # bf16 operands for the |x||W|^T term of the single-pass denominator
    elif bf16:
        flags |= _lib.FLAG_ZPLUS_BF16
    if variant == "lrp":
        flags, y = _lib.FLAG_RULES_LRP, None
    elif variant != "ours":
        raise ValueError("variant: 'ours' or 'lrp'")
    if y is not None:
        check(_lib.load().te_linear_relprop_ex(ptr(x), ptr(w), ptr(bias), ptr(y), ptr(r), ptr(out), ptr(scratch), rows,
                                               x.shape[-1], w.shape[0], flags, _stream()), "te_linear_relprop_ex")
    else:
        check(_lib.load().te_linear_relprop(ptr(x), ptr(w), ptr(r), ptr(out), ptr(scratch), rows, x.shape[-1], w.shape[0],
                                            flags, _stream()), "te_linear_relprop")
    return out


@_on_device
def add_relprop(x1, x2, r, variant="ours"):
    """``Add.relprop`` (layers_ours.py:97-120), sums per sample (dim 0).  variant="lrp": ``modules/layers_lrp.py:98-100``
    (x1*S, x2*S with S = sd(r, x1+x2); no ratio normalisation)."""
    _req(x1, x2, r)
    _same_shape("add_relprop", x1, x2, r)           # a broadcast operand (pos_embed [1,N,D]) must be expanded by the caller
    if (x1.numel() // max(x1.shape[0], 1)) % 4 != 0:
        raise ValueError("add_relprop: elements per sample must be a multiple of 4")
    b = x1.shape[0]
    r1, r2 = torch.empty_like(x1), torch.empty_like(x1)
    scratch = None if variant == "lrp" else torch.empty(b * 48, device=x1.device, dtype=torch.float64)
    check(_lib.load().te_add_relprop(ptr(x1), ptr(x2), ptr(r), ptr(r1), ptr(r2), ptr(scratch), b, x1.numel() // b,
                                     _stream()), "te_add_relprop")
    return r1, r2


@_on_device
def clone_relprop(x, rs):
    """``Clone.relprop`` (layers_ours.py:151-169) for 2 or 3 branches."""
    rs = list(rs)
    _req(x, *rs)
    if len(rs) not in (2, 3):
        raise ValueError("clone_relprop: 2 or 3 branches")
    _same_shape("clone_relprop", x, *rs)
    out = torch.empty_like(x)
    r3 = rs[2] if len(rs) > 2 else None
    check(_lib.load().te_clone_relprop(ptr(x), ptr(rs[0]), ptr(rs[1]), ptr(r3), ptr(out), x.numel(), _stream()),
          "te_clone_relprop")
    return out


@_on_device
def index_select_relprop(x, r):
    """``IndexSelect.relprop`` (layers_ours.py:129-147), dim=1, index 0: x [B,N,D], r [B,1,D]|[B,D]."""
    if x.dim() != 3 or r.numel() != x.shape[0] * x.shape[2]:
        raise ValueError("index_select_relprop: x [B,N,D], r [B,1,D] expected")
    r = r.reshape(x.shape[0], x.shape[2]).contiguous()
    _req(x, r)
    out = torch.empty_like(x)
    check(_lib.load().te_index_select_relprop(ptr(x), ptr(r), ptr(out), x.shape[0], x.shape[1], x.shape[2], _stream()),
          "te_index_select_relprop")
    return out


@_on_device
def matmul_av_relprop(p, v, r):
    """``einsum('bhij,bhjd->bhid').relprop``: returns UN-halved (R_attn, R_v)."""
    _req(p, v, r)
    if v.dim() != 4 or p.shape != v.shape[:2] + (v.shape[2], v.shape[2]):
        raise ValueError("matmul_av_relprop: p [B,H,N,N], v [B,H,N,d], r [B,H,N,d] expected")
    _same_shape("matmul_av_relprop", v, r)
    b, h, n, d = v.shape
    rp, rv = torch.empty_like(p), torch.empty_like(v)
    scratch = torch.empty(b * h * n * d, device=p.device, dtype=torch.float32)
    check(_lib.load().te_matmul_av_relprop(ptr(p), ptr(v), ptr(r), ptr(rp), ptr(rv), ptr(scratch), b * h, n, d,
                                           _stream()), "te_matmul_av_relprop")
    return rp, rv


@_on_device
def matmul_qk_relprop(q, k, r):
    """``einsum('bhid,bhjd->bhij').relprop``: returns UN-halved (R_q, R_k)."""
    _req(q, k, r)
    if q.dim() != 4 or r.shape != q.shape[:2] + (q.shape[2], q.shape[2]):
        raise ValueError("matmul_qk_relprop: q, k [B,H,N,d], r [B,H,N,N] expected")
    _same_shape("matmul_qk_relprop", q, k)
    b, h, n, d = q.shape
    rq, rk = torch.empty_like(q), torch.empty_like(k)
    scratch = torch.empty(b * h * n * n, device=q.device, dtype=torch.float32)
    check(_lib.load().te_matmul_qk_relprop(ptr(q), ptr(k), ptr(r), ptr(rq), ptr(rk), ptr(scratch), b * h, n, d,
                                           _stream()), "te_matmul_qk_relprop")
    return rq, rk


def _attn_layout(t):
    """[B,H,N,N] view (row stride ld >= N, as handed out by the engine accessors) -> (tensor, ld)."""
    if t.dim() != 4 or t.shape[-1] != t.shape[-2] or t.dtype != torch.float32 or not t.is_cuda:
        raise ValueError("expected an fp32 CUDA tensor [B,H,N,N]")
    B, H, N, _ = t.shape
    ld = t.stride(2)
    if t.stride(3) != 1 or ld < N or t.stride(1) != N * ld or t.stride(0) != H * N * ld:
        t = t.contiguous()
        ld = N
    return t, ld


@_on_device
def head_reduce(a, g=None, head_weight=None, mode="mean"):
    """Reduce an attention-shaped tensor over its heads: a [B,H,N,N] (optionally * g, * head_weight[B,H]) -> [B,N,N].
    mode: "mean" | "relu_mean" (``clamp(min=0).mean(heads)``) | "mean_relu" (``mean(heads).clamp(min=0)``)."""
    a, ld = _attn_layout(a)
    if g is not None:
        g, ldg = _attn_layout(g)
        if ldg != ld:
            a, g, ld = a.contiguous(), g.contiguous(), a.shape[-1]
    B, H, N, _ = a.shape
    if head_weight is not None:
        _req(head_weight)
    out = torch.empty(B, N, N, device=a.device, dtype=torch.float32)
    m = {"mean": 0, "relu_mean": 1, "mean_relu": 2}[mode]
    check(_lib.load().te_head_reduce(ptr(a), ptr(g), ptr(head_weight), B, H, N, ld, m, ptr(out), _stream()),
          "te_head_reduce")
    return out


@_on_device
def head_region_mean(g, rows=None, cols=None):
    """``g[b,h, rows, cols].mean()`` per (b,h): [B,H,N,N] -> [B,H] (``grad.mean(dim=[1,2])`` of the GradCAM baselines)."""
    g, ld = _attn_layout(g)
    B, H, N, _ = g.shape
    r0, r1 = rows if rows is not None else (0, N)
    c0, c1 = cols if cols is not None else (0, N)
    out = torch.empty(B, H, device=g.device, dtype=torch.float32)
    check(_lib.load().te_head_region_mean(ptr(g), B, H, N, ld, r0, r1, c0, c1, ptr(out), _stream()), "te_head_region_mean")
    return out


@_on_device
def patch_embed_relprop(images, weight, r, per_channel=True):
    """``PatchEmbed.relprop`` -> ``Conv2d.relprop`` z^B branch (ViT_LRP.py:238-242, layers_ours.py:242-259).
    images [B,C,S,S]; weight [D,C,P,P] (or flattened [D,C*P*P]); r [B,(S/P)^2,D] -> [B,C,S,S] (or [B,S,S] channel sum)."""
    _req(images, weight, r)
    B, C, S, _ = images.shape
    D = weight.shape[0]
    P = int(round((weight.numel() // (D * C)) ** 0.5))
    lib = _lib.load()
    nbytes = check(lib.te_patch_embed_relprop_workspace_bytes(B, C, S, P, D), "te_patch_embed_relprop_workspace_bytes")
    ws = _workspace(nbytes, images.device)
    out = torch.empty((B, C, S, S) if per_channel else (B, S, S), device=images.device, dtype=torch.float32)
    check(lib.te_patch_embed_relprop(ptr(images), ptr(weight), ptr(r), B, C, S, P, D, ptr(out) if per_channel else None,
                                     None if per_channel else ptr(out), ptr(ws), ws.numel() * 4, _stream()),
          "te_patch_embed_relprop")
    return out


@_on_device
def attribution_rollout(grad, cam, start_layer=0, normalize=False, fused=False, want_joint=True):
    """grad, cam [L,B,H,N,N] -> (joint [B,N,N] or None, row0 [B,N]).
    ``ViT_LRP.py:357-368`` (normalize=False) / ``ExplanationGenerator.py:47-57`` (normalize=True)."""
    _req(grad, cam)
    _same_shape("attribution_rollout", grad, cam)
    if grad.dim() != 5 or grad.shape[4] < grad.shape[3]:
        raise ValueError("attribution_rollout: grad, cam [L,B,H,N,ld] with ld >= N expected")
    L, B, H, N, ld = grad.shape
    lib = _lib.load()
    nbytes = check(lib.te_rollout_workspace_bytes(L, B, N), "te_rollout_workspace_bytes")
    ws = _workspace(nbytes, grad.device)
    joint = torch.empty(B, N, N, device=grad.device, dtype=torch.float32) if want_joint else None
    row0 = torch.empty(B, N, device=grad.device, dtype=torch.float32)
    flags = _lib.FLAG_ROLLOUT_FUSED if fused else 0
    check(lib.te_attribution_rollout(ptr(grad), ptr(cam), L, B, H, N, ld, start_layer, int(normalize), flags, ptr(joint),
                                     ptr(row0), ptr(ws), ws.numel() * 4, _stream()), "te_attribution_rollout")
    return joint, row0


@_on_device
def compute_rollout_attention(all_layer_matrices, start_layer=0, normalize=False):
    """``compute_rollout_attention`` (ViT_LRP.py:38-49; BERT variant with normalize=True,
    ExplanationGenerator.py:7-18): list of [B,N,N] -> [B,N,N]."""
    mats = torch.stack([m.to(torch.float32) for m in all_layer_matrices]).contiguous()
    _req(mats)
    L, B, N, _ = mats.shape
    lib = _lib.load()
    nbytes = check(lib.te_rollout_workspace_bytes(L, B, N), "te_rollout_workspace_bytes")
    ws = _workspace(nbytes, mats.device)
    joint = torch.empty(B, N, N, device=mats.device, dtype=torch.float32)
    check(lib.te_compute_rollout_attention(ptr(mats), L, B, N, start_layer, int(normalize), ptr(joint), ptr(ws),
                                           ws.numel() * 4, _stream()), "te_compute_rollout_attention")
    return joint
