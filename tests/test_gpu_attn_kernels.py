"""The attention-shaped contractions (csrc/te_tc_attn.cu, te_gemm.cu, the row softmax) called directly, against fp64.

``ops.attention_nn`` / ``ops.attention_nk`` go through the engines' own dispatch (``te_util::attn_nn`` / ``attn_probs`` /
``attn_nk``), so every flag selects exactly the kernel an engine would run for that shape:
  flags 0                                    fp32 SIMT GEMM (+ the row-softmax kernel for SOFTMAX)
  FLAG_ATTN_TENSOR_CORES                     tcgen05 3xTF32: N x N (STORE / MUL / SD / fused SOFTMAX for N <= 256,
                                             scores + row-softmax kernel above), N x d (K-major or transposed map)
  | FLAG_RELPROP_TF32                        single-pass TF32 for STORE / MUL (N x N only for N <= 256: 3xTF32 above)
Operands are head slices of a packed qkv-like buffer ``[batch*N, 3*H*dh]`` addressed in place, exactly as the engines
address them: with batch 3 the row tiles straddle sample boundaries and the last sample's tile runs past the allocation.

Error is judged per element, relative to that element's own scale ``alpha * (|A_h| |B_h|^T)`` (x |E| for MUL), so that an
error in a small entry is not hidden by a large one.  Bounds, with the largest errors measured on a B200 (1000 W):
  fp32 SIMT      (K + 3) 2^-24 — the classical worst-case bound of a K-term fp32 dot product plus the epilogue roundings
                 (measured <= 3.7e-7, and 6.7e-7 for SD).
  3xTF32         TC_SLOPE * K + TC_FLOOR.  The hi/lo split leaves ~2^-22 per product; the tensor core truncates its fp32
                 accumulator at every MMA, which adds a drift linear in K.  Measured: N x N 4.9e-7 (K = 32) and 6.5e-7
                 (K = 64) on signed operands, 1.3e-6 (K = 64) on the positive operands of the SD test, where the
                 truncation errors all have one sign; N x d 5.8e-7 (K = 65), 1.1e-6 (K = 224), 1.6e-6 (K = 512).  The
                 bound is 1.8x the worst of these (SD, K = 64) and 4x at K = 512.
  single pass    2e-3 of scale: two operands truncated to TF32 (2^-10 each) and compensated by 1.00068 on average.
                 Measured <= 4.9e-4 at K >= 32, 1.0e-3 at K = 1 (one product, nothing averages).  The bias check: on
                 all-positive operands the mean signed relative error must stay below SP_BIAS = 1e-4.  That is 1/7 of
                 the 6.8e-4 shrink of the uncompensated form.  Measured: 2.6e-6 (N x N) and 1.6e-5 (N x d).
The map operand of the N x d contraction has row stride NP > N; its pad columns [N, NP) are filled with 7.0 (they must be
finite: the tensor core multiplies them by zero-filled rows, and NaN * 0 = NaN) and must not change the result.
"""
import ctypes

import pytest
import torch

from oracle import bert as obert
from oracle import conditioned
from oracle import cpu as ocpu
from oracle import rules
from oracle import vit as ovit

gpu = pytest.mark.gpu

U = 2.0 ** -24
TC_SLOPE, TC_FLOOR = 1e-8, 1.5e-6          # 3xTF32 per-element bound: TC_SLOPE * K + TC_FLOOR of scale
SP_BOUND = 2e-3                            # single-pass TF32 per-element bound, of scale
SP_BIAS = 1e-4                             # |mean signed relative error| of the single-pass form on positive operands
GUARD = 4096                               # floats after every output that must stay untouched

NS = [1, 4, 17, 65, 127, 128, 129, 197, 198, 224, 225, 256, 257, 300, 512]
CASES_NN = [(3, 2, n, dh) for n in NS for dh in (32, 64)] + [(2, 12, 197, 64), (2, 12, 512, 64)]
CASES_NK = [(3, 2, n) for n in NS] + [(2, 12, 197), (2, 12, 512)]


def simt_bound(k):
    return (k + 3) * U


def tc_bound(k):
    return TC_SLOPE * k + TC_FLOOR


def f32(x):
    """x as the fp32 value the kernels receive (the references use the same alpha)."""
    return float(torch.tensor(x, dtype=torch.float32))


def rup4(n):
    return (n + 3) // 4 * 4


def _lib():
    from transformer_explainability_b200 import _lib as L
    return L


def _packed(batch, n, heads, dh, seed, positive=False):
    """[batch*n, 3*heads*dh] fp32: q | k | v column blocks of a packed activation."""
    g = torch.Generator().manual_seed(seed)
    if positive:
        return torch.rand(batch * n, 3 * heads * dh, generator=g) + 0.05
    return torch.randn(batch * n, 3 * heads * dh, generator=g)


def _heads(t, batch, n, heads):
    """[batch*n, heads*dh] -> fp64 [batch, heads, n, dh]."""
    return t.double().reshape(batch, n, heads, -1).permute(0, 2, 1, 3)


def _unheads(t):
    """fp64 [batch, heads, n, dh] -> [batch*n, heads*dh]."""
    b, h, n, d = t.shape
    return t.permute(0, 2, 1, 3).reshape(b * n, h * d)


def _nn_out(batch, heads, n, ld):
    """NaN-filled output [batch, heads, n, ld] followed by a guard block in the same allocation."""
    buf = torch.full((batch * heads * n * ld + GUARD,), float("nan"), device="cuda")
    return buf, buf[:batch * heads * n * ld].view(batch, heads, n, ld)


def _elem_err(got, ref, scale):
    return ((got.double().cpu() - ref).abs() / scale.clamp_min(1e-300)).max().item()


def _check_nn_footprint(buf, out, n, kind):
    """kind "gemm": the SIMT GEMM writes columns [0, n) only; "tc": the tcgen05 kernel also zeroes the row padding
    [n, round_up(n, 4)) and leaves [round_up(n, 4), ld) alone; "rowsoftmax": the row-softmax kernel zeroes [n, ld)."""
    o = out.cpu()
    np_ = rup4(n)
    assert torch.isnan(buf[-GUARD:]).all(), "guard block after the output was written"
    if kind == "gemm":
        assert torch.isnan(o[..., n:]).all()
    elif kind == "tc":
        assert (o[..., n:np_] == 0).all(), "row padding [N, round_up(N,4)) not zeroed"
        assert torch.isnan(o[..., np_:]).all(), "columns past round_up(N,4) were written"
    else:
        assert (o[..., n:] == 0).all()
    assert not torch.isnan(o[..., :n]).any(), "output columns left unwritten"


# ---- N x N ----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("batch,heads,n,dh", CASES_NN)
def test_attention_nn_store_mul(batch, heads, n, dh):
    """out = alpha Q K^T and alpha Q K^T * E: SIMT, 3xTF32 and single-pass against fp64 and against each other."""
    from transformer_explainability_b200 import ops
    L = _lib()
    TC, SP = L.FLAG_ATTN_TENSOR_CORES, L.FLAG_ATTN_TENSOR_CORES | L.FLAG_RELPROP_TF32
    w = heads * dh
    t = _packed(batch, n, heads, dh, seed=n * 131 + dh)
    d = t.cuda()
    a, b = d[:, :w], d[:, w:2 * w]
    A, B = _heads(t[:, :w], batch, n, heads), _heads(t[:, w:2 * w], batch, n, heads)
    alpha = f32(dh ** -0.5)
    S = alpha * A @ B.transpose(-1, -2)
    scale = alpha * A.abs() @ B.abs().transpose(-1, -2)
    ld = rup4(n) + 4
    E = torch.randn(batch, heads, n, ld, generator=torch.Generator().manual_seed(n + 7))
    Ed, Ev = E.cuda(), E[..., :n].double()
    # single-pass N x N runs only for N <= 256 (the dispatch takes 3xTF32 above)
    bounds = {0: simt_bound(dh), TC: tc_bound(dh), SP: SP_BOUND if n <= 256 else tc_bound(dh)}
    over = []                                   # every case is measured and printed before the bounds are asserted
    for epi, ref, sc in (("store", S, scale), ("mul", S * Ev, scale * Ev.abs())):
        got = {}
        for flags in (0, TC, SP):
            buf, out = _nn_out(batch, heads, n, ld)
            ops.attention_nn(a, b, batch, heads, epi=epi, e=Ed if epi == "mul" else None, out=out, alpha=alpha, flags=flags)
            torch.cuda.synchronize()
            _check_nn_footprint(buf, out, n, "gemm" if flags == 0 else "tc")
            got[flags] = out[..., :n].double().cpu()
            e = _elem_err(got[flags], ref, sc)
            print("nn %s B%d H%d N%d dh%d flags %d: per-element err %.2e of scale (bound %.1e)" % (
                epi, batch, heads, n, dh, flags, e, bounds[flags]))
            if e >= bounds[flags]:
                over.append("nn %s flags %d: %g" % (epi, flags, e))
        # the tensor-core results agree with the library's SIMT result within the sum of the two bounds
        for flags in (TC, SP):
            assert ((got[flags] - got[0]).abs() <= (bounds[flags] + bounds[0]) * sc).all()
    assert not over, over


@gpu
@pytest.mark.parametrize("batch,heads,n,dh", CASES_NN)
def test_attention_nn_safe_divide(batch, heads, n, dh):
    """out = safe_divide(E, alpha Q K^T) (layers_ours.py:10-13) on positive operands (denominator = its own scale, well
    conditioned), with one all-zero Q row and one all-zero K row: their denominators are exactly 0, so the ``b != 0``
    mask makes the output exactly 0 there although E is not."""
    from transformer_explainability_b200 import ops
    L = _lib()
    TC = L.FLAG_ATTN_TENSOR_CORES
    w = heads * dh
    t = _packed(batch, n, heads, dh, seed=n * 17 + dh, positive=True)
    zq = (0, n // 2, 0)                       # sample 0, query row n // 2, head 0
    zk = (batch - 1, n - 1, heads - 1)        # last sample, last key row, last head
    t[zq[0] * n + zq[1], zq[2] * dh:(zq[2] + 1) * dh] = 0.0
    t[zk[0] * n + zk[1], w + zk[2] * dh:w + (zk[2] + 1) * dh] = 0.0
    d = t.cuda()
    A, B = _heads(t[:, :w], batch, n, heads), _heads(t[:, w:2 * w], batch, n, heads)
    alpha = f32(dh ** -0.5)
    S = alpha * A @ B.transpose(-1, -2)
    ld = rup4(n) + 4
    E = torch.randn(batch, heads, n, ld, generator=torch.Generator().manual_seed(n + 11))
    E[E == 0] = 1.0
    ref = rules.safe_divide(E[..., :n].double(), S)
    zero = torch.zeros(batch, heads, n, n, dtype=torch.bool)
    zero[zq[0], zq[2], zq[1], :] = True
    zero[zk[0], zk[2], :, zk[1]] = True
    assert (S[zero] == 0).all() and (S[~zero] > 0).all()
    got = {}
    for flags, bound in ((0, simt_bound(dh)), (TC, tc_bound(dh) + 4 * U)):         # + rcp.approx of the quotient
        buf, out = _nn_out(batch, heads, n, ld)
        ops.attention_nn(d[:, :w], d[:, w:2 * w], batch, heads, epi="sd", e=E.cuda(), out=out, alpha=alpha, flags=flags)
        torch.cuda.synchronize()
        _check_nn_footprint(buf, out, n, "gemm" if flags == 0 else "tc")
        g = got[flags] = out[..., :n].double().cpu()
        assert (g[zero] == 0).all(), "safe_divide by an exact zero must give 0 (flags %d)" % flags
        e = ((g - ref).abs() / ref.abs().clamp_min(1e-300))[~zero].max().item()
        print("nn sd B%d H%d N%d dh%d flags %d: relative err %.2e (bound %.1e)" % (batch, heads, n, dh, flags, e, bound))
        assert e < bound
    assert ((got[TC] - got[0]).abs() <= (simt_bound(dh) + tc_bound(dh) + 4 * U) * ref.abs()).all()


@gpu
@pytest.mark.parametrize("alpha_scale", [1.0, 100.0])
@pytest.mark.parametrize("batch,heads,n,dh", CASES_NN)
def test_attention_nn_softmax(batch, heads, n, dh, alpha_scale):
    """P = softmax(alpha Q K^T) over the keys: fused into the tcgen05 epilogue for N <= 256, scores + row-softmax kernel
    above.  Rows sum to 1 within (N + 8) 2^-24 (rounding of the sum and of the normalisation only); every element within
    P (2 delta + (N + 8) 2^-24 + 2^-22 (1 + |s| + |max s|)), delta the row's score error bound.  Includes rows of equal
    scores (zero query rows: P = 1/N) and, at alpha_scale 100, rows where almost every exponential underflows."""
    from transformer_explainability_b200 import ops
    L = _lib()
    TC = L.FLAG_ATTN_TENSOR_CORES
    w = heads * dh
    t = _packed(batch, n, heads, dh, seed=n * 7 + dh)
    t[0, :dh] = 0.0                                           # sample 0, head 0, query row 0: all scores equal
    t[(batch - 1) * n + n // 2, w - dh:w] = 0.0               # last sample, last head, middle row
    d = t.cuda()
    A, B = _heads(t[:, :w], batch, n, heads), _heads(t[:, w:2 * w], batch, n, heads)
    alpha = f32(alpha_scale * dh ** -0.5)
    s = alpha * A @ B.transpose(-1, -2)
    ref = torch.softmax(s, dim=-1)
    mx = s.amax(dim=-1, keepdim=True)
    scale_row = (alpha * A.abs() @ B.abs().transpose(-1, -2)).amax(dim=-1, keepdim=True)
    if alpha_scale > 1 and n >= 128:
        assert (ref < 2.0 ** -126).double().mean() > 0.9           # most exponentials below the fp32 normal range
    ld = rup4(n) + 4
    got = {}
    for flags, eb in ((0, simt_bound(dh)), (TC, tc_bound(dh))):
        buf, out = _nn_out(batch, heads, n, ld)
        ops.attention_nn(d[:, :w], d[:, w:2 * w], batch, heads, epi="softmax", out=out, alpha=alpha, flags=flags)
        torch.cuda.synchronize()
        _check_nn_footprint(buf, out, n, "tc" if (flags and n <= 256) else "rowsoftmax")
        g = got[flags] = out[..., :n].double().cpu()
        if n == 1 and alpha_scale == 1:
            assert (g == 1.0).all()          # exp(s - max) / itself (at alpha_scale 100 the rounding of alpha * log2(e) shows)
        rs = (g.sum(dim=-1) - 1).abs().max().item()
        bound = ref * (2 * eb * scale_row + (n + 8) * U + 2.0 ** -22 * (1 + s.abs() + mx.abs())) + 1e-30
        e = ((g - ref).abs() / bound).max().item()
        print("nn softmax B%d H%d N%d dh%d alpha %.3g flags %d: |row sum - 1| %.2e (bound %.1e), err / bound %.2f" % (
            batch, heads, n, dh, alpha, flags, rs, (n + 8) * U, e))
        assert rs <= (n + 8) * U
        assert e <= 1.0
        assert (g[0, 0, 0] == g[0, 0, 0, 0]).all() and abs(g[0, 0, 0, 0].item() * n - 1) < 4 * U     # equal scores
    assert ((got[TC] - got[0]).abs() <= 2 * (ref * (2 * (tc_bound(dh) + simt_bound(dh)) * scale_row + (n + 8) * U +
                                                    2.0 ** -22 * (1 + s.abs() + mx.abs())) + 1e-30)).all()


@gpu
@pytest.mark.parametrize("batch,heads,n,dh", CASES_NN)
def test_attention_nn_persistent_kernel(batch, heads, n, dh):
    """te_set_option("attn_persistent", 1): the persistent, TMEM-double-buffered N x N kernel (N <= 224) issues the same
    three MMAs per k-step in the same order as the one-tile kernel and shares its epilogue, so every epilogue is
    bit-equal to it; at N > 224 the option must not change anything (the one-tile kernel runs)."""
    from transformer_explainability_b200 import ops
    L = _lib()
    lib = L.load()
    TC = L.FLAG_ATTN_TENSOR_CORES
    w = heads * dh
    t = _packed(batch, n, heads, dh, seed=n * 3 + dh, positive=True)
    d = t.cuda()
    ld = rup4(n) + 4
    E = (torch.rand(batch, heads, n, ld, generator=torch.Generator().manual_seed(n)) - 0.3).cuda()
    alpha = f32(dh ** -0.5)

    def run_all():
        res = []
        for epi in ("store", "mul", "sd", "softmax"):
            buf, out = _nn_out(batch, heads, n, ld)
            ops.attention_nn(d[:, :w], d[:, w:2 * w], batch, heads, epi=epi, e=E, out=out, alpha=alpha, flags=TC)
            res.append(buf.cpu())
        return res

    one = run_all()
    L.check(lib.te_set_option(b"attn_persistent", 1), "te_set_option")
    try:
        pers = run_all()
        torch.cuda.synchronize()
    finally:
        L.check(lib.te_set_option(b"attn_persistent", 0), "te_set_option")
    for epi, x, y in zip(("store", "mul", "sd", "softmax"), one, pers):
        diff = (x - y).abs().nan_to_num(0.0).max().item()
        print("nn persistent %s B%d H%d N%d dh%d: max |persistent - one-tile| %.2e" % (epi, batch, heads, n, dh, diff))
        assert torch.equal(torch.isnan(x), torch.isnan(y)) and diff == 0.0, "%s: persistent kernel differs" % epi


# ---- N x d (token-reduced) ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("batch,heads,n", CASES_NK)
def test_attention_nk(batch, heads, n):
    """out[b, m, h*64 + c] = alpha sum_k A_h[m,k] X[b, k, h*64 + c] (* E), A_h = map[b,h] or its transpose, written
    into a column slice of a wider packed buffer; K = N up to 512, so the 3xTF32 accumulator drift is visible here."""
    from transformer_explainability_b200 import ops
    L = _lib()
    TC, SP = L.FLAG_ATTN_TENSOR_CORES, L.FLAG_ATTN_TENSOR_CORES | L.FLAG_RELPROP_TF32
    dh, w = 64, heads * 64
    np_ = rup4(n + 1)                                               # always at least one pad column
    t = _packed(batch, n, heads, dh, seed=n * 5 + 1)
    d = t.cuda()
    x = d[:, 2 * w:]
    X = _heads(t[:, 2 * w:], batch, n, heads)
    g = torch.Generator().manual_seed(n + 3)
    amap = torch.randn(batch, heads, n, np_, generator=g)
    amap[..., n:] = 7.0
    amap0 = amap.clone()
    amap0[..., n:] = 0.0
    M = amap[..., :n].double()
    off, ldo = 4, w + 16
    E = torch.randn(batch * n, ldo, generator=g)
    Ed = E.cuda()
    Ev = E[:, off:off + w].double()
    alpha = 0.75
    bounds = {0: simt_bound(n), TC: tc_bound(n), SP: SP_BOUND}
    over = []
    for transpose in (False, True):
        Ah = M.transpose(-1, -2) if transpose else M
        ref0 = _unheads(alpha * Ah @ X)
        sc0 = _unheads(alpha * Ah.abs() @ X.abs())
        for epi, ref, sc in (("store", ref0, sc0), ("mul", ref0 * Ev, sc0 * Ev.abs())):
            got = {}
            for flags in (0, TC, SP):
                res = []
                for m in (amap, amap0):
                    buf = torch.full((batch * n + 64, ldo), float("nan"), device="cuda")
                    out = buf[:batch * n, off:off + w]
                    ops.attention_nk(m.cuda(), x, heads, transpose=transpose, epi=epi,
                                     e=Ed[:, off:off + w] if epi == "mul" else None, out=out, alpha=alpha, flags=flags)
                    res.append(buf.cpu())
                torch.cuda.synchronize()
                full = res[0]
                assert torch.equal(full.nan_to_num(-1.0), res[1].nan_to_num(-1.0)), "pad columns of the map changed the result"
                assert torch.isnan(full[:, :off]).all() and torch.isnan(full[:, off + w:]).all(), "columns outside the slice written"
                assert torch.isnan(full[batch * n:]).all(), "guard rows written"
                got[flags] = full[:batch * n, off:off + w].double()
                e = _elem_err(got[flags], ref, sc)
                print("nk %s transpose %d B%d H%d N%d flags %d: per-element err %.2e of scale (bound %.1e)" % (
                    epi, transpose, batch, heads, n, flags, e, bounds[flags]))
                if e >= bounds[flags]:
                    over.append("nk %s transpose %d flags %d: %g" % (epi, transpose, flags, e))
            for flags in (TC, SP):
                assert ((got[flags] - got[0]).abs() <= (bounds[flags] + bounds[0]) * sc).all()
    assert not over, over


# ---- single pass: no bias ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [65, 197, 256, 512])
def test_single_pass_is_unbiased(n):
    """On all-positive operands every product enters with the same sign, so the mean signed relative error of the
    single-pass TF32 form exposes its compensation: two operands truncated to TF32 shrink a product by 6.8e-4 on average,
    the epilogue multiplies by 1.00068.  |mean| must stay below SP_BIAS for N x N (N <= 256) and both N x d maps."""
    from transformer_explainability_b200 import ops
    L = _lib()
    SP = L.FLAG_ATTN_TENSOR_CORES | L.FLAG_RELPROP_TF32
    batch, heads, dh = 3, 2, 64
    w = heads * dh
    t = _packed(batch, n, heads, dh, seed=n + 1000, positive=True)
    d = t.cuda()
    A, B, X = (_heads(t[:, i * w:(i + 1) * w], batch, n, heads) for i in range(3))
    g = torch.Generator().manual_seed(n + 2000)
    results = []
    if n <= 256:
        ld = rup4(n)
        E = torch.rand(batch, heads, n, ld, generator=g) + 0.5
        S = A @ B.transpose(-1, -2)
        for epi, ref in (("store", S), ("mul", S * E[..., :n].double())):
            out = ops.attention_nn(d[:, :w], d[:, w:2 * w], batch, heads, epi=epi, e=E.cuda() if epi == "mul" else None,
                                   flags=SP)
            results.append(("nn " + epi, out[..., :n].double().cpu(), ref))
    amap = torch.rand(batch, heads, n, rup4(n), generator=g)
    Ep = torch.rand(batch * n, w, generator=g) + 0.5
    for transpose in (False, True):
        Ah = amap[..., :n].double()
        Ah = Ah.transpose(-1, -2) if transpose else Ah
        ref = _unheads(Ah @ X)
        for epi, r in (("store", ref), ("mul", ref * Ep.double())):
            out = ops.attention_nk(amap.cuda(), d[:, 2 * w:], heads, transpose=transpose, epi=epi,
                                   e=Ep.cuda() if epi == "mul" else None, flags=SP)
            results.append(("nk %s transpose %d" % (epi, transpose), out.double().cpu(), r))
    torch.cuda.synchronize()
    over = []
    for what, got, ref in results:
        bias = ((got - ref) / ref).mean().item()
        print("single pass %s N%d: mean signed relative error %.2e (uncompensated: -6.8e-4)" % (what, n, bias))
        if abs(bias) >= SP_BIAS:
            over.append("%s: single-pass bias %g" % (what, bias))
    assert not over, over


# ---- what the tensor-core path refuses -------------------------------------------------------------------------------
@gpu
def test_unsupported_shapes_raise():
    """With the tensor-core flag a shape or epilogue the tcgen05 kernels do not take raises instead of running SIMT."""
    from transformer_explainability_b200 import ops
    L = _lib()
    TC, SP = L.FLAG_ATTN_TENSOR_CORES, L.FLAG_ATTN_TENSOR_CORES | L.FLAG_RELPROP_TF32
    n, heads = 33, 2
    for dh in (16, 48):
        d = torch.randn(n, 3 * heads * dh, device="cuda")
        with pytest.raises(L.TeError, match="head_dim"):
            ops.attention_nn(d[:, :heads * dh], d[:, heads * dh:2 * heads * dh], 1, heads, flags=TC)
        ops.attention_nn(d[:, :heads * dh], d[:, heads * dh:2 * heads * dh], 1, heads, flags=0)     # SIMT takes it
    d = torch.randn(n, 3 * heads * 64, device="cuda")
    e = torch.rand(1, heads, n, rup4(n), device="cuda")
    for epi in ("sd", "softmax"):
        with pytest.raises(L.TeError, match="single-pass"):
            ops.attention_nn(d[:, :128], d[:, 128:256], 1, heads, epi=epi, e=e, flags=SP)
    d32 = torch.randn(n, 3 * heads * 32, device="cuda")
    amap = torch.rand(1, heads, n, rup4(n), device="cuda")
    with pytest.raises(L.TeError, match="head_dim 64"):
        ops.attention_nk(amap, d32[:, 128:], heads, flags=TC)
    ops.attention_nk(amap, d32[:, 128:], heads, flags=0)
    torch.cuda.synchronize()


def test_argument_validation_without_gpu():
    """Bad arguments return TE_ERR_ARG with a message and unsupported tensor-core requests TE_ERR_UNSUPPORTED — both
    before any CUDA call, so this runs without a device (the pointers are never dereferenced)."""
    L = _lib()
    lib = L.load()
    P = ctypes.c_void_p(4096)
    TC, SP = L.FLAG_ATTN_TENSOR_CORES, L.FLAG_ATTN_TENSOR_CORES | L.FLAG_RELPROP_TF32
    ARG, UNSUP = -1, -4

    def nn(a=P, lda=384, b=P, ldb=384, batch=2, heads=2, n=17, dh=64, e=P, out=P, ld_out=20, epi=0, flags=TC):
        return lib.te_attention_nn(a, lda, b, ldb, batch, heads, n, dh, e, out, ld_out, 1.0, epi, flags, None)

    def nk(m=P, np_=20, tr=0, x=P, ldx=384, batch=2, heads=2, n=17, dh=64, e=P, out=P, ld_out=128, epi=0, flags=TC):
        return lib.te_attention_nk(m, np_, tr, x, ldx, batch, heads, n, dh, e, out, ld_out, 1.0, epi, flags, None)

    bad = [(nn, dict(a=None), b"bad argument"), (nn, dict(out=None), b"bad argument"), (nn, dict(n=0), b"bad argument"),
           (nn, dict(ld_out=19), b"ld_out"), (nn, dict(n=18, ld_out=18), b"ld_out"), (nn, dict(epi=4), b"epi"),
           (nn, dict(epi=-1), b"epi"), (nn, dict(epi=1, e=None), b"need e"), (nn, dict(epi=2, e=None), b"need e"),
           (nn, dict(lda=64), b"lda"), (nn, dict(batch=32768), b"65535"), (nn, dict(flags=1), b"flags"),
           (nn, dict(flags=L.FLAG_RELPROP_TF32), b"flags"),
           (nk, dict(m=None), b"bad argument"), (nk, dict(x=None), b"bad argument"), (nk, dict(np_=16), b"bad argument"),
           (nk, dict(tr=2), b"transpose"), (nk, dict(epi=2), b"epi"), (nk, dict(epi=3), b"epi"),
           (nk, dict(epi=1, e=None), b"needs e"), (nk, dict(ld_out=127), b"ld_out"), (nk, dict(heads=3), b"ld_out"),
           (nk, dict(ldx=100), b"ldx"), (nk, dict(batch=40000), b"65535"), (nk, dict(flags=L.FLAG_RELPROP_TF32), b"flags")]
    for fn, kw, msg in bad:
        assert fn(**kw) == ARG, (kw, msg)
        assert msg in lib.te_last_error(), (kw, msg, lib.te_last_error())
    for dh in (16, 48):
        assert nn(dh=dh, lda=3 * 2 * dh, ldb=3 * 2 * dh) == UNSUP and b"head_dim" in lib.te_last_error()
    assert nn(epi=2, flags=SP) == UNSUP and b"single-pass" in lib.te_last_error()
    assert nn(epi=3, flags=SP) == UNSUP and b"single-pass" in lib.te_last_error()
    assert nk(dh=32, ldx=192, ld_out=64) == UNSUP and b"head_dim 64" in lib.te_last_error()


# ---- engine-level parity at token counts and head widths the other suites do not run -------------------------------------
BERT_SEQS = [7, 129, 257, 300]
VIT_CASES = [(8, 64), (4, 128)]               # (heads, img): head_dim 32 at N = 65, head_dim 64 at N = 257 (patch 8)


def _rel(a, b):
    b = torch.as_tensor(b).double()
    return ((a.double().cpu() - b).abs().max() / b.abs().max().clamp_min(1e-300)).item()


def _vit_case(heads, img):
    params, h = ovit.init_params("vit_tiny_test", seed=11, rand_affine=True, img=img, patch=8, dim=256, depth=2, heads=heads,
                                 mlp=512, classes=10)
    params = conditioned.condition_vit(params)
    xs = torch.randn(2, 3, img, img, generator=torch.Generator().manual_seed(img))
    ocpu.set_torch_threads()
    ref, ridx, taps = ovit.explain({k: v.double() for k, v in params.items()}, xs.double(), h, return_taps=True)
    ref32, _ = ovit.explain(params, xs, h)
    return params, xs, ref, ridx, taps, max(_rel(ref32[s], ref[s]) for s in range(2))


def _bert_case(seq):
    params, h = obert.init_params(seed=5, vocab=8000, max_pos=320, dim=256, depth=2, heads=4, inter=512, rand_affine=True)
    params = conditioned.condition_bert(params)
    g = torch.Generator().manual_seed(seq)
    ids = torch.randint(1000, 5000, (2, seq), generator=g)
    ids[:, 0], ids[:, -1] = 101, 102
    mask = torch.ones(2, seq, dtype=torch.long)
    mask[1, seq * 3 // 4:] = 0                                 # one row padded over its last quarter
    ocpu.set_torch_threads()
    ref, ridx, taps = obert.explain({k: v.double() for k, v in params.items()}, ids, mask, h, start_layer=0, return_taps=True)
    ref32, _ = obert.explain(params, ids, mask, h, start_layer=0)
    return params, h, ids, mask, ref, ridx, taps, max(_rel(ref32[s], ref[s]) for s in range(2))


@pytest.mark.parametrize("heads,img", VIT_CASES)
def test_vit_cases_are_conditioned(heads, img):
    """The fp32 oracle agrees with the fp64 oracle, so the GPU comparison below has bounds that can fail."""
    err = _vit_case(heads, img)[-1]
    assert err < 1e-4, "regime is not conditioned: fp32 oracle vs fp64 oracle %g" % err


@pytest.mark.parametrize("seq", BERT_SEQS)
def test_bert_cases_are_conditioned(seq):
    err = _bert_case(seq)[-1]
    assert err < 1e-4, "regime is not conditioned: fp32 oracle vs fp64 oracle %g" % err


def _engine_flag_sets():
    L = _lib()
    return [(0, 2e-4), (L.FLAG_ALL_FAST, 5e-3), (L.FLAG_BENCH_DEFAULT, 5e-3)]


@gpu
@pytest.mark.parametrize("heads,img", VIT_CASES)
def test_vit_engine_token_counts_and_head_widths(heads, img):
    """ViT dim 256 at head_dim 32 (N = 65: tcgen05 N x N products next to SIMT N x d ones) and head_dim 64 (N = 257: two
    key tiles, softmax outside the fused epilogue), against the fp64 oracle: class index bit-exact, logits 2e-5, attention
    gradient and attn_cam of every layer and the map 2e-4 (SIMT) / 5e-3 (tensor-core selections) of their maxima."""
    from transformer_explainability_b200.baselines.ViT.ViT_LRP import VisionTransformer
    params, xs, ref, ridx, taps, err_ref = _vit_case(heads, img)
    assert err_ref < 1e-4
    model = VisionTransformer(img_size=img, patch_size=8, embed_dim=256, depth=2, num_heads=heads, mlp_ratio=2.,
                              qkv_bias=True, num_classes=10)
    model.load_state_dict(params)
    model = model.cuda().eval()
    eng = model.engine()
    for flags, tol in _engine_flag_sets():
        maps, idx, logits = eng.explain(xs.cuda(), flags=flags, return_logits=True)
        torch.cuda.synchronize()
        assert torch.equal(idx.cpu().long(), ridx)
        e_logit = _rel(logits, taps["logits"])
        e_g = [_rel(b.attn.get_attn_gradients(), taps["grads"][l]) for l, b in enumerate(model.blocks)]
        e_c = [_rel(b.attn.get_attn_cam(), taps["cams"][l]) for l, b in enumerate(model.blocks)]
        e_map = max(_rel(maps[s], ref[s]) for s in range(2))
        print("vit heads %d img %d flags %d: logits %.1e | attn_grad %s | attn_cam %s | map %.1e (fp32 oracle %.1e)" % (
            heads, img, flags, e_logit, ["%.1e" % v for v in e_g], ["%.1e" % v for v in e_c], e_map, err_ref))
        assert e_logit < 2e-5
        assert max(e_g) < tol and max(e_c) < tol and e_map < tol


@gpu
@pytest.mark.parametrize("seq", BERT_SEQS)
def test_bert_engine_sequence_lengths(seq):
    """BERT hidden 256, 4 heads, 2 layers, start_layer 0, batch 2 with one row padded over its last quarter, at sequence
    lengths below one tile, just past it, one past the fused-softmax limit, and 300.  Same bounds as the ViT case; the
    padded tokens' relevance is exactly 0."""
    transformers = pytest.importorskip("transformers")
    from transformer_explainability_b200.BERT_explainability.modules.BERT.BertForSequenceClassification import \
        BertForSequenceClassification
    params, heads, ids, mask, ref, ridx, taps, err_ref = _bert_case(seq)
    assert err_ref < 1e-4
    cfg = transformers.BertConfig(hidden_size=256, num_hidden_layers=2, num_attention_heads=heads, intermediate_size=512,
                                  vocab_size=8000, max_position_embeddings=320, num_labels=2)
    model = BertForSequenceClassification(cfg)
    res = model.load_state_dict({k: v.float() for k, v in params.items()}, strict=False)
    assert not res.unexpected_keys and all("position_ids" in k for k in res.missing_keys)
    model = model.cuda().eval()
    eng = model.engine()
    layers = model.bert.encoder.layer
    for flags, tol in _engine_flag_sets():
        maps, idx, logits = eng.explain(ids.cuda(), mask.cuda(), start_layer=0, flags=flags, return_logits=True)
        torch.cuda.synchronize()
        assert torch.equal(idx.cpu().long(), ridx)
        e_logit = _rel(logits, taps["logits"])
        e_g = [_rel(l.attention.self.get_attn_gradients(), taps["grads"][i]) for i, l in enumerate(layers)]
        e_c = [_rel(l.attention.self.get_attn_cam(), taps["cams"][i]) for i, l in enumerate(layers)]
        e_map = max(_rel(maps[s], ref[s]) for s in range(2))
        print("bert S=%d flags %d: logits %.1e | attn_grad %s | attn_cam %s | map %.1e (fp32 oracle %.1e)" % (
            seq, flags, e_logit, ["%.1e" % v for v in e_g], ["%.1e" % v for v in e_c], e_map, err_ref))
        assert e_logit < 2e-5
        assert max(e_g) < tol and max(e_c) < tol and e_map < tol
        assert float(maps[1, seq * 3 // 4:].abs().max()) == 0.0
