// C-ABI wrappers for the stand-alone rules and rollout entry points declared in include/te_b200.h.
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <string>

#include "../../include/te_b200.h"
#include "te_kernels.h"
#include "te_rollout.h"
#include "te_zplus.h"
#include "te_gemm_tc.h"
#include "te_engine_util.h"

static thread_local std::string g_last_error;
void te_set_last_error(const char* msg) { g_last_error = msg ? msg : ""; }

static std::atomic<long long> g_launches{0};
void te_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" long long te_kernel_launch_count(void) { return g_launches.load(); }

extern "C" const char* te_last_error(void) { return g_last_error.c_str(); }
extern "C" int te_version(void) { return 100; }

#define ST(s) reinterpret_cast<cudaStream_t>(s)
#define REQ(c, msg) do { if (!(c)) { te_set_last_error(msg); return TE_ERR_ARG; } } while (0)

static TeGemm g0(int nb) {
    TeGemm p;
    memset(&p, 0, sizeof(p));
    p.nb1 = nb; p.nb2 = 1; p.alpha = 1.f;
    return p;
}

extern "C" int te_linear_forward(const float* x, const float* w, const float* bias, float* y, int rows,
                                 int in_features, int out_features, void* stream) {
    REQ(x && w && y && rows > 0 && in_features > 0 && out_features > 0, "te_linear_forward: bad argument");
    TeGemm p = g0(1);
    p.A = x; p.lda = in_features; p.B = w; p.ldb = in_features; p.C = y; p.ldc = out_features; p.bias = bias;
    p.M = rows; p.N = out_features; p.K = in_features;
    return te_gemm_launch(p, TE_L_K, TE_L_K, TE_XF_NONE, TE_EPI_BIAS, ST(stream));
}

extern "C" int te_linear_forward_ex(const float* x, const float* w, const float* bias, float* y, float* scratch, int rows,
                                    int in_features, int out_features, unsigned flags, void* stream) {
    REQ(x && w && y && rows > 0 && in_features > 0 && out_features > 0, "te_linear_forward_ex: bad argument");
    if ((flags & TE_FLAG_LINEAR_TENSOR_CORES) && (flags & TE_FLAG_LINEAR_F16_SPLIT) && scratch &&
        te_tc_fwd16_supported(rows, in_features, out_features, in_features)) {
        // scratch layout with both flags: [16*in*out derived | round_up(rows*in,64) fp16 hi,lo split of x | rows*ceil(in/128) block scales]
        TE_TRY(te_tc_prepare_weights(w, scratch, in_features, out_features, ST(stream)));
        float* split = scratch + te_tc_derived_floats(in_features, out_features);
        float* scale = split + (((long long)rows * in_features + 63) & ~63LL);
        return te_tc_linear_fwd16(x, in_features, split, scale, scratch, in_features, out_features, bias, y, nullptr, nullptr,
                                  rows, TE_TC_EPI_BIAS, ST(stream));
    }
    if ((flags & TE_FLAG_LINEAR_TENSOR_CORES) && scratch && te_tc_gemm3x_supported(rows, in_features, out_features, in_features)) {
        TE_TRY(te_tc_prepare_weights(w, scratch, in_features, out_features, ST(stream)));
        return te_tc_linear_fwd(x, in_features, scratch, in_features, out_features, bias, y, nullptr, nullptr, rows,
                                TE_TC_EPI_BIAS, ST(stream));
    }
    return te_linear_forward(x, w, bias, y, rows, in_features, out_features, stream);
}

extern "C" int te_f16_block_split(const float* x, int rows, int cols, void* hi, void* lo, float* scale_inv, void* stream) {
    REQ(x && hi && lo && scale_inv && rows > 0 && cols > 0 && cols % 4 == 0, "te_f16_block_split: bad argument");
    REQ(reinterpret_cast<char*>(lo) == reinterpret_cast<char*>(hi) + (long long)rows * cols * 2,
        "te_f16_block_split: lo must follow hi ([hi | lo] in one buffer, as the kernels lay the split out)");
    return te_tc_blocksplit_f16(x, cols, rows, cols, reinterpret_cast<float*>(hi), scale_inv, ST(stream));
}

extern "C" int te_linear_backward_ex(const float* dy, const float* w, float* dx, float* scratch, int rows, int in_features,
                                     int out_features, unsigned flags, void* stream) {
    REQ(dy && w && dx && rows > 0 && in_features > 0 && out_features > 0, "te_linear_backward_ex: bad argument");
    if ((flags & TE_FLAG_LINEAR_TENSOR_CORES) && scratch && te_tc_gemm3x_supported(rows, out_features, in_features, out_features)) {
        TE_TRY(te_tc_prepare_weights(w, scratch, in_features, out_features, ST(stream)));
        if ((flags & TE_FLAG_BACKWARD_F16) && te_tc_f16_single_supported(rows, out_features, in_features, out_features)) {
            // scratch layout with the flag: [16*in*out derived | round_up(rows*out/2,64) fp16 dy | rows*ceil(out/128) block scales]
            float* split = scratch + te_tc_derived_floats(in_features, out_features);
            float* scale = split + (((long long)rows * out_features / 2 + 63) & ~63LL);
            return te_tc_linear_bwd16(dy, out_features, split, scale, scratch, in_features, out_features, dx, nullptr, rows,
                                      TE_TC_EPI_STORE, ST(stream));
        }
        if ((flags & TE_FLAG_BACKWARD_TF32) && te_tc_pair_supported(rows, out_features, in_features, out_features))
            return te_tc_pair_linear_bwd(dy, out_features, scratch, in_features, out_features, dx, nullptr, rows, TE_TC_EPI_STORE,
                                         ST(stream));
        return te_tc_linear_bwd(dy, scratch, in_features, out_features, dx, nullptr, rows, TE_TC_EPI_STORE, ST(stream));
    }
    TeGemm p = g0(1);
    p.A = dy; p.lda = out_features; p.B = w; p.ldb = in_features; p.C = dx; p.ldc = in_features;
    p.M = rows; p.N = in_features; p.K = out_features;
    return te_gemm_launch(p, TE_L_K, TE_L_MN, TE_XF_NONE, TE_EPI_STORE, ST(stream));
}

extern "C" int te_linear_relprop(const float* x, const float* w, const float* r, float* out, float* scratch, int rows,
                                 int in_features, int out_features, unsigned flags, void* stream) {
    REQ(x && w && r && out && scratch && rows > 0 && in_features > 0 && out_features > 0, "te_linear_relprop: bad argument");
    if (flags & TE_FLAG_RULES_LRP)
        return te_zplus_linear_relprop_lrp(x, in_features, w, r, out_features, out, scratch, rows, in_features, out_features,
                                           ST(stream));
    const float* derived = nullptr;
    if ((flags & TE_FLAG_ZPLUS_TENSOR_CORES) && te_tc_zplus_supported(rows, in_features, out_features, in_features)) {
        // scratch layout with the flag: [rows*out S | 16*in*out derived weight copies]
        float* d = scratch + (((long long)rows * out_features + 63) & ~63LL);
        TE_TRY(te_tc_prepare_weights(w, d, in_features, out_features, ST(stream)));
        derived = d;
    }
    return te_zplus_linear_relprop(x, in_features, w, derived, r, out, scratch, rows, in_features, out_features,
                                   ST(stream));
}

extern "C" int te_linear_relprop_ex(const float* x, const float* w, const float* bias, const float* y, const float* r,
                                    float* out, float* scratch, int rows, int in_features, int out_features,
                                    unsigned flags, void* stream) {
    REQ(x && w && r && out && scratch && rows > 0 && in_features > 0 && out_features > 0, "te_linear_relprop_ex: bad argument");
    const float* derived = nullptr;
    float* xabs = nullptr;
    if ((flags & TE_FLAG_ZPLUS_TENSOR_CORES) && te_tc_zplus_supported(rows, in_features, out_features, in_features)) {
        // scratch layout with the flag: [rows*out S (64-float aligned) | 16*in*out derived weight copies | rows*in tf32(|x|)]
        float* d = scratch + (((long long)rows * out_features + 63) & ~63LL);
        TE_TRY(te_tc_prepare_weights(w, d, in_features, out_features, ST(stream)));
        derived = d;
        xabs = d + te_tc_derived_floats(in_features, out_features);
    }
    return te_zplus_linear_relprop_ldr(x, in_features, w, derived, r, out_features, out, scratch, rows, in_features,
                                       out_features, ST(stream), y, out_features, bias,
                                       ((flags & TE_FLAG_ZPLUS_BF16) ? 1 : 0) | ((flags & TE_FLAG_ZPLUS_S1_BF16) ? 2 : 0) |
                                           ((flags & TE_FLAG_ZPLUS_R_F16) ? 4 : 0),
                                       0, xabs);
}

extern "C" int te_add_relprop(const float* x1, const float* x2, const float* r, float* r1, float* r2, void* scratch,
                              int batch, long long per_sample, void* stream) {
    REQ(x1 && x2 && r && r1 && r2 && batch > 0 && per_sample > 0, "te_add_relprop: bad argument");
    return te_launch_add_relprop(x1, x2, r, r1, r2, reinterpret_cast<double*>(scratch), batch, per_sample, ST(stream));
}

extern "C" int te_clone_relprop(const float* x, const float* r1, const float* r2, const float* r3, float* out,
                                long long n, void* stream) {
    REQ(x && r1 && r2 && out && n > 0, "te_clone_relprop: bad argument");
    return te_launch_clone_relprop(x, r1, r2, r3, out, n, ST(stream));
}

extern "C" int te_index_select_relprop(const float* x, const float* r, float* out, int batch, int n, int d,
                                       void* stream) {
    REQ(x && r && out && batch > 0 && n > 0 && d > 0, "te_index_select_relprop: bad argument");
    return te_launch_index_select_relprop(x, r, nullptr, out, batch, n, d, ST(stream));
}

extern "C" int te_matmul_av_relprop(const float* p_, const float* v, const float* r, float* rp, float* rv,
                                    float* scratch, int bh, int n, int d, void* stream) {
    REQ(p_ && v && r && rp && rv && scratch && bh > 0 && n > 0 && d > 0 && d % 4 == 0, "te_matmul_av_relprop: bad argument");
    cudaStream_t st = ST(stream);
    const long long nn = (long long)n * n, nd = (long long)n * d;
    // Z = P V
    TeGemm g = g0(bh);
    g.A = p_; g.lda = n; g.sA1 = nn; g.B = v; g.ldb = d; g.sB1 = nd; g.C = scratch; g.ldc = d; g.sC1 = nd;
    g.M = n; g.N = d; g.K = n;
    TE_TRY(te_gemm_launch(g, TE_L_K, TE_L_MN, TE_XF_NONE, TE_EPI_STORE, st));
    // S = sd(R, Z)
    TE_TRY(te_launch_sd(r, scratch, scratch, (long long)bh * nd, st));
    // R_P = P * (S V^T)
    g = g0(bh);
    g.A = scratch; g.lda = d; g.sA1 = nd; g.B = v; g.ldb = d; g.sB1 = nd; g.C = rp; g.ldc = n; g.sC1 = nn;
    g.E0 = p_; g.lde0 = n; g.sE1 = nn; g.M = n; g.N = n; g.K = d;
    TE_TRY(te_gemm_launch(g, TE_L_K, TE_L_K, TE_XF_NONE, TE_EPI_MUL, st));
    // R_V = V * (P^T S)
    g = g0(bh);
    g.A = p_; g.lda = n; g.sA1 = nn; g.B = scratch; g.ldb = d; g.sB1 = nd; g.C = rv; g.ldc = d; g.sC1 = nd;
    g.E0 = v; g.lde0 = d; g.sE1 = nd; g.M = n; g.N = d; g.K = n;
    TE_TRY(te_gemm_launch(g, TE_L_MN, TE_L_MN, TE_XF_NONE, TE_EPI_MUL, st));
    return TE_OK;
}

extern "C" int te_matmul_qk_relprop(const float* q, const float* k, const float* r, float* rq, float* rk,
                                    float* scratch, int bh, int n, int d, void* stream) {
    REQ(q && k && r && rq && rk && scratch && bh > 0 && n > 0 && d > 0, "te_matmul_qk_relprop: bad argument");
    cudaStream_t st = ST(stream);
    const long long nn = (long long)n * n, nd = (long long)n * d;
    // S = sd(R, Q K^T)
    TeGemm g = g0(bh);
    g.A = q; g.lda = d; g.sA1 = nd; g.B = k; g.ldb = d; g.sB1 = nd; g.C = scratch; g.ldc = n; g.sC1 = nn;
    g.E0 = r; g.lde0 = n; g.sE1 = nn; g.M = n; g.N = n; g.K = d;
    TE_TRY(te_gemm_launch(g, TE_L_K, TE_L_K, TE_XF_NONE, TE_EPI_SD, st));
    // R_Q = Q * (S K)
    g = g0(bh);
    g.A = scratch; g.lda = n; g.sA1 = nn; g.B = k; g.ldb = d; g.sB1 = nd; g.C = rq; g.ldc = d; g.sC1 = nd;
    g.E0 = q; g.lde0 = d; g.sE1 = nd; g.M = n; g.N = d; g.K = n;
    TE_TRY(te_gemm_launch(g, TE_L_K, TE_L_MN, TE_XF_NONE, TE_EPI_MUL, st));
    // R_K = K * (S^T Q)
    g = g0(bh);
    g.A = scratch; g.lda = n; g.sA1 = nn; g.B = q; g.ldb = d; g.sB1 = nd; g.C = rk; g.ldc = d; g.sC1 = nd;
    g.E0 = k; g.lde0 = d; g.sE1 = nd; g.M = n; g.N = d; g.K = n;
    TE_TRY(te_gemm_launch(g, TE_L_MN, TE_L_MN, TE_XF_NONE, TE_EPI_MUL, st));
    return TE_OK;
}

// ---- attention-shaped contractions through the engines' dispatch (te_engine_util.h), for kernel unit tests -------------
static const unsigned kAttnFlags = TE_FLAG_ATTN_TENSOR_CORES | TE_FLAG_RELPROP_TF32;

extern "C" int te_attention_nn(const float* a, int lda, const float* b, int ldb, int batch, int heads, int n, int head_dim,
                               const float* e, float* out, int ld_out, float alpha, int epi, unsigned flags, void* stream) {
    REQ(a && b && out && batch > 0 && heads > 0 && n > 0 && head_dim > 0, "te_attention_nn: bad argument");
    REQ(epi >= TE_ATTN_STORE && epi <= TE_ATTN_SOFTMAX, "te_attention_nn: epi out of range");
    REQ(e || epi == TE_ATTN_STORE || epi == TE_ATTN_SOFTMAX, "te_attention_nn: MUL / SD need e");
    REQ(lda >= heads * head_dim && ldb >= heads * head_dim, "te_attention_nn: lda / ldb < heads * head_dim");
    REQ(ld_out >= ((n + 3) & ~3), "te_attention_nn: ld_out < round_up(n, 4)");
    REQ((long long)batch * heads <= 65535, "te_attention_nn: batch * heads > 65535");
    REQ((flags & ~kAttnFlags) == 0 && (flags == 0 || (flags & TE_FLAG_ATTN_TENSOR_CORES)),
        "te_attention_nn: flags other than TE_FLAG_ATTN_TENSOR_CORES [| TE_FLAG_RELPROP_TF32]");
    const bool tc = (flags & TE_FLAG_ATTN_TENSOR_CORES) != 0, tf32 = (flags & TE_FLAG_RELPROP_TF32) != 0;
    if (tc) {
        // no SIMT stand-in for a shape the tcgen05 kernels do not take: a passing test must have run them
        if (head_dim != 32 && head_dim != 64) { te_set_last_error("te_attention_nn: tcgen05 kernels take head_dim 32 / 64"); return TE_ERR_UNSUPPORTED; }
        if (tf32 && epi != TE_ATTN_STORE && epi != TE_ATTN_MUL) {
            te_set_last_error("te_attention_nn: the single-pass form has STORE / MUL epilogues only");
            return TE_ERR_UNSUPPORTED;
        }
        if (!te_tc_attn_supported(n, head_dim, lda, ldb, ld_out)) {
            te_set_last_error("te_attention_nn: shape / strides not supported by the tcgen05 kernel (or no driver)");
            return TE_ERR_UNSUPPORTED;
        }
    }
    cudaStream_t st = ST(stream);
    if (epi == TE_ATTN_SOFTMAX) return te_util::attn_probs(tc, batch, heads, n, ld_out, head_dim, a, lda, b, ldb, out, alpha, st);
    const int gepi = (epi == TE_ATTN_STORE) ? TE_EPI_STORE : (epi == TE_ATTN_MUL) ? TE_EPI_MUL : TE_EPI_SD;
    return te_util::attn_nn(tc, batch, heads, n, ld_out, head_dim, a, lda, b, ldb, out, e, alpha, gepi, st, tf32);
}

extern "C" int te_attention_nk(const float* map, int np, int transpose, const float* x, int ldx, int batch, int heads, int n,
                               int head_dim, const float* e, float* out, int ld_out, float alpha, int epi, unsigned flags,
                               void* stream) {
    REQ(map && x && out && batch > 0 && heads > 0 && n > 0 && head_dim > 0 && np >= n, "te_attention_nk: bad argument");
    REQ(transpose == 0 || transpose == 1, "te_attention_nk: transpose is 0 or 1");
    REQ(epi == TE_ATTN_STORE || epi == TE_ATTN_MUL, "te_attention_nk: epi out of range (STORE / MUL)");
    REQ(e || epi == TE_ATTN_STORE, "te_attention_nk: MUL needs e");
    REQ(ldx >= heads * head_dim, "te_attention_nk: ldx < heads * head_dim");
    REQ(ld_out >= heads * head_dim, "te_attention_nk: ld_out < heads * head_dim");
    REQ((long long)batch * heads <= 65535, "te_attention_nk: batch * heads > 65535");
    REQ((flags & ~kAttnFlags) == 0 && (flags == 0 || (flags & TE_FLAG_ATTN_TENSOR_CORES)),
        "te_attention_nk: flags other than TE_FLAG_ATTN_TENSOR_CORES [| TE_FLAG_RELPROP_TF32]");
    const bool tc = (flags & TE_FLAG_ATTN_TENSOR_CORES) != 0, tf32 = (flags & TE_FLAG_RELPROP_TF32) != 0;
    if (tc) {
        if (head_dim != 64) { te_set_last_error("te_attention_nk: the tcgen05 kernel takes head_dim 64"); return TE_ERR_UNSUPPORTED; }
        if (!te_tc_attn_nk_supported(n, head_dim, np, ldx, ld_out)) {
            te_set_last_error("te_attention_nk: shape / strides not supported by the tcgen05 kernel (or no driver)");
            return TE_ERR_UNSUPPORTED;
        }
    }
    return te_util::attn_nk(tc, batch, heads, n, np, head_dim, map, transpose, x, ldx, out, ld_out, e, alpha,
                            epi == TE_ATTN_STORE ? TE_EPI_STORE : TE_EPI_MUL, ST(stream), tf32);
}

static int g_cls_rows = 1;
bool te_engine_cls_rows() { return g_cls_rows != 0; }
void te_engine_set_cls_rows(int on) { g_cls_rows = on ? 1 : 0; }
static int g_gelu_split = -1;
bool te_engine_gelu_split() {
    if (g_gelu_split < 0) {
        const char* e = getenv("TE_B200_GELU_SPLIT");
        g_gelu_split = (e && e[0] == '0') ? 0 : 1;
    }
    return g_gelu_split != 0;
}
void te_engine_set_gelu_split(int on) { g_gelu_split = on ? 1 : 0; }

extern "C" int te_set_option(const char* name, int value) {
    REQ(name != nullptr, "te_set_option: null name");
    if (strcmp(name, "zplus_pair_kernels") == 0) { te_tc_set_pair_kernels(value); return TE_OK; }
    if (strcmp(name, "linear_pair_kernels") == 0) { te_tc_set_pair_linear(value); return TE_OK; }
    if (strcmp(name, "attn_persistent") == 0) { te_tc_set_attn_persistent(value); return TE_OK; }
    if (strcmp(name, "linear_mixed") == 0) { te_tc_set_mixed_linear(value); return TE_OK; }
    if (strcmp(name, "zplus_persistent") == 0) { te_tc_set_zplus_persistent(value); return TE_OK; }
    if (strcmp(name, "cls_row_top_block") == 0) { te_engine_set_cls_rows(value); return TE_OK; }
    if (strcmp(name, "gelu_split_fused") == 0) { te_engine_set_gelu_split(value); return TE_OK; }
    te_set_last_error("te_set_option: unknown option");
    return TE_ERR_ARG;
}

extern "C" int te_relevance_heatmap(const float* maps, int batch, int grid, int scale, float* out, void* stream) {
    REQ(maps && out && batch > 0 && grid > 0 && scale > 0, "te_relevance_heatmap: bad argument");
    return te_launch_relevance_heatmap(maps, out, batch, grid, scale, ST(stream));
}

// ---- head reductions of the secondary methods ------------------------------------------------------------
extern "C" int te_head_reduce(const float* a, const float* g, const float* head_w, int batch, int heads, int n, int ld,
                              int mode, float* out, void* stream) {
    REQ(a && out && batch > 0 && heads > 0 && n > 0 && ld >= n && mode >= 0 && mode <= 2, "te_head_reduce: bad argument");
    return te_launch_head_reduce(a, g, head_w, out, batch, heads, n, ld, mode, ST(stream));
}
extern "C" int te_head_region_mean(const float* g, int batch, int heads, int n, int ld, int r0, int r1, int c0, int c1,
                                   float* out, void* stream) {
    REQ(g && out && batch > 0 && heads > 0 && n > 0 && ld >= n, "te_head_region_mean: bad argument");
    return te_launch_head_region_mean(g, out, batch * heads, n, ld, r0, r1, c0, c1, ST(stream));
}

// ---- rollout -------------------------------------------------------------------------------------
static long long ro_align(long long bytes) { return ((bytes + 255) / 256) * 256; }

extern "C" long long te_rollout_workspace_bytes(int layers, int batch, int n) {
    if (layers <= 0 || batch <= 0 || n <= 0) return TE_ERR_ARG;
    const long long ld = (n + 3) & ~3;
    return ro_align((long long)layers * batch * n * ld * 4) + 2 * ro_align((long long)batch * n * ld * 4) +
           ro_align((long long)layers * batch * n * 4);
}

static int ro_carve(void* workspace, long long bytes, int layers, int batch, int n, float** mats, float** ja,
                    float** jb, int* ld, float** diag = nullptr) {
    REQ(workspace && (((uintptr_t)workspace) & 255u) == 0, "rollout: workspace null or not 256-byte aligned");
    if (te_rollout_workspace_bytes(layers, batch, n) > bytes) { te_set_last_error("rollout: workspace too small"); return TE_ERR_WORKSPACE; }
    *ld = (n + 3) & ~3;
    char* b = reinterpret_cast<char*>(workspace);
    *mats = reinterpret_cast<float*>(b);
    b += ro_align((long long)layers * batch * n * (*ld) * 4);
    *ja = reinterpret_cast<float*>(b);
    b += ro_align((long long)batch * n * (*ld) * 4);
    *jb = reinterpret_cast<float*>(b);
    b += ro_align((long long)batch * n * (*ld) * 4);
    if (diag) *diag = reinterpret_cast<float*>(b);
    return TE_OK;
}

// ---- first layer: Conv2d z^B rule / PatchEmbed.relprop (layers_ours.py:242-259, ViT_LRP.py:238-242) ----------------
extern "C" long long te_patch_embed_relprop_workspace_bytes(int batch, int in_chans, int img_size, int patch_size, int dim) {
    if (batch <= 0 || in_chans <= 0 || patch_size <= 0 || img_size % patch_size != 0 || dim <= 0) return TE_ERR_ARG;
    return te_patch_relprop_scratch_floats(batch, in_chans, img_size, patch_size, dim) * 4 + 256;
}
extern "C" int te_patch_embed_relprop(const float* images, const float* weight, const float* r, int batch, int in_chans,
                                      int img_size, int patch_size, int dim, float* r_pixels, float* r_sum, void* workspace,
                                      long long workspace_bytes, void* stream) {
    REQ(images && weight && r && (r_pixels || r_sum) && batch > 0, "te_patch_embed_relprop: bad argument");
    REQ(workspace && (((uintptr_t)workspace) & 255u) == 0, "te_patch_embed_relprop: workspace null or not 256-byte aligned");
    const long long need = te_patch_embed_relprop_workspace_bytes(batch, in_chans, img_size, patch_size, dim);
    if (need < 0) { te_set_last_error("te_patch_embed_relprop: bad shape"); return TE_ERR_ARG; }
    if (need > workspace_bytes) { te_set_last_error("te_patch_embed_relprop: workspace too small"); return TE_ERR_WORKSPACE; }
    const long long np = (long long)(img_size / patch_size) * (img_size / patch_size);
    return te_patch_relprop_run(images, weight, r, np * dim, batch, in_chans, img_size, patch_size, dim,
                                reinterpret_cast<float*>(workspace), r_pixels, r_sum, ST(stream));
}

extern "C" int te_attribution_rollout(const float* grad, const float* cam, int layers, int batch, int heads, int n,
                                      int ld, int start_layer, int normalize, unsigned flags, float* joint,
                                      float* row0, void* workspace, long long workspace_bytes, void* stream) {
    REQ(grad && cam && layers > 0 && batch > 0 && heads > 0 && n > 0 && ld >= n, "te_attribution_rollout: bad argument");
    float *mats, *ja, *jb, *diag;
    int ldw;
    TE_TRY(ro_carve(workspace, workspace_bytes, layers, batch, n, &mats, &ja, &jb, &ldw, &diag));
    return te_rollout_layers(grad, cam, (long long)batch * heads * n * ld, layers, batch, heads, n, ld, ldw, start_layer,
                             normalize, flags, mats, ja, jb, joint, row0, /*first=*/0, /*bert_fix=*/0, ST(stream), diag);
}

extern "C" int te_compute_rollout_attention(const float* mats_in, int layers, int batch, int n, int start_layer,
                                            int normalize, float* joint, void* workspace, long long workspace_bytes,
                                            void* stream) {
    REQ(mats_in && joint && layers > 0 && batch > 0 && n > 0 && start_layer >= 0 && start_layer < layers,
        "te_compute_rollout_attention: bad argument");
    float *mats, *ja, *jb;
    int ldw;
    TE_TRY(ro_carve(workspace, workspace_bytes, layers, batch, n, &mats, &ja, &jb, &ldw));
    cudaStream_t st = ST(stream);
    TE_TRY(te_launch_prep_mats(mats_in, mats, (long long)layers * batch * n, n, n, ldw, normalize, st));
    const float* res = nullptr;
    TE_TRY(te_rollout_chain(mats, layers, batch, n, ldw, start_layer, ja, jb, &res, st));
    if (cudaMemcpy2DAsync(joint, sizeof(float) * n, res, sizeof(float) * ldw, sizeof(float) * n, (size_t)batch * n,
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
        te_set_last_error("te_compute_rollout_attention: copy failed");
        return TE_ERR_CUDA;
    }
    return TE_OK;
}
