/* te_b200 — C ABI of the B200-native transformer-attribution engine.
 *
 * Drop-in boundary for the `transformer_attribution` path of hila-chefer/Transformer-Explainability.
 * The reference has no FFI: its interface for this path is a Python "relprop protocol"
 * (every layer has forward()/relprop(R, alpha); generators call model(x) -> backward -> model.relprop()).
 * Each entry point below names the reference interface (file:line under /root/reference) it replaces.
 *
 * Conventions
 *  - all tensors are contiguous row-major fp32 in DEVICE memory, borrowed from the caller
 *    (the library never allocates or frees caller memory; scratch comes from a caller `workspace`
 *    whose size is queried with the matching *_workspace_bytes function);
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *  - return value: 0 = ok, negative = error (TE_ERR_*); te_last_error() returns a message.
 *    No exceptions cross the boundary; there is NO CPU fallback: a missing GPU is an error;
 *  - a "batch" is a set of INDEPENDENT B=1 explanations: every reduction the reference does over
 *    a whole B=1 tensor (Add.relprop's sums) is done per sample.
 */
#ifndef TE_B200_H
#define TE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TE_API __attribute__((visibility("default")))
#else
#define TE_API
#endif

#define TE_OK 0
#define TE_ERR_ARG (-1)
#define TE_ERR_WORKSPACE (-2)
#define TE_ERR_CUDA (-3)
#define TE_ERR_UNSUPPORTED (-4)

/* te_vit_attribute / te_vit_explain flags */
#define TE_FLAG_ZPLUS_TENSOR_CORES 1u /* z+ Linear-rule GEMMs on tcgen05 (TF32 in, fp32 acc) instead of fp32 SIMT */
#define TE_FLAG_ROLLOUT_FUSED 2u      /* single fused aggregation+rollout kernel instead of aggregate + bmm chain */
#define TE_FLAG_KEEP_ALL_CAMS 4u      /* run the relprop below start_layer too (accessor parity with the reference) */
#define TE_FLAG_LINEAR_TENSOR_CORES 16u /* forward / backward Linear GEMMs on tcgen05 with the fp32-grade 3xTF32 split */
#define TE_FLAG_ATTN_TENSOR_CORES 32u  /* the N x N attention contractions (QK^T, dctx V^T, S2 V^T) on tcgen05, 3xTF32 */
#define TE_FLAG_ZPLUS_BF16 64u          /* with TE_FLAG_ZPLUS_TENSOR_CORES: S = R/Z stored as bf16 and the second z+ contraction
                                         (R_in = x+ (S W+) + x- (S W-)) on tcgen05 kind::f16 with bf16 operands */
#define TE_FLAG_GRADIENTS_ONLY 128u    /* te_*_attribute stops after the class-gradient backward: only "attn_grad" of the layers
                                         >= start_layer is produced (maps may be NULL) — the attention-GradCAM baselines */
#define TE_FLAG_BACKWARD_TF32 256u     /* with TE_FLAG_LINEAR_TENSOR_CORES: the activation-gradient backward Linears run as
                                         single-pass TF32 GEMMs (persistent CTA-pair kernel) instead of the 3xTF32 split.
                                         The gradients only enter the result linearly (relu(G * cam)), never a
                                         safe_divide denominator: measured effect in profiles/ (r02 parity table) */
#define TE_FLAG_RELPROP_TF32 1024u     /* with TE_FLAG_ATTN_TENSOR_CORES: the attention-shaped contractions of the relprop whose
                                         result is relevance (attn_cam = P * (S V^T) / 2, P^T S, S1 K, S1^T Q) run single-pass
                                         TF32 like the z+ rule does; the denominator Q K^T keeps the 3xTF32 split */
#define TE_FLAG_ZPLUS_S1_BF16 2048u    /* with TE_FLAG_ZPLUS_TENSOR_CORES: the |x| |W|^T term of the single-pass z+ denominator with bf16
                                         operands (a sum of K non-negative products: rounding errors average to ~2^-9 / sqrt(K)) */
#define TE_FLAG_LINEAR_F16_SPLIT 4096u  /* with TE_FLAG_LINEAR_TENSOR_CORES: the forward Linears on tcgen05 kind::f16 with a row-scaled
                                         * fp16 (hi, lo) split of both operands (3 MMAs per k-step, same 22-bit operand precision
                                         * as the 3xTF32 split at half the tensor cycles and a third of the staged bytes) */
#define TE_FLAG_ZPLUS_R_F16 8192u        /* with TE_FLAG_ZPLUS_TENSOR_CORES: the second contraction of the z+ rule, x+ (S W+) + x- (S W-), on
                                         * tcgen05 kind::f16: S as block-scaled fp16 (one power of two per row and 128 columns),
                                         * W+^T / W-^T as row-scaled fp16 — the 11 significant bits of the TF32 form, rounded to
                                         * nearest instead of truncated, at twice the tensor rate */
#define TE_FLAG_BACKWARD_F16 16384u      /* with TE_FLAG_LINEAR_TENSOR_CORES: the activation-gradient backward Linears as ONE fp16 MMA per
                                         * k-step (block-scaled fp16 gradients, row-scaled fp16 weights) instead of one TF32 MMA
                                         * (TE_FLAG_BACKWARD_TF32): same 11 significant bits, twice the tensor rate */
#define TE_FLAG_RULES_LRP 512u         /* the rule library of modules/layers_lrp.py (baselines/ViT/ViT_orig_LRP.py) instead of
                                         modules/layers_ours.py: Linear divides its two halves by their OWN denominators
                                         (layers_lrp.py:199-200), Add has no ratio normalisation (:98-100).  fp32 SIMT rules. */
#define TE_FLAG_RELPROP_TO_INPUT 8u   /* finish the lowest block as well: relevance at the encoder input (what
                                         model.relprop() returns in the reference) is left in tensor "relevance_in" */

TE_API const char* te_last_error(void);
/* Process-wide tuning switches (not part of the reference surface).  name = "zplus_pair_kernels": run the z+ Linear rule
 * with the CTA-pair (tcgen05 cta_group::2, 256 x 256 MMA) kernels instead of the single-CTA ones (2: R kernel only);
 * name = "linear_pair_kernels": the same for the 3xTF32 forward / backward Linear GEMMs.  Both default to 0.
 * name = "zplus_persistent": 1 (default) runs the z+ rule with the persistent CTA-pair kernels (te_tc_pair.cu), 0 with
 * the round-1 kernels selected by "zplus_pair_kernels".
 * name = "attn_persistent": 1 runs the fp32-grade N x N attention kernel in its persistent, TMEM-double-buffered form (N <= 224),
 * 0 (default) one tile per CTA, two CTAs per SM.
 * name = "linear_mixed": 1 runs the forward Linears with the mixed-kind split (main term TF32, the two correction terms as bf16
 * MMAs: two thirds of the tensor cycles of the 3xTF32 kernel at the same fp32-grade accuracy), 2 its persistent CTA-pair form
 * (48 KiB staged per k-block instead of 80), 0 with 3xTF32.
 * name = "cls_row_top_block": 1 (default) runs the three z+ rules of the top block on the pooled-token rows only (exact:
 * the relevance entering the top block is zero in every other row), 0 on all rows.
 * Returns TE_OK, or a negative status for an unknown name. */
TE_API int te_set_option(const char* name, int value);
TE_API int te_version(void);
/* number of kernels this library has launched in this process (bench.py reports the delta as gpu_launches) */
TE_API long long te_kernel_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * ViT / DeiT model description  (baselines/ViT/ViT_LRP.py:247-303 VisionTransformer.__init__)
 * ---------------------------------------------------------------------------------------------- */
typedef struct te_vit_config {
    int img_size;     /* 224 */
    int patch_size;   /* 16  */
    int in_chans;     /* 3   */
    int num_classes;  /* 1000 */
    int dim;          /* embed_dim */
    int depth;        /* number of blocks */
    int heads;
    int mlp_dim;      /* int(dim*mlp_ratio) */
    int distilled;    /* 1: extra dist_token + head_dist, logits averaged (DeiT-distilled extension) */
    float eps_block;  /* 1e-6, ViT_LRP.py:184,187 */
    float eps_final;  /* 1e-5, ViT_LRP.py:266 */
} te_vit_config;

/* Frozen weights live in ONE flat fp32 device buffer (also the unit of the NCCL broadcast).
 * Tensor i has the reference state_dict key te_vit_weight_name(i), te_vit_weight_numel(i) floats,
 * and starts at float offset te_vit_weight_offset(i) (every offset is a multiple of 32 floats). */
TE_API int te_vit_num_weights(const te_vit_config* cfg);
TE_API const char* te_vit_weight_name(const te_vit_config* cfg, int i);
TE_API long long te_vit_weight_numel(const te_vit_config* cfg, int i);
TE_API long long te_vit_weight_offset(const te_vit_config* cfg, int i);
TE_API long long te_vit_weight_total(const te_vit_config* cfg); /* floats */

/* Tensor-core copies of the frozen Linear weights (W+, W-, W+^T, W-^T rounded to TF32, all K-major) used by
 * the z+ rule when TE_FLAG_ZPLUS_TENSOR_CORES is set: te_vit_derived_total() floats, filled once per weight
 * load by te_vit_prepare_derived().  `derived` may be NULL when the flag is not used. */
TE_API long long te_vit_derived_total(const te_vit_config* cfg);
TE_API int te_vit_prepare_derived(const te_vit_config* cfg, const float* weights, float* derived, void* stream);

/* Scratch for `batch` samples processed together (activations of every block are kept for the
 * relprop, like the reference's forward hooks, modules/layers_ours.py:16-27). */
TE_API long long te_vit_workspace_bytes(const te_vit_config* cfg, int batch);

/* model(x): VisionTransformer.forward (ViT_LRP.py:305-322).  images [batch,in_chans,img,img];
 * logits [batch,num_classes] (may be NULL).  Leaves every saved activation in `workspace`. */
TE_API int te_vit_forward(const te_vit_config* cfg, const float* weights, const float* derived, const float* images,
                   int batch, unsigned flags, float* logits, void* workspace, long long workspace_bytes, void* stream);

/* The rest of LRP.generate_LRP (ViT_explanation_generator.py:27-41) + VisionTransformer.relprop with
 * method="transformer_attribution" (ViT_LRP.py:324-369) on the activations te_vit_forward left behind:
 * arg-max (where index[b] < 0), one-hot, class gradient of every attention map, LRP relprop through
 * every block >= start_layer, relu(grad*cam) head-mean, +I, rollout, row 0 without the prefix token(s).
 * index [batch] int32 in/out (device); maps [batch, tokens-prefix] (device). */
TE_API int te_vit_attribute(const te_vit_config* cfg, const float* weights, const float* derived, int batch, int* index,
                     int start_layer, unsigned flags, float* maps, void* workspace, long long workspace_bytes,
                     void* stream);

/* te_vit_forward + te_vit_attribute: one call per batch = LRP.generate_LRP for `batch` independent inputs. */
TE_API int te_vit_explain(const te_vit_config* cfg, const float* weights, const float* derived, const float* images,
                   int batch, int* index, int start_layer, unsigned flags, float* maps, float* logits, void* workspace,
                   long long workspace_bytes, void* stream);

/* Accessors into the workspace — get_attn / get_attn_gradients / get_attn_cam / get_v ...
 * (ViT_LRP.py:102-130).  name in {"attn","attn_grad","attn_cam","qkv","x_in","ctx","logits","rollout_mats"}.
 * Returns a device pointer, 4 dims and 4 element strides (unused dims are 1). */
TE_API int te_vit_tensor(const te_vit_config* cfg, int batch, void* workspace, const char* name, int layer,
                  float** ptr, long long dims[4], long long strides[4]);
/* method="full" (ViT_LRP.py:337-343): relevance carried through ``self.add`` (tokens + pos_embed), ``[:, 1:]``,
 * PatchEmbed.relprop (:238-242) and the z^B rule of the patch convolution (layers_ours.py:242-259).
 * Call after te_vit_forward + te_vit_attribute(flags | TE_FLAG_RELPROP_TO_INPUT) on the same workspace and images.
 * pixel_maps [batch, img, img] (channels summed — what relprop returns) and / or pixel_relevance
 * [batch, in_chans, img, img] (Conv2d.relprop's own output) are written when non-NULL. */
TE_API int te_vit_relprop_pixels(const te_vit_config* cfg, const float* weights, const float* images, int batch,
                          float* pixel_maps, float* pixel_relevance, void* workspace, long long workspace_bytes,
                          void* stream);
/* Same with the engine flags of the preceding te_vit_attribute call: TE_FLAG_RULES_LRP selects the layers_lrp Add rule for
 * self.add.relprop (baselines/ViT/ViT_orig_LRP.py, method="full"). */
TE_API int te_vit_relprop_pixels_ex(const te_vit_config* cfg, const float* weights, const float* images, int batch,
                                    unsigned flags, float* pixel_maps, float* pixel_relevance, void* workspace,
                                    long long workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * BERT sequence classifier  (BERT_explainability/modules/BERT/BertForSequenceClassification.py:12-88,
 * BERT.py:533-651; transformers.BertConfig fields)
 * ---------------------------------------------------------------------------------------------- */
typedef struct te_bert_config {
    int vocab_size;       /* 30522 */
    int max_position;     /* 512 */
    int type_vocab;       /* 2 */
    int hidden;           /* 768 */
    int layers;           /* 12 */
    int heads;            /* 12 */
    int intermediate;     /* 3072 */
    int num_labels;       /* 2 */
    float layer_norm_eps; /* 1e-12 */
} te_bert_config;

/* flat fp32 weight buffer keyed by the HF state_dict names (query|key|value of a layer are adjacent and are
 * used as one packed [3*hidden, hidden] weight); derived = tensor-core copies as for ViT. */
TE_API int te_bert_num_weights(const te_bert_config* cfg);
TE_API const char* te_bert_weight_name(const te_bert_config* cfg, int i);
TE_API long long te_bert_weight_numel(const te_bert_config* cfg, int i);
TE_API long long te_bert_weight_offset(const te_bert_config* cfg, int i);
TE_API long long te_bert_weight_total(const te_bert_config* cfg);
TE_API long long te_bert_derived_total(const te_bert_config* cfg);
TE_API int te_bert_prepare_derived(const te_bert_config* cfg, const float* weights, float* derived, void* stream);
TE_API long long te_bert_workspace_bytes(const te_bert_config* cfg, int batch, int seq);

/* model(input_ids, attention_mask)[0]: ids / mask are int64 [batch, seq] (device); token_type_ids = 0,
 * position_ids = arange(seq) as in BERT.py:69-75; logits [batch, num_labels] (may be NULL). */
TE_API int te_bert_forward(const te_bert_config* cfg, const float* weights, const float* derived,
                    const long long* input_ids, const long long* attention_mask, int batch, int seq, unsigned flags,
                    float* logits, void* workspace, long long workspace_bytes, void* stream);
/* The rest of Generator.generate_LRP (ExplanationGenerator.py:33-59): arg-max (index[b] < 0), one-hot, class
 * gradient of every attention_probs, relprop (BertForSequenceClassification.relprop), relu(grad*cam) head mean,
 * +I, row-normalised rollout from start_layer, row 0 with element 0 replaced by the row minimum.
 * maps [batch, seq]. */
TE_API int te_bert_attribute(const te_bert_config* cfg, const float* weights, const float* derived, int batch, int seq,
                      int* index, int start_layer, unsigned flags, float* maps, void* workspace,
                      long long workspace_bytes, void* stream);
TE_API int te_bert_explain(const te_bert_config* cfg, const float* weights, const float* derived,
                    const long long* input_ids, const long long* attention_mask, int batch, int seq, int* index,
                    int start_layer, unsigned flags, float* maps, float* logits, void* workspace,
                    long long workspace_bytes, void* stream);
/* get_attn / get_attn_gradients / get_attn_cam of BertSelfAttention (BERT.py:281-297):
 * name in {"attn","attn_grad","attn_cam","hidden","logits"}. */
TE_API int te_bert_tensor(const te_bert_config* cfg, int batch, int seq, void* workspace, const char* name, int layer,
                   float** ptr, long long dims[4], long long strides[4]);

/* ------------------------------------------------------------------------------------------------
 * Stand-alone LRP rules (modules/layers_ours.py) — the same kernels the engine chains, exported so
 * that each rule can be parity-tested against the reference layer class it replaces.
 * ---------------------------------------------------------------------------------------------- */
/* Linear.relprop, alpha=1 (layers_ours.py:207-230): x [rows,in], w [out,in], r [rows,out] -> out [rows,in].
 * flags & TE_FLAG_RULES_LRP: the layers_lrp variant (modules/layers_lrp.py:187-210, separate denominators).
 * scratch: rows*out floats; with TE_FLAG_ZPLUS_TENSOR_CORES: round_up(rows*out,64) + 16*in*out floats. */
TE_API int te_linear_relprop(const float* x, const float* w, const float* r, float* out, float* scratch, int rows,
                      int in_features, int out_features, unsigned flags, void* stream);
/* Same rule with the Linear's saved forward output y = x W^T + bias [rows,out] supplied (what the engines do): with
 * TE_FLAG_ZPLUS_TENSOR_CORES the denominator is then formed in ONE tensor-core pass through the exact identity
 * x+ W+^T + x- W-^T == ((y - bias) + |x| |W|^T) / 2.  bias may be NULL (no bias).
 * scratch: rows*out floats; with TE_FLAG_ZPLUS_TENSOR_CORES: round_up(rows*out,64) + 16*in*out + rows*in floats
 * (S, the derived weight copies, the tf32(|x|) operand of the single-pass kernel). */
TE_API int te_linear_relprop_ex(const float* x, const float* w, const float* bias, const float* y, const float* r,
                         float* out, float* scratch, int rows, int in_features, int out_features, unsigned flags,
                         void* stream);
/* Add.relprop (layers_ours.py:97-120) per sample: x1,x2,r [batch,per_sample] -> r1,r2.
 * scratch: batch*48 doubles; scratch == NULL selects the layers_lrp variant (modules/layers_lrp.py:48-60,98-100:
 * r1 = x1*sd(r, x1+x2), r2 = x2*sd(r, x1+x2), no ratio normalisation). */
TE_API int te_add_relprop(const float* x1, const float* x2, const float* r, float* r1, float* r2, void* scratch,
                   int batch, long long per_sample, void* stream);
/* Clone.relprop (layers_ours.py:151-169): out = x * (sd(r1,x)+sd(r2,x)[+sd(r3,x)]); r3 may be NULL. */
TE_API int te_clone_relprop(const float* x, const float* r1, const float* r2, const float* r3, float* out, long long n,
                     void* stream);
/* einsum('bhij,bhjd->bhid').relprop (layers_ours.py:48-60,122-127): p [bh,n,n], v [bh,n,d], r [bh,n,d]
 * -> rp [bh,n,n], rv [bh,n,d]  (UN-halved).  scratch: bh*n*d floats. */
TE_API int te_matmul_av_relprop(const float* p, const float* v, const float* r, float* rp, float* rv, float* scratch,
                         int bh, int n, int d, void* stream);
/* einsum('bhid,bhjd->bhij').relprop: q,k [bh,n,d], r [bh,n,n] -> rq, rk [bh,n,d] (UN-halved).
 * scratch: bh*n*n floats. */
TE_API int te_matmul_qk_relprop(const float* q, const float* k, const float* r, float* rq, float* rk, float* scratch,
                         int bh, int n, int d, void* stream);
/* IndexSelect.relprop for token 0 (layers_ours.py:129-147): x [b,n,d], r [b,d] -> out [b,n,d]. */
TE_API int te_index_select_relprop(const float* x, const float* r, float* out, int batch, int n, int d, void* stream);
/* Conv2d.relprop, 3-channel-input (z^B) branch (layers_ours.py:242-259) for a kernel == stride patch convolution, as
 * called by PatchEmbed.relprop (ViT_LRP.py:238-242).  images [batch, in_chans, img, img]; weight [dim, in_chans*patch*patch];
 * r [batch, (img/patch)^2, dim] (token-major: the ``cam`` PatchEmbed.relprop receives).  r_pixels [batch,in_chans,img,img]
 * and / or r_sum [batch,img,img] (channel sum) are written when non-NULL.  Min / max are taken per sample. */
TE_API long long te_patch_embed_relprop_workspace_bytes(int batch, int in_chans, int img_size, int patch_size, int dim);
TE_API int te_patch_embed_relprop(const float* images, const float* weight, const float* r, int batch, int in_chans,
                           int img_size, int patch_size, int dim, float* r_pixels, float* r_sum, void* workspace,
                           long long workspace_bytes, void* stream);

/* generate_visualization's tensor part (example.ipynb:57-60): maps [batch, grid*grid] -> reshape grid x grid -> bilinear
 * x scale (align_corners=False) -> per-sample min-max normalisation -> out [batch, grid*scale, grid*scale]. */
TE_API int te_relevance_heatmap(const float* maps, int batch, int grid, int scale, float* out, void* stream);
/* Head reductions of attention-shaped tensors [batch, heads, n, ld] -> out [batch, n, n] (contiguous), the building
 * block of the secondary methods (ViT_LRP.py:345-398; ViT_explanation_generator.py:51-83; BERT
 * ExplanationGenerator.py:61-155):   v_h = a_h (* g_h if g) (* head_w[b,h] if head_w);
 *   mode 0: mean_h v_h          mode 1: mean_h relu(v_h)  ("clamp(min=0).mean")      mode 2: relu(mean_h v_h). */
TE_API int te_head_reduce(const float* a, const float* g, const float* head_w, int batch, int heads, int n, int ld, int mode,
                   float* out, void* stream);
/* out[b,h] = mean of g[b,h, r0:r1, c0:c1]  (``grad.mean(dim=[1,2])`` of the GradCAM baselines). */
TE_API int te_head_region_mean(const float* g, int batch, int heads, int n, int ld, int r0, int r1, int c0, int c1, float* out,
                        void* stream);

/* ------------------------------------------------------------------------------------------------
 * Aggregation + rollout  (ViT_LRP.py:357-368, :38-49 ; ExplanationGenerator.py:47-59, :7-18)
 * ---------------------------------------------------------------------------------------------- */
/* grad, cam: [layers, batch, heads, n, ld] (ld >= n row stride).  Computes
 * M_l = mean_h relu(grad_l*cam_l) + I (rows normalised if normalize), J = M_{L-1}...M_{start};
 * joint [batch,n,n] (may be NULL) receives J, row0 [batch,n] (may be NULL) receives J[:,0,:]. */
TE_API long long te_rollout_workspace_bytes(int layers, int batch, int n);
TE_API int te_attribution_rollout(const float* grad, const float* cam, int layers, int batch, int heads, int n, int ld,
                           int start_layer, int normalize, unsigned flags, float* joint, float* row0,
                           void* workspace, long long workspace_bytes, void* stream);
/* compute_rollout_attention(all_layer_matrices, start_layer): mats [layers,batch,n,n] -> joint [batch,n,n]. */
TE_API int te_compute_rollout_attention(const float* mats, int layers, int batch, int n, int start_layer, int normalize,
                                 float* joint, void* workspace, long long workspace_bytes, void* stream);

/* Plain Linear GEMMs — exported for kernel unit tests only.  flags & TE_FLAG_LINEAR_TENSOR_CORES selects the
 * tcgen05 3xTF32 path (scratch: 16*in*out floats for the derived weight copies; may be NULL otherwise); with
 * TE_FLAG_LINEAR_F16_SPLIT as well, te_linear_forward_ex runs the fp16-split kernel (scratch: 16*in*out +
 * round_up(rows*in,64) + rows*ceil(in/128) floats). */
TE_API int te_linear_forward(const float* x, const float* w, const float* bias, float* y, int rows, int in_features,
                      int out_features, void* stream);
TE_API int te_linear_forward_ex(const float* x, const float* w, const float* bias, float* y, float* scratch, int rows,
                         int in_features, int out_features, unsigned flags, void* stream);
/* The operand format of the fp16-split forward Linear (TE_FLAG_LINEAR_F16_SPLIT) — exported for unit tests of the format: x [rows, cols]
 * -> hi, lo fp16 [rows, cols] (hi = fp16(2^e x), lo = fp16(2^e x - hi)) and scale_inv [rows, ceil(cols / 128)] = 2^-e, one e per row
 * and 128 columns chosen so that 2^e max|x| lies in [2^14, 2^15) (e = 0 for an all-zero or non-finite block).  cols % 4 == 0. */
TE_API int te_f16_block_split(const float* x, int rows, int cols, void* hi, void* lo, float* scale_inv, void* stream);
TE_API int te_linear_backward_ex(const float* dy, const float* w, float* dx, float* scratch, int rows, int in_features,
                          int out_features, unsigned flags, void* stream);

/* The attention-shaped contractions of the engines, through the engines' own dispatch — exported for kernel unit tests
 * only.  A, B and X are head slices of packed activations [batch*n, ld] (head h at columns h*head_dim ..), addressed in
 * place; rows of one sample follow those of the previous one.
 *   te_attention_nn:  out[b,h,i,j] = epi(alpha * sum_d A[b*n+i, h*head_dim+d] * B[b*n+j, h*head_dim+d])
 *     out and e are [batch, heads, n, ld_out] with ld_out >= round_up(n, 4).  epi: TE_ATTN_STORE, TE_ATTN_MUL (* e),
 *     TE_ATTN_SD (safe_divide(e, .), layers_ours.py:10-13) or TE_ATTN_SOFTMAX (over j; e unused).
 *   te_attention_nk:  out[b*n+m, h*head_dim+c] = epi(alpha * sum_k A_h[m,k] * X[b*n+k, h*head_dim+c])
 *     A_h = map[b,h] (transpose = 0) or its transpose (transpose = 1); map is [batch, heads, n, np] (np >= n), X / out / e
 *     are packed with row strides ldx / ld_out / ld_out.  epi: TE_ATTN_STORE or TE_ATTN_MUL.  The pad columns [n, np) of
 *     map must hold finite values: the tensor-core kernel multiplies them by zero-filled operand rows, and NaN * 0 = NaN.
 * flags: 0 runs the fp32 SIMT kernels; TE_FLAG_ATTN_TENSOR_CORES the tcgen05 3xTF32 kernels (te_set_option
 * "attn_persistent" applies); | TE_FLAG_RELPROP_TF32 their single-pass TF32 form for STORE / MUL, which the N x N
 * dispatch takes for n <= 256 only (beyond that it runs 3xTF32, as the engines do).  With the tensor-core flag a shape or
 * epilogue the tcgen05 kernels do not take (head_dim other than 32 / 64, N x d at head_dim != 64, single-pass SD or
 * SOFTMAX, row strides that are not multiples of 4) returns TE_ERR_UNSUPPORTED instead of running the SIMT kernel.
 * SOFTMAX at n > 256 runs the tensor-core scores followed by the row-softmax kernel. */
#define TE_ATTN_STORE 0
#define TE_ATTN_MUL 1
#define TE_ATTN_SD 2
#define TE_ATTN_SOFTMAX 3
TE_API int te_attention_nn(const float* a, int lda, const float* b, int ldb, int batch, int heads, int n,
                           int head_dim, const float* e, float* out, int ld_out, float alpha, int epi, unsigned flags,
                           void* stream);
TE_API int te_attention_nk(const float* map, int np, int transpose, const float* x, int ldx, int batch, int heads, int n,
                           int head_dim, const float* e, float* out, int ld_out, float alpha, int epi, unsigned flags,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TE_B200_H */
