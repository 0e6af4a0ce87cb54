/* psam_b200 - C ABI of the B200-native Point-SAM hot path.
 *
 * This is the drop-in boundary.  In the reference the native boundary for this path is the pybind11
 * module torkit3d._C (third_party/torkit3d/torkit3d/csrc/torkit3d.cpp:10-23,
 * csrc/include/sample_farthest_points.h:6-8) plus the ATen/cuBLAS/apex kernels PyTorch dispatches to
 * from pc_sam/model/*.py.  Every entry point below names the reference interface it stands in for.
 *
 * Conventions: plain pointers and sizes only (no torch types); all pointers are DEVICE pointers unless
 * stated; tensors are contiguous row-major fp32 unless stated; no allocation inside (caller passes
 * outputs and workspace, `*_workspace_bytes` tells how much); no global mutable state, thread-safe,
 * work is enqueued on `stream` and nothing synchronises; return 0 on success, a negative PSAM_ERR_*
 * for bad arguments, a positive cudaError_t if a CUDA call failed (1000+CUresult for driver errors).
 *
 * "split-bf16" operands: two bf16 planes [2][rows][row_stride] with x ~= hi + lo (|err| <= 2^-17 |x|);
 * plane 0 = hi, plane 1 = lo, lo plane `plane_stride` elements after the hi plane.
 */
#ifndef PSAM_B200_H
#define PSAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define PSAM_ACT_NONE 0
#define PSAM_ACT_GELU 1
#define PSAM_ACT_RELU 2

/* ---- tokenizer ------------------------------------------------------------------------------ */

/* Farthest-point sampling + gather of the centres.
 * Replaces torkit3d._C.sample_farthest_points_cuda (sample_farthest_points_kernel.cu:106-165, called
 * from pc_sam/model/common.py:91) and batch_index_select (torkit3d/nn/functional.py:34-69, common.py:92).
 * xyz [B,N,3] -> idx_out [B,G] int64 (bit-exact with the reference kernel incl. tie-break),
 * centers_out [B,G,3].  Errors mirror the reference TORCH_CHECKs (:111-115): G<=0 or N<G -> PSAM_ERR_ARG. */
size_t psam_fps_workspace_bytes(int B, int N, int G);
int psam_fps_f32(const float* xyz, int B, int N, int G, long long* idx_out, float* centers_out, void* workspace,
                 cudaStream_t stream);

/* K nearest keys of every query (exact, direct-difference squared distance, ties by lower index),
 * sorted by (distance, index).  Replaces knn_points = torch.cdist + torch.topk
 * (pc_sam/model/common.py:27-56; call sites :97 and :251).  query [B,Q,3], key [B,N,3] ->
 * idx_out [B,Q,K] int64, d2_out [B,Q,K] squared distances (may be NULL). */
int psam_knn_f32(const float* query, const float* key, int B, int Q, int N, int K, long long* idx_out, float* d2_out,
                 cudaStream_t stream);

/* Group-feature gather: groups[b2,g,k,:] = [(xyz[b,idx]-centers[b,g])/radius, feats[b2,idx,0:C]], b=b2/rep.
 * Replaces the fancy-index gathers of KNNGrouper.forward (common.py:99-120) and
 * group_with_centers_and_knn (common.py:126-187).  radius<=0 means None.  feats [B*rep,N,C].
 * center_idx [B,G] (may be NULL) selects centralize_features=True (common.py:116-118, :181-185): C more channels
 * feats[b2,idx] - feats[b2,center_idx[b,g]] are appended (groups_out row = 3 + 2C floats). */
int psam_group_gather_f32(const float* xyz, const float* feats, const float* centers, const long long* knn_idx,
                          const long long* center_idx, int B, int rep, int N, int G, int K, int C, float radius,
                          float* groups_out, cudaStream_t stream);

/* Voronoi tokenizer features: out[b2,n,:] = [(xyz[b,n]-c)/max(|xyz[b,n]-c|,1e-8), |xyz[b,n]-c|, feats[b2,n,0:C]] with
 * c = centers[b, nn_idx[b,n]], b = b2/rep.  Replaces NNGrouper.forward / group_with_centers_and_nn
 * (common.py:190-236).  out fp32 [B*rep,N,4+C] and / or the split-bf16 copy y_hi (row pitch `pitch` >= 4+C, zero
 * padded) that feeds PatchEmbedNN.in_proj (pc_encoder.py:186) on the tensor cores. */
int psam_voronoi_features_f32(const float* xyz, const float* centers, const long long* nn_idx, const float* feats, int B,
                              int rep, int N, int G, int C, float* out, void* y_hi, long long y_plane, long long pitch,
                              cudaStream_t stream);

/* y[b, nn_idx[b,n], :] = max over the points of a Voronoi cell of x[b,n,:]; cells without a point are 0.
 * Replaces y.scatter_reduce_(1, nn_idx, x, "amax", include_self=False) on a zero tensor (pc_encoder.py:189-193).
 * x [B,N,D], y [B,G,D], D % 4 == 0. */
int psam_scatter_amax_f32(const float* x, const long long* nn_idx, int B, int N, int G, int D, float* y,
                          cudaStream_t stream);

/* 3 nearest centres per point and inverse-squared-distance weights.
 * Replaces compute_interp_weights (common.py:238-255).  idx_out [B,N,3] int64, w_out [B,N,3]. */
int psam_knn3_interp_f32(const float* xyz, const float* centers, int B, int N, int G, long long* idx_out, float* w_out,
                         cudaStream_t stream);

/* Nearest-neighbour squared distance (and index) of every query point to a key set; single cloud.
 * Replaces torkit3d chamfer_distance_forward (csrc/cuda/chamfer_distance_kernel.cu:10-151) as used by the
 * ground-truth prompt sampler (pc_sam/model/common.py:447-474): dist1/idx1 only.  idx_out may be NULL. */
int psam_nn_distance_f32(const float* query, const float* key, int n1, int n2, float* dist_out, long long* idx_out,
                         cudaStream_t stream);

/* Batched ground-truth prompt sampler: replaces the per-(cloud, mask) Python loops of sample_fixed_points /
 * sample_furthest_points_from_border (pc_sam/model/common.py:371-474) and their chamfer_distance calls with four launches
 * and no host synchronisation.  gt_masks [B*M, N] (0/1 bytes); prediction either as logits (mask = logit > 0,
 * common.py:392) or as 0/1 bytes (thresholded by the caller), or both NULL (first iteration: pred_logits is None).
 * from_error_region != 0: sample the point of (fn | fp) farthest from its complement (common.py:402-410);
 * == 0: the farther of the fn- and fp-region candidates, falling back to the ground-truth region (common.py:411-431).
 * Distances and tie-breaks equal the reference's (chamfer arithmetic, torch.argmax = lowest index).
 * Outputs: prompt_xyz_out [B*M, 3], prompt_label_out [B*M] (the ground-truth value at the sampled point), *status is
 * set to 1 if some mask had no valid candidate (the reference raises in torch.stack there); the caller zeroes it.
 * workspace: psam_border_prompt_workspace_bytes(B, M, N) bytes, 4-byte aligned (region counters, compacted foreground /
 * background index lists and per-point minima: the distance sweep costs |fg| x |bg| evaluations like the reference's
 * compacted chamfer call, spread over (fg block x background chunk) thread blocks). */
size_t psam_border_prompt_workspace_bytes(int B, int M, int N);
int psam_border_prompt_f32(const float* coords, const unsigned char* gt_masks, const float* pred_logits,
                           const unsigned char* pred_masks, int B, int M, int N, int from_error_region,
                           float* prompt_xyz_out, unsigned char* prompt_label_out, int* status, void* workspace,
                           cudaStream_t stream);

/* ---- dense contractions ---------------------------------------------------------------------- */

typedef struct {
    const void* hi;         /* bf16 hi plane, 16-byte aligned */
    long long plane_stride; /* elements from hi plane to lo plane (0: rows*row_stride) */
    int rows, k;            /* logical extents; k tail and row tail are zero-filled by TMA */
    long long row_stride;   /* elements, multiple of 8 */
    int nb1, nb2;           /* batch extents (0/1 = none) */
    long long b1_stride, b2_stride; /* elements, multiples of 8 */
} psam_operand;

typedef struct {
    float* out_f32;         /* optional fp32 output [.., M, ldo] */
    long long ldo, out_b1, out_b2;
    void* out_hi;           /* optional split-bf16 output (hi plane; lo at +out_plane elements) */
    long long out_plane, ldo_s, outs_b1, outs_b2;
    const float* bias;      /* [N] or NULL */
    const float* resid;     /* fp32, geometry of out_f32 (may alias it) or NULL */
    float alpha;            /* accumulator scale (1.0f for a plain linear) */
    int act;                /* PSAM_ACT_* applied after bias/residual */
    int accumulate;         /* 1: out_f32 += alpha*acc (+bias) with red.add; required when split_k>1 */
    int swiglu;             /* 1: W rows interleaved (gate_i, value_i); out_f32[:, i] = silu(gate_i)*value_i (fp32 out only) */
    int tile_hint;          /* 0: tile width for lowest latency; 1: for lowest SM-time (several clouds in flight); 32..256: explicit */
    float* gmax;            /* optional fused max-pool: gmax[(row / group_rows) * ld_gmax + col] = max over the group rows
                               (atomic; caller pre-fills with -inf; group_rows multiple of 32); replaces torch.max(x, dim=-2) */
    long long ld_gmax;
    int group_rows;
    const float* rd_w;      /* optional fused row-dot (replaces masks = hyper_in @ upscaled^T, mask_decoder.py:176):        */
    float* rd_out;          /*   rd_out[z, c, n] += sum_col act(alpha*acc + bias)[z*rd_rows + n, col] * rd_w[z, c, col]    */
    int rd_rows, rd_c;      /*   rd_out pre-zeroed [Z, rd_c, rd_rows]; rd_rows % 32 == 0; rd_c <= 8; no other output allowed */
    float* stats_out;       /* stats_out[row] (2 floats, pre-zeroed) accumulates (sum, sum of squares) of the row this GEMM
                             * WRITES as split-bf16 - the statistics a LayerNorm-folded consumer GEMM needs: with swiglu +
                             * out_hi the SwiGLU products (timm SwiGLU.norm), otherwise (out_hi, split_k == 1, no
                             * accumulate) the final values after bias / residual / activation (norm1 / norm2 / fc_norm) */
    const float* ln_stats;  /* LayerNorm folded into this GEMM: A = the un-normalised rows, W pre-multiplied by gamma,
                             * ln_c[n] = sum_k gamma_k W[n,k], bias[n] = sum_k beta_k W[n,k] + b[n];
                             * out = act(rstd_row * (acc - mean_row * ln_c[n]) + bias[n] (+ resid)) with mean / rstd from
                             * ln_stats[row] = (sum, sum sq) over ln_h columns.  Works with every output form of the
                             * vectorised epilogue (fp32, split-bf16, SwiGLU pairs) and with accumulate / split_k (each
                             * split scales its partial sum). */
    const float* ln_c;
    int ln_h;
    float ln_eps;
    int variant;            /* 0 = policy default.  Experiment switches (the library reads no environment variable):
                             * 0x1 cta_group::2 pairs, 0x2 BK=32 4-stage ring, 0x4 scalar epilogue, 0x8 the dual-resident
                             * wide-tile kernel (two 97 KB CTAs per SM; 0x10 overrides it),
                             * 0x80 two MMA-issuing warps for wide one-shot tiles (measured no gain: opt-in),
                             * 0x20 force / 0x40 forbid the persistent kernel (tile loop inside the CTA, double-buffered TMEM
                             * accumulator; default when the launch has >= 2 tiles per SM), bits 16-19 tiles per CTA to aim for,
                             * bits 8-11 W-tile multicast cluster size (2|4), bits 12-15 L2 prefetch depth in k-blocks */
} psam_gemm_out;

/* C[M,N] = A[M,K] * W[N,K]^T on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 * passes=3: split-bf16 emulation of the reference's fp32 nn.Linear / bmm; passes=1: hi planes only.
 * Replaces nn.Linear / F.linear / @ on the PatchEncoder, ViT blocks and upscaling MLP
 * (common.py:486-497, pc_encoder.py:99-116,136-143, timm EvaBlock, mask_decoder.py:53-59). */
int psam_gemm_bf16x3(const psam_operand* a, const psam_operand* w, const psam_gemm_out* out, int passes, int split_k,
                     cudaStream_t stream);

/* Row-complete GEMM with LayerNorm and activation in the epilogue:
 *   Y = act(LayerNorm(A W^T + gbias[row / group_rows])) as split-bf16, A [M,K<=128], W [N,K] with N = 256 or 512 (a CTA owns
 * 128 rows x the full width, so the row statistics stay on the SM and the fp32 pre-activation never reaches memory).
 * Replaces conv2[0..2] of PatchEncoder (Linear on cat[max, x] = W_a max + W_b x, LayerNorm, GELU; common.py:491-495):
 * gbias carries W_a max + b per group.  gamma / beta [N]; out_hi [M, ldo_s] hi plane, lo plane out_plane elements further. */
int psam_gemm_rowln_bf16x3(const psam_operand* a, const psam_operand* w, const float* gbias, long long ld_gbias, int group_rows,
                           const float* gamma, const float* beta, float eps, int act, void* out_hi, long long out_plane,
                           long long ldo_s, int passes, cudaStream_t stream);

/* Fused encoder self-attention on tensor cores: out = softmax(Q K^T * scale) V per (cloud, head).
 * q/k/v are split-bf16 operand views [L rows x dh] with nb1 = heads, nb2 = clouds (typically three column windows of
 * the fused qkv activation).  dh == 64 or 88 (EVA-giant; the 88-wide head is handled as 64 + 24 columns, zero padded by
 * TMA), any L >= 1 (PSAM_ERR_UNSUPPORTED otherwise - the caller then uses
 * psam_gemm_bf16x3 + psam_softmax_split).  Key blocks are streamed once: S_j lands in a ring of tensor-memory slots,
 * P_j = exp2(S_j c - m_ref) is written back into the slot as split-bf16 and consumed as the TMEM A operand of the PV
 * MMA; the reference maximum is moved (and O rescaled) only when a block exceeds it by more than 2^8.
 * Replaces F.scaled_dot_product_attention in timm EvaAttention (blocks called at pc_encoder.py:138-139). */
int psam_attention_bf16x3(const psam_operand* q, const psam_operand* k, const psam_operand* v, void* out_hi,
                          long long out_plane, long long ldo, long long out_head_stride, long long out_cloud_stride,
                          float scale, cudaStream_t stream);

/* Same contract, computed by the first-generation kernels (exact two-pass softmax with S resident in tensor memory for
 * L <= 512, two-sweep ring for longer rows, P staged through shared memory).  Kept as an independent implementation
 * the tests cross-check the streaming kernel against. */
int psam_attention_bf16x3_twopass(const psam_operand* q, const psam_operand* k, const psam_operand* v, void* out_hi,
                                  long long out_plane, long long ldo, long long out_head_stride,
                                  long long out_cloud_stride, float scale, cudaStream_t stream);

/* y = split-bf16(x (+ add)) with zero fill up to `pitch` (add may be NULL; same row stride as x). */
int psam_split_add_f32(const float* x, const float* add, long long ld, long long rows, int D, void* y_hi, long long y_plane,
                       long long ldy_s, long long pitch, cudaStream_t stream);

/* Small fp32 SIMT linear for the prompt decoder (rows < one MMA tile):
 * Y[z][M,N] = act((X[z] (+X2[z]))[M,K] * W[z][N,K]^T + b[z]) (+R[z]); strides in elements; any pointer
 * stride may be 0 to broadcast.  Replaces nn.Linear in transformer.py:199-202,239-253 and the MLP
 * heads mask_decoder.py:189-211. */
typedef struct {
    const float* x;  long long ldx, x_z;
    const float* x2; long long x2_z;      /* optional addend with the geometry of x */
    const float* w;  long long ldw, w_z;
    const float* b;  long long b_z;       /* optional */
    const float* r;  long long r_z;       /* optional residual with the geometry of y */
    float* y;        long long ldy, y_z;
    int M, N, K, Z, act;
} psam_linear_args;
int psam_linear_f32(const psam_linear_args* args, cudaStream_t stream);

/* ---- normalisation / activation / glue -------------------------------------------------------- */

/* y = LayerNorm(x (+ r) (+ gbias[row / group_rows])) * gamma + beta, optional GELU afterwards; writes
 * fp32 and/or split-bf16 (columns D..pitch of the split output are zero-filled).
 * Replaces apex FusedLayerNorm / nn.LayerNorm (+nn.GELU) (torch_utils.py:28-38, common.py:487-495,
 * transformer.py norms, timm norm1/norm2/fc_norm). */
typedef struct {
    const float* x; long long ldx;
    const float* r; long long ldr;            /* optional residual */
    const float* gbias; long long ld_gbias; int group_rows; /* optional per-group row addend */
    const float* gamma; const float* beta; float eps;
    int rows, D, act;
    float* y; long long ldy;                  /* optional */
    void* y_hi; long long y_plane, ldy_s, pitch; /* optional split output */
    int padded;                               /* 1: x rows (zeros), gamma, beta and outputs are valid up to roundup4(D) */
    int policy;                               /* 0: lowest latency (CTA per row for short token streams); 1: least SM-time
                                               * (warp per row, no block barriers) - used when several clouds are in flight */
    const float* post_add; long long ld_post; /* optional: a SECOND split-bf16 output y2 = split(y + post_add[row]) - the     */
    void* y2_hi; long long y2_plane, ldy2_s;  /* "keys + positional encoding" operand of the decoder's projections         */
} psam_ln_args;
int psam_layernorm_f32(const psam_ln_args* args, cudaStream_t stream);

/* SwiGLU with inner LayerNorm (timm SwiGLU, scale_mlp=True): h = silu(g)*x, y = LN(h); gx holds g in
 * columns [0,H) and x in columns [x_off, x_off+H).  Output split-bf16, zero padded to pitch. */
int psam_swiglu_ln(const float* gx, long long ld, long long x_off, int rows, int H, const float* gamma,
                   const float* beta, float eps, void* y_hi, long long y_plane, long long ldy_s, long long pitch,
                   cudaStream_t stream);

/* First layer of the mini-PointNet / positional MLP: y = act(LN?(x[rows,Cin] * W[Cout,Cin]^T + b)),
 * Cin <= 8, Cout multiple of 32 and <= 512; split-bf16 output.  Replaces conv1[0..2] of PatchEncoder
 * (common.py:486-489) and pos_embed[0..1] (pc_encoder.py:102-104). */
int psam_small_in_linear(const float* x, int rows, int Cin, const float* W, const float* b, const float* gamma,
                         const float* beta, float eps, int use_ln, int act, int Cout, void* y_hi, long long y_plane,
                         long long ldy_s, cudaStream_t stream);

/* Max over the K rows of each group: x [groups*K, D] -> y [groups, D] fp32 (optional) and split-bf16
 * (optional).  Replaces torch.max(x, dim=-2) (common.py:501,505). */
int psam_group_max(const float* x, long long ldx, int groups, int K, int D, float* y, long long ldy, void* y_hi,
                   long long y_plane, long long ldy_s, cudaStream_t stream);

/* Row softmax of fp32 scores with scale, split-bf16 output (attention probabilities). */
int psam_softmax_split(const float* s, long long lds, long long rows, int L, float scale, void* p_hi,
                       long long p_plane, long long ldp, cudaStream_t stream);

/* Transposed copy of a split-bf16 matrix block per batch: dst[z][c][r] = src[z][r][c] (both planes). */
int psam_transpose_split(const void* src_hi, long long src_plane, long long src_ld, long long src_z1,
                         long long src_z2, void* dst_hi, long long dst_plane, long long dst_ld, long long dst_z1,
                         long long dst_z2, int rows, int cols, int nz1, int nz2, cudaStream_t stream);

/* Random-Fourier positional encoding (+ optional prompt-label embedding):
 * out[r,:] = [sin(2*pi*c@G), cos(2*pi*c@G)] (+ emb[label[r]]).  Also raises the out-of-range flag
 * (*bad_flag = 1) if any coordinate is outside [-1-1e-6, 1+1e-6] (prompt_encoder.py:44-46).
 * Replaces PositionEmbeddingRandom / PointEncoder (prompt_encoder.py:13-77). labels int32 or NULL. */
int psam_posenc_f32(const float* coords, long long rows, const float* gauss, int F, const int* labels,
                    const float* emb0, const float* emb1, float* out, int* bad_flag, cudaStream_t stream);

/* Multi-head softmax attention for short sequences (fp32, one warp per query):
 * O[z,i,h,:] = softmax(Q[z,i,h,:] . K[z,:,h,:]^T / sqrt(dh)) V[z,:,h,:].  Replaces
 * Attention.forward core (transformer.py:214-233). */
int psam_attention_f32(const float* q, const float* k, const float* v, float* o, int Z, int Lq, int Lk, int H, int dh,
                       long long ldq, long long ldk, long long ldv, long long ldo, cudaStream_t stream);

/* Mask-decoder glue (mask_decoder.py:126-139): tokens[z] = cat(iou_token, mask_tokens, sparse[z]);
 * src[z,g,:] = pc_emb[z/rep,g,:] + dense[(z % dense_mod)...]; see engine for exact broadcast rules. */
int psam_decoder_prepare(const float* iou_token, const float* mask_tokens, int n_mask_tokens, const float* sparse,
                         int P, const float* pc_emb, const float* dense, long long dense_z, long long dense_g, int Z,
                         int rep, int G, int D, float* tokens, float* src, cudaStream_t stream);

/* 3-NN feature upsampling fused with LayerNorm + GELU: y[z*N+n,:] = GELU(LN(sum_k w[b,n,k]*f[z,idx[b,n,k],:])),
 * b = z/rep; split-bf16 output.  Replaces interpolate_features (common.py:258-274) + output_upscaling[1..2]
 * (mask_decoder.py:55-56) after output_upscaling[0] has been applied to the patch features. */
int psam_interp_ln_gelu(const float* f, int Z, int rep, int G, int D, const long long* idx, const float* w, int N,
                        const float* gamma, const float* beta, float eps, void* y_hi, long long y_plane,
                        long long ldy_s, cudaStream_t stream);

/* masks[z,c,n] = sum_d hyper[z,c,d] * u[z*N+n,d]  (mask_decoder.py:176). */
int psam_mask_dot(const float* u, long long ldu, const float* hyper, int Z, int C, int N, int D, float* masks,
                  cudaStream_t stream);

/* out[i] = a[i] + b[(((i / chunk) / rep) * chunk + i % chunk) % b_period]  (repeat_interleave-style broadcast,
 * pc_sam/model/common.py:277-284) */
int psam_add_bcast_f32(const float* a, const float* b, long long n, long long chunk, long long rep, long long b_period,
                       float* out, cudaStream_t stream);

/* fp32 [rows,D] (row stride ld) -> split-bf16 planes (weight packing, activations entering a GEMM) */
int psam_split_f32(const float* x, long long ld, long long rows, int D, void* y_hi, long long y_plane,
                   long long ldy_s, long long pitch, cudaStream_t stream);

/* ---- automatic mask generation ----------------------------------------------------------------- */
/* Candidate masks are bit-packed: bits [R, W] uint32 with W = ceil(N / 32), bit j of word w = point 32 w + j, tail bits 0.
 * The reference ships no automatic mask generator; the semantics are this project's, following SAM's
 * SamAutomaticMaskGenerator (segment_anything/automatic_mask_generator.py): see DESIGN.md, "Automatic mask generation". */

/* For R rows of logits [R, N] (one row per candidate) and their predicted IoU iou_pred [R], in one pass:
 * bits[r] = (logit > mask_threshold), area[r] = popcount, stability[r] = #(logit > t + off) / #(logit > t - off) as an fp32
 * division of the integer counts (0 when the denominator is 0; SAM's calculate_stability_score), keep[r] = 1 iff
 * iou_pred > pred_iou_thresh && stability >= stability_thresh && area > 0.  Output pointers may point into a larger
 * candidate table (the caller offsets them by the chunk's first row). */
int psam_mask_stats_f32(const float* logits, const float* iou_pred, int R, int N, float mask_threshold, float stability_offset,
                        float pred_iou_thresh, float stability_thresh, uint32_t* bits, int* area, float* stability,
                        unsigned char* keep, cudaStream_t stream);

/* Pairwise IoU of two bit-mask sets a [Ka, W], b [Kb, W]: iou [Ka, Kb] = inter / (area_a + area_b - inter) as an fp32
 * division of exact integer counts (0 when the union is 0); inter [Ka, Kb] int32 may be NULL. */
int psam_mask_iou_u32(const uint32_t* a_bits, int Ka, const uint32_t* b_bits, int Kb, int W, float* iou, int* inter,
                      cudaStream_t stream);

/* Greedy mask NMS over K candidates (bits [K, W], area / score / keep [K] from psam_mask_stats_f32):
 * the candidates with keep != 0, in order of score descending (ties: lower index first), are kept unless an earlier KEPT
 * candidate has IoU > nms_thresh with them.  keep_idx [K] int32 = kept candidate indices in that order, -1 after the last;
 * *kept_count (device) = their number.  No host synchronisation: every launch is sized for K.  K <= 16384
 * (PSAM_ERR_UNSUPPORTED beyond).  workspace: psam_mask_nms_workspace_bytes(K, W) bytes, 16-byte aligned. */
size_t psam_mask_nms_workspace_bytes(int K, int W);
int psam_mask_nms(const uint32_t* bits, const int* area, const float* score, const unsigned char* keep, int K, int W,
                  float nms_thresh, int* keep_idx, int* kept_count, void* workspace, cudaStream_t stream);

/* out [k, N] bytes (0 / 1) = the bits of rows rows[0..k) (rows NULL: rows 0..k-1). */
int psam_mask_unpack_u8(const uint32_t* bits, int W, const int* rows, int k, int N, unsigned char* out, cudaStream_t stream);

const char* psam_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PSAM_B200_H */
