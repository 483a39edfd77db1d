/* es3.h -- C ABI of libes3.so: hand-written sm_100a kernels for the EfficientSAM3 hot path.
 *
 * The reference (SimonZeng7108/efficientsam3) has no FFI of its own: its hot path bottoms out in
 * torch.nn.functional calls (SURVEY.md section 8b).  Each entry point below therefore names the reference
 * Python call site whose device work it replaces; the Python module shells in efficientsam3_b200/
 * (same class names / state_dict keys as the reference) are the only callers.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; es3_last_error() gives the message
 *     (thread-local).  There is no CPU fallback: non-Blackwell devices fail in es3_init().
 *   - all pointers are DEVICE pointers unless stated; `stream` is a cudaStream_t passed as void*.
 *   - activations are NHWC (pixels x channels) / tokens x features, bf16, 16-byte aligned; `ld*` are
 *     row strides in ELEMENTS.  fp32 vectors (scale / bias / folded BN) are per output channel.
 *   - act codes: 0 none, 1 relu, 2 hardswish, 3 gelu(erf), 4 gelu(tanh), 5 relu6, 6 sigmoid.
 */
#ifndef ES3_H_
#define ES3_H_

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ runtime */
const char* es3_last_error(void);
int es3_version(void);
/* Queries `device`; fails unless it is compute capability 10.x. */
int es3_init(int device, int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------ GEMMs */
/* out[m,n] = act(scale[n] * sum_k A[m,k] W[n,k] + bias[n]) (+ residual[m,n]);  tcgen05 + TMEM + TMA.
 * Replaces nn.Conv2d(k=1)+BatchNorm2d+act of ConvLayer (sam3/sam3/backbones/efficientvit/nn/ops.py:39-80),
 * the student head 1x1 (stage1/model.py:194-197) and every nn.Linear on the path (vitdet.py:466-515,
 * sam/transformer.py:185-264).  N % 32 == 0, K % 8 == 0; bn_hint in {0 (auto), 32, 64, 128, 256}. */
int es3_gemm_bf16(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_f32,
                  int M, int N, int K, const float* scale, const float* bias, int act, const void* residual,
                  long long ldr, int bn_hint, void* stream);

/* Extended epilogue: fp32 residual (res_f32 = 1: the ViT residual stream stays fp32), and 2-D axial RoPE applied to
 * columns [0, rope_cols) (the q|k part of a fused QKV projection, heads of 64) before rounding -- rope is a
 * [positions][32] table of (cos, sin) float pairs, position = raster index of the token inside its
 * rope_win x rope_win window (rope_win > 0) or inside the rope_H x rope_W map (rope_win = 0).
 * act_after_res = 1 applies the activation after the residual add (TinyViT MBConv: act3(conv3(x) + shortcut),
 * tiny_vit.py:112-125).  Replaces Attention.qkv + apply_rotary_enc (vitdet.py:68-90, 480-486). */
int es3_gemm_bf16_ex(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int out_f32,
                     int M, int N, int K, const float* scale, const float* bias, int act, const void* residual,
                     long long ldr, int res_f32, const float* rope, int rope_cols, int rope_H, int rope_W, int rope_win,
                     int act_after_res, int bn_hint, void* stream);

/* ConvTranspose2d(k=2, s=2) on NHWC as a tcgen05 GEMM (N = 4*Cout) with a depth-to-space epilogue.
 * Wt [4*Cout][Cin] bf16, Wt[(dy*2+dx)*Cout+co][ci] = w[ci][co][dy][dx]; bias4 [4*Cout]; out [B,2H,2W,Cout].
 * Replaces MaskDecoder.output_upscaling ConvTranspose2d (mask_decoder.py:59-70) and the FPN upsamplers (necks.py). */
int es3_convt2x2_bf16(const void* x, const void* Wt, void* out, int out_f32, int B, int H, int Wd, int Cin, int Cout,
                      const float* bias4, int act, const void* residual, int res_f32, int act_after_res, void* stream);

/* Dense 3x3 / stride 1 / pad 1 conv as an implicit tcgen05 GEMM (halo via TMA zero fill).
 * x [B,H,W,C] bf16 NHWC; W [N][9*C] with k = (ky*3+kx)*C + c; out [B,H,W,N].
 * Replaces head.3 = nn.Conv2d(1024,1024,3,padding=1) (stage1/model.py:198) and the FPN 3x3s (necks.py). */
int es3_conv3x3_bf16(const void* x, const void* W, void* out, int out_f32, int B, int H, int Wd, int C, int N,
                     const float* scale, const float* bias, int act, const void* residual, int bn_hint, void* stream);

/* CUDA-core GEMM, same epilogue; for tiny M (decoder tokens, SE MLPs) and as the on-device cross-check
 * of the tensor-core kernel.  a_f32 / w_f32 / res_f32 select fp32 (1) or bf16 (0) operands. */
int es3_gemm_simt(const void* A, long long lda, int a_f32, const void* W, long long ldw, int w_f32, void* out,
                  long long ldo, int out_f32, int M, int N, int K, const float* scale, const float* bias, int act,
                  const void* residual, long long ldr, int res_f32, void* stream);

/* ------------------------------------------------------------------------------------------ convs */
/* 3x3 stride-2 pad-1 conv from the NCHW fp32 image to NHWC bf16, folded BN + act.
 * w [27][Cout] fp32 tap-major ((ci*9+ky*3+kx)), Cout in {8,16,24,32,48}.
 * Replaces EfficientViT input_stem op 0 (efficientvit/backbone.py:49-57). */
int es3_stem_conv3x3_s2(const float* x, const float* w, const float* bias, void* out, int B, int H, int W, int Cout,
                        int act, void* stream);

/* Depthwise ks x ks (3|5), stride 1|2, pad ks/2.  w [ks*ks][C] fp32 tap-major (BN scale folded), bias [C]|NULL.
 * Replaces ConvLayer(groups=C) in DSConv / MBConv (efficientvit/nn/ops.py:273-367). */
int es3_dwconv_bf16(const void* x, long long ldx, const float* w, const float* bias, void* out, long long ldo, int B,
                    int H, int W, int C, int ks, int stride, int act, void* stream);

/* Same contract as es3_dwconv_bf16 (C % 32 == 0): shared-memory tiled, 4-pixel register strips. */
int es3_dwconv_tiled_bf16(const void* x, long long ldx, const float* w, const float* bias, void* out, long long ldo,
                          int B, int H, int W, int C, int ks, int stride, int act, void* stream);

/* y = x + BN(pw(act(BN(dw3x3(x))))) in one pass; C in {8,16,24,32}.
 * Replaces the stem ResidualBlock(DSConv) (efficientvit/backbone.py:58-67). */
int es3_dsconv_res_bf16(const void* x, const float* wdw, const float* bdw, const float* wpw, const float* bpw,
                        void* out, int B, int H, int W, int C, int act, void* stream);

/* EfficientViT-B1 input stem in one kernel on mma.sync: x1 = hswish(BN(conv3x3_s2(img))), y = x1 + BN(pw(hswish(BN(dw3x3(x1))))).
 * img [B,3,H,W] fp32 NCHW -> out [B,Ho,Wo,16] bf16 NHWC.  w0 [16][32] bf16 (k = ci*9+ky*3+kx, zero padded), s0/b0
 * folded BN [16]; wdw [9][16] fp32 (BN scale folded), bdw [16]; wpw [16][16] bf16 [n][k], spw/bpw folded BN [16].
 * Replaces input_stem op 0 + op 1 (efficientvit/backbone.py:49-67) for width_list[0] == 16, hswish. */
int es3_stem_fused_c16(const float* img, const void* w0, const float* s0, const float* b0, const float* wdw,
                       const float* bdw, const void* wpw, const float* spw, const float* bpw, void* out, int B, int H,
                       int W, void* stream);

/* Whole MBConv block in one kernel: y = [x +] BN3(pw2(act(BN2(dw3x3_s(act(BN1(pw1(x)))))))) with the 4x-expanded
 * tensor kept in shared memory (mma.sync expand/project around an fp32 depthwise).  w1 [Mid][Cin], w3 [Cout][Mid]
 * bf16; s1,b1,b2 [Mid], s3,b3 [Cout] fp32 (BN folded; ones/zeros where the reference has bias-only convs);
 * wdw [9][Mid] fp32.  Returns -1 (no error set) when the shape is not instantiated -- the caller then runs
 * es3_gemm_bf16 + es3_dwconv_tiled_bf16.  Replaces MBConv inside ResidualBlock (efficientvit/nn/ops.py:315-367,
 * 740-770) for efficientvit_b1 stages 1-3 heads. */
int es3_mbconv_fused_bf16(const void* x, void* y, const void* w1, const float* s1, const float* b1, const float* wdw,
                          const float* b2, const void* w3, const float* s3, const float* b3, int B, int H, int W,
                          int Cin, int Mid, int Cout, int stride, int residual, int act, void* stream);
/* Same contract on tcgen05 for the stride-1 residual blocks (Cin == Cout in {32, 64}, Mid = 4 Cin, hardswish): the two
 * pointwise GEMMs are UMMAs (TMA-staged 128B-swizzled operands, TMEM accumulators, project accumulating over 64-channel
 * chunks), the depthwise stays on mma.sync with diagonal B fragments.  Returns -1 for any other shape. */
int es3_mbconv_tc_bf16(const void* x, void* y, const void* w1, const float* s1, const float* b1, const float* wdw,
                       const float* b2, const void* w3, const float* s3, const float* b3, int B, int H, int W, int Cin, int Mid,
                       int Cout, int stride, int residual, int act, void* stream);
/* Same contract on tcgen05 for the stride-2, no-residual blocks (Cin, Mid, Cout) in {(16,64,32), (32,128,64), (64,256,128)}:
 * 4 x 16 output tiles, 9 x 33 input tiles = three M=128 UMMA row blocks, 32-channel chunks.  Returns -1 for any other shape. */
int es3_mbconv_tc_s2_bf16(const void* x, void* y, const void* w1, const float* s1, const float* b1, const float* wdw,
                          const float* b2, const void* w3, const float* s3, const float* b3, int B, int H, int W, int Cin,
                          int Mid, int Cout, int stride, int residual, int act, void* stream);
/* Depthwise 3x3 (stride 1) + bias + hardswish + pointwise projection + BN (+ residual) in one tcgen05 kernel, for MBConv blocks
 * whose expanded tensor is too wide for the fully fused kernels (EfficientViT stages 3/4): mid [B,H,W,Mid] bf16 is TMA-staged in
 * 64-channel chunks with its halo, the depthwise runs as diagonal m16n8k8 MMAs, its output goes straight into the swizzled A
 * operand of UMMAs accumulating [128 px x Cout] in TMEM.  wdw [9][Mid] fp32 (BN scale folded), b2 [Mid], w3 [Cout][Mid] bf16,
 * s3/b3 [Cout]; residual [B,H,W,Cout] bf16 or NULL.  Instantiated (Mid, Cout) = (512,128), (1024,256); -1 otherwise.
 * Replaces es3_dwconv_tiled_bf16 + es3_gemm_bf16 for ops.py:315-367 (depth_conv + point_conv). */
int es3_dwproj_tc_bf16(const void* mid, const float* wdw, const float* b2, const void* w3, const float* s3, const float* b3,
                       const void* residual, void* y, int B, int H, int W, int Mid, int Cout, int act, void* stream);

/* Bilinear (align_corners=False) NHWC bf16 -> NCHW fp32.  Replaces F.interpolate at stage1/model.py:204-210. */
int es3_bilinear_nhwc_to_nchw(const void* in, float* out, int B, int Hi, int Wi, int C, int Ho, int Wo, void* stream);
/* MaxPool2d(2,2) on NHWC bf16 (FPN 0.5x level, necks.py:64-69). */
int es3_maxpool2x2_bf16(const void* x, void* out, int B, int H, int W, int C, void* stream);
/* Layout conversions at the module boundary. */
int es3_nhwc_to_nchw_f32(const void* in, float* out, int B, int HW, int C, void* stream);
int es3_nchw_f32_to_nhwc(const float* in, void* out, int B, int HW, int C, void* stream);

/* ------------------------------------------------------------------------------------------ LiteMLA */
/* ms [B,H,W,ld] bf16: reads qkv in channels [0,C3), writes aggreg(qkv) = grouped1x1(dw5x5(qkv)) into
 * channels [C3,2*C3).  wdw [25][C3] fp32, wpw [C3][16] fp32.  Replaces LiteMLA.aggreg (ops.py:560-575,655-660). */
int es3_litemla_aggreg(void* ms, long long ld, const float* wdw, const float* wpw, int B, int H, int W, int C3,
                       void* stream);
/* Same contract as es3_litemla_aggreg (C3 % 64 == 0): tiled dw5x5 with the grouped 1x1 fused in registers. */
int es3_litemla_aggreg_tiled(void* ms, long long ld, const float* wdw, const float* wpw, int B, int H, int W, int C3,
                             void* stream);
/* Tensor-core aggreg: the depthwise 5x5 and the grouped 1x1 are folded into one grouped 5x5 conv,
 * wcomb [C3/16][25][16][16] bf16 with wcomb[g][tap][n][i] = wpw[g*16+n][i] * wdw[tap][g*16+i] (K = 400 per group). */
int es3_litemla_aggreg_tc(void* ms, long long ld, const void* wcomb, int B, int H, int W, int C3, void* stream);
/* Same contract with the two weight tensors kept apart: depthwise 5x5 as diagonal m16n8k8 MMAs, its bf16-rounded result fed
 * from registers into the grouped 16x16 pointwise MMA.  wdw [C3/16][25][16] bf16 (group, tap, channel), wpw [C3][16] bf16. */
int es3_litemla_aggreg_dwpw(void* ms, long long ld, const void* wdw, const void* wpw, int B, int H, int W, int C3,
                            void* stream);
/* ReLU linear attention over the multi-scale qkv buffer (head h = channels [48h,48h+48) = q|k|v, dim 16).
 * kv_ws: es3_litemla_ws_floats(B,HW,heads2) floats of scratch (two-stage deterministic reduction, no atomics).  att [B,HW,ldo] bf16.  Replaces relu_linear_att (ops.py:584-621). */
long long es3_litemla_ws_floats(int B, int HW, int heads2);
int es3_litemla_attn(const void* ms, long long ld, float* kv_ws, void* att, long long ldo, int B, int HW, int heads2,
                     float eps, void* stream);
/* Same contract for any head dim in {16, 32} (efficientvit_b2 / b3: dim 32): head h occupies channels [h*3*dim, +3*dim)
 * of ms as q|k|v and [h*dim, +dim) of att.  CUDA-core fp32 formulation; kv_ws = es3_litemla_generic_ws_floats floats. */
long long es3_litemla_generic_ws_floats(int B, int HW, int heads2, int dim);
int es3_litemla_attn_generic(const void* ms, long long ld, float* kv_ws, void* att, long long ldo, int B, int HW, int heads2,
                             int dim, float eps, void* stream);

/* ------------------------------------------------------------------------------------------ ViT trunk */
/* LayerNorm over C (C % 128 == 0) of fp32 rows, optional tiled abs-pos add first (pos [pos_size^2, C], token
 * (h, w) uses entry (h % pos_size, w % pos_size)); writes bf16 and/or fp32.  Replaces nn.LayerNorm in Block
 * (vitdet.py:597-613) and get_abs_pos(tiling) + ln_pre (vitdet.py:205-214, 820-828). */
int es3_layernorm_f32(const float* x, const float* pos, int pos_size, int H, int W, const float* gamma,
                      const float* beta, float eps, void* y_bf16, float* y_f32, long long M, int C, void* stream);
/* Patch-embedding im2col: x [B,3,S,S] fp32 -> [B*(S/P)^2, Kp] bf16, column = c*P*P + ky*P + kx, zero padded to Kp.
 * With es3_gemm_bf16 this replaces PatchEmbed.proj (vitdet.py:299-336). */
int es3_im2col_patch(const float* x, void* cols, int B, int S, int P, int Kp, void* stream);
/* Softmax attention, head_dim 64, inside win x win windows (win > 0) or global (win = 0), on the fused qkv
 * activation [B*H*W, 3C] bf16 -> [B*H*W, C] bf16; windows are gathered in place (no partition copies).
 * Replaces window_partition + F.scaled_dot_product_attention + window_unpartition (vitdet.py:93-139, 502). */
int es3_attention_bf16(const void* qkv, void* out, int B, int H, int W, int C, int num_heads, int win, float scale,
                       void* stream);
/* The two implementations behind es3_attention_bf16: tcgen05 / TMEM flash attention (QK^T and PV as UMMAs, P kept in
 * TMEM; used for L >= 128) and the warp-level mma.sync kernel (short windows; also the on-device cross-check). */
int es3_attention_tc_bf16(const void* qkv, void* out, int B, int H, int W, int C, int num_heads, int win, float scale,
                          void* stream);
int es3_attention_mma_bf16(const void* qkv, void* out, int B, int H, int W, int C, int num_heads, int win, float scale,
                           void* stream);
/* [B, HW, C] fp32 tokens -> [B, C, HW] fp32 (the NCHW map ViT.forward returns, vitdet.py:846-857). */
int es3_tokens_f32_to_nchw(const float* in, float* out, int B, int HW, int C, void* stream);
/* fp32 -> fp16 (RN) over n contiguous elements: the stored format of the teacher-embedding dump
 * (save_embedding_image_stage1.py:92); done on the device so the D2H copy moves 2 bytes per element. */
int es3_cast_f32_to_f16(const float* in, void* out, long long n, void* stream);

/* Same contract as es3_litemla_attn; KV state and the apply step run on mma.sync (KV split hi+lo bf16). */
int es3_litemla_attn_tc(const void* ms, long long ld, float* kv_ws, void* att, long long ldo, int B, int HW, int heads2,
                        float eps, void* stream);

/* ------------------------------------------------------------------------------------------ SAM heads */
/* PositionEmbeddingRandom over an h x w grid -> [h*w, 2F] fp32 (PromptEncoder.get_dense_pe, prompt_encoder.py:61-69). */
int es3_dense_pe(const float* gauss, int F, int h, int w, float* out, void* stream);
/* Point prompts with labels -1 (not a point) / 0,1 (point) / 2,3 (box corners) -> sparse embeddings [B, P+pad, 2F] fp32;
 * pad != 0 appends the padding point used when no box is given (prompt_encoder.py:71-131). */
int es3_point_embed(const float* coords, const int* labels, const float* gauss, const float* not_a_point,
                    const float* point_emb, int F, int B, int P, int pad, float img_w, float img_h, float* out, void* stream);
/* Mask prompt: PromptEncoder.mask_downscaling (prompt_encoder.py:45-63) on mask [B,1,4h,4w] fp32, fused with the decoder's
 * `image_embeddings + dense` (mask_decoder.py:189) and written token-major: keys[row] = base[row % base_rows] + dense[row],
 * rows = B*h*w (base NULL -> the dense embedding alone).  Weights are the module's tensors in their native layouts. */
int es3_mask_downscale_tokens(const float* mask, const float* w0, const float* b0, const float* g1, const float* be1,
                              const float* w1, const float* b1, const float* g2, const float* be2, const float* w2,
                              const float* b2, const float* base, long long base_rows, float* out_f32, void* out_bf16, int B,
                              int h, int w, int C, float eps, void* stream);
/* Hole / sprinkle filling of low-res mask logits (SAM2Transforms.postprocess_masks, sam1_utils.py:77-105): 8-connected
 * components of (score <= thr) with area <= max_hole_area become thr + 10, components of (score > thr) of the input with
 * area <= max_sprinkle_area become thr - 10.  in/out [N,H,W] fp32, not aliased; labels_ws, area_ws: N*H*W ints each. */
int es3_fill_small_components(const float* in, float* out, int* labels_ws, int* area_ws, int N, int H, int W, float thr,
                              float max_hole_area, float max_sprinkle_area, void* stream);
/* y[m] = x[m] + add[m % R] over C channels; bf16 and/or fp32 output (queries + pe, keys + key_pe). */
int es3_add_rows(const float* x, const float* add, long long M, int C, int R, void* y_bf16, float* y_f32, void* stream);
/* [B,C,HW] fp32 (+ per-channel vector, e.g. no_mask_embed) -> token-major [B,HW,C] fp32 and/or bf16. */
int es3_nchw_f32_to_tokens(const float* in, const float* addc, float* out_f32, void* out_bf16, int B, int HW, int C,
                           void* stream);
/* Softmax attention, few queries (prompt tokens) x many keys; q fp32, k/v bf16 (kv_f32 = 0) or fp32; out fp32.
 * Replaces Attention core for self_attn / cross_attn_token_to_image (transformer.py:185-264). head_dim 16|32. */
int es3_attn_few_queries(const float* q, long long ldq, const void* k, const void* v, long long ldkv, int kv_f32, float* out,
                         long long ldo, int B, int H, int head_dim, int Tq, int Tk, float scale, void* stream);
/* Softmax attention, many queries (image tokens, bf16) x <= 16 keys (fp32); out bf16 (cross_attn_image_to_token). */
int es3_attn_few_keys(const void* q, long long ldq, const float* k, const float* v, long long ldkv, void* out, long long ldo,
                      int B, int H, int head_dim, int Nq, int Tk, float scale, void* stream);
/* y = gelu(LayerNorm_C(x) * w + b) on rows of C <= 128 channels -> bf16 (LayerNorm2d + GELU, mask_decoder.py:59-70). */
int es3_ln_rows_gelu(const float* x, const float* w, const float* bias, float eps, void* y, long long M, int C, void* stream);
/* masks[b,k,p] = hyper[b,k_off+k,:] . up[b,p,:] (+ object gating) -> [B,K,HW] fp32 (mask_decoder.py:225-226). */
int es3_hyper_masks(const float* up, const float* hyper, const float* obj_logits, float no_obj, float* masks, int B, int HW,
                    int CU, int Ktot, int K, int k_off, void* stream);
/* Bilinear (align_corners=False) on NCHW fp32 planes; optional uint8 (x > thr) output (tracker_base.py:355-360). */
int es3_bilinear_nchw_f32(const float* in, float* out, void* bin, float thr, long long planes, int Hi, int Wi, int Ho,
                          int Wo, void* stream);

/* ------------------------------------------------------------------------------------------ RepViT / TinyViT */
/* Dense 3x3, stride 2, pad 1 with a narrow input (second patch-embed conv: repvit.py:222-223, tiny_vit.py:75-81) on
 * mma.sync.  x [B,H,W,Cin] bf16; w [9][Cout][Cin] bf16 (tap, out channel, in channel); folded-BN scale/bias;
 * out [B,Ho,Wo,Cout].  Instantiated: Cin 32 -> Cout 32/48/64, Cin 48 -> Cout 80/96 (narrower first convs are zero padded). */
int es3_conv3x3_s2_narrow_bf16(const void* x, const void* w, const float* scale, const float* bias, void* out, int B, int H,
                               int W, int Cin, int Cout, int act, void* stream);
/* SqueezeExcite pieces (timm.layers.SqueezeExcite, repvit.py:136,150): per-image channel means of x [B,HW,C] bf16
 * (ws: B*ceil(HW/128)*C floats; deterministic two-stage) and y = x * gate[b,c]. */
int es3_channel_mean(const void* x, float* ws, float* mean, int B, int HW, int C, void* stream);
int es3_scale_channels(const void* x, const float* gate, void* y, int B, int HW, int C, void* stream);

/* Window attention with the learned relative-position bias over zero-padded window partitions, head_dim 32, window 7 or 14
 * (tiny_vit.py:219-293, 344-375).  qkv [B*H*W, 3C] with per-head [q|k|v] blocks of 32; qkv_pad [3C] = qkv(LN(0)), the value
 * the reference's padded tokens take; bias [heads][ws^2][ws^2] fp32; out [B*H*W, C] bf16. */
int es3_win_attn_bias_bf16(const void* qkv, const void* qkv_pad, const float* bias, void* out, int B, int H, int W, int C,
                           int num_heads, int ws, float scale, void* stream);
/* LayerNorm over bf16 rows, C % 8 == 0 (TinyViT token stream: Attention.norm / Mlp.norm, tiny_vit.py:206,240). */
int es3_layernorm_bf16(const void* x, const float* gamma, const float* beta, float eps, void* y, long long M, int C, void* stream);

/* ------------------------------------------------------------------------------------------ stage-1 loss */
/* Masked MSE + masked cosine KD loss, forward (stage1/train_image_encoder_stage1.py:205-210, 271-307).
 * preds / teacher [B,C,E,E] fp32 NCHW; sizes_hw int32 [B][2] (h, w before padding); ws: B*ceil(E*E/256)*3 floats;
 * out3 = (loss, mse, cosine); per_sample [B][3] optional. */
int es3_kd_loss_fwd(const float* preds, const float* teacher, const int* sizes_hw, int B, int C, int E, int img_size,
                    float cosine_weight, float* ws, float* out3, float* per_sample, void* stream);
/* d loss / d preds of es3_kd_loss_fwd (masked MSE + cosine_weight * masked cosine, batch mean), times grad_scale and --
 * when scale_dev != NULL -- the device-resident loss scale scale_dev[0] (GradScaler.scale(loss).backward()).
 * per_sample: the [B][3] array es3_kd_loss_fwd wrote (its mask counts are the denominators).  dpreds [B,C,E,E] fp32. */
int es3_kd_loss_bwd(const float* preds, const float* teacher, const int* sizes_hw, const float* per_sample,
                    const float* scale_dev, float grad_scale, int B, int C, int E, int img_size, float cosine_weight,
                    float* dpreds, void* stream);

/* ------------------------------------------------------------------------------------------ optimiser (A20) */
/* Sum of squares + non-finite flag over a flat fp32 gradient arena (deterministic two-stage): norm_ws[0] = sum g^2 (raw,
 * still loss-scaled), norm_ws[1] = 1 if any inf / nan.  part_ws: es3_grad_norm_ws_floats(n) floats.
 * Replaces GradScaler.unscale_'s inf check + clip_grad_norm_'s norm (stage1/utils.py:341-368). */
long long es3_grad_norm_ws_floats(long long n);
int es3_grad_norm(const float* g, long long n, float* part_ws, float* norm_ws, void* stream);
/* One fused AdamW step over flat arenas p/g/m/v of n floats (torch.optim.AdamW update rule; stage1/optimizer.py:6-30 puts
 * 1-D params and biases in a no-decay group: here the first n_decay elements are the decay group).  The gradient is
 * multiplied by inv_world / state[0] (allreduce-sum -> mean, loss-scale unscale) and by the clip_grad_norm_ coefficient
 * min(1, max_norm / (norm + 1e-6)) computed from norm_ws on the device; when norm_ws[1] != 0 the update is skipped.
 * state (device, 4 floats): [0] loss scale, [1] growth tracker, [2] step count, [3] last total norm; advanced after the
 * update as GradScaler.update does (dynamic_scale: growth x after `growth_interval` clean steps, backoff x on inf). */
int es3_adamw_flat(float* p, const float* g, float* m, float* v, long long n, long long n_decay, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float max_norm, float inv_world, const float* norm_ws,
                   float* state, int dynamic_scale, float growth, float backoff, int growth_interval, void* stream);

/* ------------------------------------------------------------------------------------------ student backward (A20) */
/* The `loss.backward()` half of train_one_epoch (stage1/train_image_encoder_stage1.py:154-268) for the EfficientViT
 * student.  Activation gradients are bf16 [M][C] row-major (NHWC), parameter gradients fp32 and ACCUMULATED (+=) into the
 * destination; every reduction is two-stage in a fixed order (bit-reproducible).  Workspaces: the *_ws_floats helpers.
 *
 * Train-mode nn.BatchNorm2d of ConvLayer (efficientvit/nn/ops.py:39-80) over the raw conv output z [M][C] bf16:
 * mean / invstd (biased variance, eps) per channel, the folded scale = gamma invstd, shift = beta - mean scale, and the
 * running-stat update (momentum on the unbiased variance; running_* / num_batches_tracked may be NULL). */
long long es3_col_reduce_ws_floats(long long M, int C);
int es3_bn_stats(const void* z, long long M, int C, float eps, float momentum, const float* gamma, const float* beta, float* ws,
                 float* mean, float* invstd, float* scale, float* shift, float* running_mean, float* running_var,
                 long long* num_batches_tracked, void* stream);
/* out = act(scale[c] z + shift[c]) (+ residual): the normalise + activation pass (scale / shift / residual may be NULL). */
int es3_affine_act(const void* z, const float* scale, const float* shift, int act, const void* residual, void* out, long long M,
                   int C, void* stream);
/* Backward of act(scale z + shift) and of the BatchNorm producing (scale, shift).  g = da act'(scale z + shift);
 * mode 0: no norm (shift = conv bias): dbeta += sum g.  mode 1: eval-mode BN (mean / invstd = running stats;
 * set_bn_state with TRAIN.EVAL_BN_WHEN_TRAINING, train_image_encoder_stage1.py:310-314): dgamma, dbeta.  mode 2: batch
 * statistics (full BN backward).  Writes coef [3][C] so that dz = coef0 g + coef1 z + coef2 (es3_bn_act_bwd_apply).
 * act in {none, relu, hswish, gelu, relu6}.  dgamma / dbeta may be NULL. */
int es3_bn_act_bwd_reduce(const void* da, const void* z, const float* scale, const float* shift, int act, int mode,
                          const float* mean, const float* invstd, long long M, int C, float* ws, float* coef, float* dgamma,
                          float* dbeta, void* stream);
int es3_bn_act_bwd_apply(const void* da, const void* z, const float* scale, const float* shift, int act, const float* coef,
                         void* dz, long long M, int C, void* stream);
/* out = a + b, bf16 [M][C] with row strides in elements (gradient fan-in at residual joins / LiteMLA multi-scale). */
int es3_add_bf16(const void* a, long long lda, const void* b, long long ldb, void* out, long long ldo, long long M, int C,
                 void* stream);
/* Weight gradient of a 1x1 conv / nn.Linear: dW[n ldn + k ldk] += sum_m dz[m][n] x[m][k]  (mma.sync, contraction over
 * pixels).  With H > 0 the x row of pixel (b, y, x) is (b, y + dy, x + dx), zero outside the H x W map: one tap of a dense
 * 3x3 conv (head.3, stage1/model.py:198).  ws: es3_wgrad_pw_ws_floats(M, N, K) floats. */
long long es3_wgrad_pw_ws_floats(long long M, int N, int K);
int es3_wgrad_pw(const void* dz, long long lddz, const void* x, long long ldx, long long M, int N, int K, int H, int W, int dy,
                 int dx, float* ws, float* dW, long long ldn, long long ldk, void* stream);
/* Dense 3x3 weight gradient on tcgen05: es3_transpose_pad_bf16 lays in [B,H,W,C] out as out [C][Mp], Mp = B (H+2) Wp (Wp >= W+2,
 * multiple of 8), every image inside a zero frame and shifted by dx in x; a tap (ky, kx) is then the plain GEMM
 * dW[ky][kx] = dYp^T[:, Wp : Mp-Wp] . Ap_{kx-1}^T[:, Wp + (ky-1) Wp : ...]^T (es3_gemm_bf16, fp32 out), added into the
 * [N][C][3][3] gradient by es3_accumulate_strided (dst[(i / inner) ld_outer + (i % inner) ld_inner] += src[i]). */
int es3_transpose_pad_bf16(const void* in, void* out, int B, int H, int W, int C, int Wp, int dx, void* stream);
int es3_accumulate_strided(const float* src, long long n, int inner, long long ld_outer, long long ld_inner, float* dst,
                           void* stream);
/* Depthwise k x k conv (pad k/2): input gradient dx [B,H,W,C] from dz [B,Ho,Wo,C] and w [k*k][C] fp32 (any stride), and
 * weight gradient dW [C][k*k] (torch layout) += from dz and the layer input x (pixel stride ldx: channel slices allowed). */
int es3_dwconv_bwd_data(const void* dz, const float* w, void* dx, int B, int H, int W, int C, int ks, int stride, void* stream);
long long es3_dwconv_wgrad_ws_floats(int B, int H, int W, int C, int ks, int stride);
int es3_dwconv_wgrad(const void* dz, const void* x, long long ldx, int B, int H, int W, int C, int ks, int stride, float* ws,
                     float* dW, void* stream);
/* Backward of es3_litemla_attn_generic (head dim 16 | 32; efficientvit_b2 uses 32): same contract as es3_litemla_attn_bwd with
 * kv_part = the workspace es3_litemla_attn_generic filled (nchunk_f = ceil(HW / 128)).  GPU parity: test_litemla_attn_bwd_generic. */
long long es3_litemla_bwd_generic_ws_floats(int B, int HW, int heads2, int dim);
int es3_litemla_attn_bwd_generic(const void* ms, long long ld, const void* dy, long long lddy, const float* kv_part, int nchunk_f,
                                 float* dkv_ws, void* dms, long long lddms, int B, int HW, int heads2, int dim, float eps, void* stream);
/* TinyViT backward pieces (tinyvit_bwd.cu).  es3_layernorm_bwd: nn.LayerNorm backward over bf16 rows [M][C]
 * (tiny_vit.py:205,262): dx = dLN(x) (+ dres), dgamma += sum dy xhat, dbeta += sum dy.  es3_win_attn_bias_bwd: backward of
 * es3_win_attn_bias_bf16 (tiny_vit.py:264-293) on a token map whose H, W are multiples of ws: dqkv in the forward's layout and the
 * per-window score gradients dS [B nWin][ldS] fp32 (row = [heads][ws^2][ws^2]); the bias gradient is the column sum of dS,
 * es3_colsum_f32: out[c] += sum_r src[r * ld + c] in a fixed order (ws: es3_colsum_f32_ws_floats(M, L) floats). */
long long es3_layernorm_bwd_ws_floats(long long M, int C);
int es3_layernorm_bwd(const void* x, const void* dy, const float* gamma, const void* dres, float eps, void* dx, long long M, int C,
                      float* ws, float* dgamma, float* dbeta, void* stream);
int es3_win_attn_bias_bwd(const void* qkv, const void* dout, const float* bias, void* dqkv, void* dS, long long ldS, int B, int H, int W,
                          int C, int num_heads, int ws, float scale, void* stream);
long long es3_colsum_f32_ws_floats(long long M, int L);
int es3_colsum_f32(const float* src, long long ld, long long M, int L, float* ws, float* out, void* stream);
/* Shared-memory tiled variant of es3_dwconv_wgrad for stride 1 and C % 32 == 0 (same result contract).  The default
 * route for these shapes since round 2 (GPU parity: test_dwconv_wgrad_tiled). */
/* Stride-1 depthwise conv (ks 3 | 5, pad ks/2, C % 32 == 0) on mma.sync with diagonal tap operands: same contract as
 * es3_dwconv_tiled_bf16 at stride 1, taps rounded to bf16 (nn.Conv2d(groups=C): efficientvit/nn/ops.py:39-80, repvit.py:84-122,
 * tiny_vit.py:97-133; also the backward-data pass of those layers, on flipped taps). */
int es3_dwconv_tc_bf16(const void* x, long long ldx, const float* w, const float* bias, void* out, long long ldo, int B, int H, int W, int C,
                       int ks, int act, void* stream);
/* bf16-representable taps (as fp32, [KK][C] tap-major) whose per-channel SUM stays at the fp32 tap sum: the operand preparation of
 * es3_dwconv_tc_bf16 (nearest rounding alone costs TinyViT 1e-2 of embedding accuracy, csrc/dw_tc.cu). */
int es3_round_taps_sum_bf16(const float* w, float* out, int KK, int C, void* stream);

/* Register sliding-window depthwise weight gradient over shared-memory tiles: same contract as es3_dwconv_wgrad for C % 32 == 0
 * (stride 1 | 2, ks 3 | 5); the route ops.dwconv_wgrad takes for such shapes (autograd of nn.Conv2d(groups=C), ops.py:39-80). */
long long es3_dwconv_wgrad_win_ws_floats(int B, int H, int W, int C, int ks, int stride);
int es3_dwconv_wgrad_win(const void* dz, const void* x, long long ldx, int B, int H, int W, int C, int ks, int stride, float* ws, float* dW,
                         void* stream);
long long es3_dwconv_wgrad_tiled_ws_floats(int B, int H, int W, int C, int ks);
int es3_dwconv_wgrad_tiled(const void* dz, const void* x, long long ldx, int B, int H, int W, int C, int ks, float* ws, float* dW,
                           void* stream);
/* SqueezeExcite backward (timm SqueezeExcite, repvit.py:23,136) in one launch each instead of per-image loops:
 * dgate[b][c] += sum_p dy x; dx = dy * gate[b][c] + add[b][c].  dy, x, dx: [B][HW][C] bf16.  Not on the default path yet
 * (no GPU parity run; ops.SE_BWD_BATCHED). */
long long es3_se_bwd_ws_floats(int B, int HW, int C);
int es3_se_bwd_dgate(const void* dy, const void* x, int B, int HW, int C, float* ws, float* dgate, void* stream);
int es3_se_bwd_apply(const void* dy, const float* gate, const float* add, void* dx, int B, int HW, int C, void* stream);
/* Weight gradient of the 3 -> Cout stride-2 stem conv on the fp32 NCHW image (efficientvit/backbone.py:47-56):
 * dW [Cout][3][3][3] += . */
long long es3_stem_wgrad_ws_floats(int B, int H, int W, int Cout);
int es3_stem_wgrad(const float* img, const void* dz, int B, int H, int W, int Cout, float* ws, float* dW, void* stream);
/* Adjoint of es3_bilinear_nhwc_to_nchw: dout [B,C,Ho,Wo] fp32 NCHW -> din [B,Hi,Wi,C] bf16 NHWC. */
int es3_bilinear_bwd(const float* dout, void* din, int B, int Hi, int Wi, int C, int Ho, int Wo, void* stream);
/* Backward of es3_litemla_attn[_tc] (ReLU linear attention, head dim 16, ops.py:592-621): dy [B,HW,lddy] (head h at
 * [16h, 16h+16)) -> dms [B,HW,lddms] in the q|k|v layout of ms.  kv_part: the partial KV sums the forward call left in its
 * workspace (nchunk_f = ceil(HW / 512)); dkv_ws: es3_litemla_bwd_ws_floats floats. */
long long es3_litemla_bwd_ws_floats(int B, int HW, int heads2);
int es3_litemla_attn_bwd(const void* ms, long long ld, const void* dy, long long lddy, const float* kv_part, int nchunk_f,
                         float* dkv_ws, void* dms, long long lddms, int B, int HW, int heads2, float eps, void* stream);

/* Narrow pointwise conv / its input gradient on the CUDA cores (pw_small.cu): out[m][n] = sum_k a[m][k] w[n][k] (+ residual), bf16 in /
 * out, fp32 accumulation, K, N in {16, 32, 64} (not both 64).  Returns -1 without setting an error for any other shape / alignment:
 * callers fall back to es3_gemm_bf16 (efficientvit/nn/ops.py:273-367, the 16..64-channel 1x1 convs of stages 0-1). */
int es3_pw_small_bf16(const void* a, long long lda, const void* w, long long ldw, void* out, long long ldo, const void* residual,
                      long long ldr, long long M, int N, int K, void* stream);
/* Weight gradient of pointwise convs / linears on tcgen05 (wgrad_tc.cu): dW[n * ldn + k] += sum_m dz[m * lddz + n] * x[m * ldx + k]
 * as a split-K UMMA with both operands MN-major (TMA tiles of [64 px][64 ch] are the transposed operand layout), deterministic
 * two-stage sum.  Returns -1 without setting an error for shapes it does not take (N or K not multiples of 64, M < 64, unaligned
 * strides): callers fall back to es3_wgrad_pw.  ws: es3_wgrad_tc_ws_floats(M, N, K) floats. */
long long es3_wgrad_tc_ws_floats(long long M, int N, int K);
int es3_wgrad_tc(const void* dz, long long lddz, const void* x, long long ldx, long long M, int N, int K, float* ws, float* dW,
                 long long ldn, void* stream);
/* ---- strict (fp32-class) precision mode (strict_f32.cu): fp32 activations / weights / FMA accumulation on the CUDA cores, the
 * parity mode for north_star's tolerances (embeddings rtol 1e-4, mask logits rtol 1e-3, binary masks bit-exact) against the
 * reference's PyTorch fp32 path (its LiteMLA is forced to fp32: efficientvit/nn/ops.py:586-589).  Same epilogue contract as
 * es3_gemm_bf16: out = act(scale[n] * A W^T + bias[n]) (+ residual), the activation after the residual when act_after_res. */
int es3_sgemm_f32(const float* A, long long lda, const float* W, long long ldw, float* out, long long ldo, long long M, int N, int K,
                  const float* scale, const float* bias, int act, const float* residual, long long ldr, int act_after_res, void* stream);
/* cols[(b,oy,ox)][(ky*ks+kx)*C + c] of an NHWC fp32 map (nchw != 0: of the NCHW fp32 image), zero padding: every dense, strided or
 * image convolution (nn.Conv2d: ops.py:39-80, stage1/model.py:194-199, necks.py) becomes es3_sgemm_f32 on it. */
int es3_im2col_f32(const float* x, float* cols, int B, int H, int W, int C, int ks, int stride, int pad, int nchw, void* stream);
/* depthwise k x k (odd k, same padding), w [k*k][C] tap-major, y = act(scale[c] * conv + bias[c]); NHWC fp32 with pixel strides
 * ldx / ldy floats (channel slices of a wider map). */
int es3_dwconv_f32(const float* x, long long ldx, const float* w, const float* scale, const float* bias, float* y, long long ldy, int B,
                   int H, int W, int C, int ks, int stride, int act, void* stream);
/* LiteMLA.relu_linear_att (ops.py:584-621) on fp32: ms [B][HW][ld], head h = q | k | v at columns [3 dim h, 3 dim (h+1));
 * out [B][HW][ldo], head h at columns [dim h, dim (h+1)).  ws: es3_litemla_attn_f32_ws_floats(B, HW, heads, dim) floats. */
long long es3_litemla_attn_f32_ws_floats(int B, int HW, int heads, int dim);
int es3_litemla_attn_f32(const float* ms, long long ld, float* ws, float* out, long long ldo, int B, int HW, int heads, int dim, float eps,
                         void* stream);
/* F.interpolate(bilinear, align_corners=False) NHWC fp32 -> NCHW fp32 (stage1/model.py:203-210); equal sizes = layout change. */
int es3_bilinear_nhwc_f32_to_nchw(const float* x, float* y, int B, int Hi, int Wi, int C, int Ho, int Wo, void* stream);
/* fp32 twins of es3_attn_few_keys / es3_ln_rows_gelu (sam/transformer.py:168-176, mask_decoder.py:59-70) and the elementwise tail
 * y = act(x + bias[c]) + residual (act_after_res: act(x + bias[c] + residual)) of the strict ConvTranspose2d path. */
int es3_attn_few_keys_f32(const float* q, long long ldq, const float* k, const float* v, long long ldkv, float* out, long long ldo, int B,
                          int H, int head_dim, int Nq, int Tk, float scale, void* stream);
int es3_ln_rows_gelu_f32(const float* x, const float* w, const float* bias, float eps, float* y, long long M, int C, void* stream);
int es3_bias_act_res_f32(const float* x, const float* bias, const float* residual, float* y, long long total, int C, int act,
                         int act_after_res, void* stream);

/* More of the strict mode: nn.LayerNorm over rows of any width (tiny_vit.py:235, 259), in-place 2-D axial RoPE on fp32 q | k heads (vitdet.py:68-90), fp32 softmax attention on the ViT qkv layout
 * (windows gathered in place, vitdet.py:93-139, 466-515; TinyViT's biased, zero-padded windows, tiny_vit.py:258-287, 352-372), SqueezeExcite gating y = x * gate[b][c] (timm SqueezeExcite, repvit.py:23,136). */
int es3_ln_rows_f32(const float* x, const float* w, const float* bias, float eps, float* y, long long M, int C, void* stream);
int es3_rope_f32(float* qkv, long long ld, long long rows, const float* table, int rope_cols, int H, int W, int win, void* stream);
int es3_attention_f32(const float* qkv, float* out, const float* bias, const float* pad_row, int B, int H, int W, int ld, int num_heads,
                      int head_dim, int q_off, int k_off, int v_off, int head_stride, int win, float scale, void* stream);
int es3_scale_channels_f32(const float* x, const float* gate, float* y, int B, long long HW, int C, void* stream);

/* ------------------------------------------------------------------------------------------ input preprocessing */
/* Decoded images of any size -> antialiased bilinear resize (torch's _upsample_bilinear2d_aa, align_corners=False: width pass,
 * fp32 intermediate, height pass) -> out = resized * a_c + b_c -> zero pad -> fp32 NCHW [B,3,S,S].  Replaces the loaders'
 * pil_to_tensor -> ResizeLongestSide.apply_image_torch -> norm -> pad (stage1/data/sa1b_dataset.py:68-69, 163-171, 216-227,
 * coco_dataset.py:146-153, transforms.py:48-54) and SAM2Transforms' ToTensor -> Resize((S,S)) -> Normalize (sam1_utils.py:17-41).
 * table: [B][16] int64 on the device, one descriptor per image: {device address, element strides of channel / row / column,
 * in_h, in_w, out_h, out_w (<= S), dtype (0 uint8, 1 fp32), staged planes (1 interleaved, 3 planar), input columns per staging
 * chunk, taps per output along x / y, offsets (floats) of the x / y tap records in `taps`, unused}.  affine: [B][6] fp32
 * (a_0..2, b_0..2).  taps: fp32 workspace of (K + 2) floats per output coordinate and axis.  max_out: largest out_h / out_w.
 * Two kernels: tap tables, then the fused resize. */
int es3_preprocess_images(const long long* table, const float* affine, float* taps, int B, int S, int max_out, float* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ES3_H_ */
