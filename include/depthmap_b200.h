/*
 * depthmap_b200 — C-ABI of the B200-native depth -> 16-bit depth -> stereo / normal-map hot path.
 *
 * Every entry point replaces one Python-level operator of thygate/stable-diffusion-webui-depthmap-script
 * (reference @ e4df29bc); the reference has no FFI of its own, so the binding a maintainer adds is the ctypes stub
 * shown in INTEGRATION.md.  Conventions:
 *   - plain C types only; every pointer is DEVICE memory owned by the caller unless it is named *_host;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), performs no host synchronisation
 *     and allocates nothing: scratch comes from the caller through (workspace, workspace_bytes), sized by the
 *     matching *_workspace_bytes() query;
 *   - return value: DM_OK (0) or a negative dm_status; dm_last_error() gives the message for the calling thread;
 *   - images are batched, B images of identical H x W, densely packed: rgb = [B][H][W][3] u8, depth = [B][H][W].
 */
#ifndef DEPTHMAP_B200_H
#define DEPTHMAP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dm_status {
    DM_OK = 0,
    DM_E_INVALID = -1,      /* bad argument (Python face raises ValueError / the reference's own exception) */
    DM_E_CUDA = -2,         /* CUDA runtime error other than OOM */
    DM_E_OOM = -3,          /* message contains "out of memory" so src/core.py:310 still recognises it */
    DM_E_UNSUPPORTED = -4,  /* valid request outside the implemented envelope (e.g. row too wide for smem) */
    DM_E_WORKSPACE = -5     /* workspace too small */
} dm_status;

const char *dm_last_error(void);
int dm_version(void);
/* Name of the device the library would run on, "" if no CUDA device; never throws. */
int dm_device_name(char *buf_host, int buf_len);

/* ---------------------------------------------------------------------------------------------------------------
 * N1 — funnel post-processing of a model prediction: per-image min/max, invert, optional "Range" clip, normalise,
 * convert_to_i16.            replaces  src/core.py:189-211 (model branch) + src/core.py:44-50
 * clip_mode: 0 none, 1 "Range" (clip_far / clip_near as in GenerationOptions CLIPDEPTH_FAR / CLIPDEPTH_NEAR).
 * All arithmetic float32, as numpy does it.  Degenerate image (max-min <= DBL_EPSILON) -> all-zero output.
 * degenerate_flags (optional, may be NULL): int32[B], 1 where the image was degenerate.
 * ------------------------------------------------------------------------------------------------------------- */
size_t dm_normalize_u16_workspace_bytes(int B);
int dm_normalize_u16(const float *pred, int B, int H, int W, int invert, int clip_mode, float clip_far,
                     float clip_near, uint16_t *depth_out, int32_t *degenerate_flags, void *workspace,
                     size_t workspace_bytes, void *stream);

/* N1, "Outliers" clip:  replaces src/core.py:200-202  (fb, nb = np.percentile(out, [far*100, near*100]); np.clip(out, fb, nb))
 * followed by the same normalise + convert_to_i16 tail, which numpy evaluates in FLOAT64 here (np.percentile returns
 * float64 scalars and np.clip promotes the float32 image).  np.percentile's "linear" method reads two order statistics
 * per percentile: ranks[0..1] / ranks[2..3] are the 0-based ranks (ascending, after the optional sign flip) of the far /
 * near percentile and gamma_far / gamma_near the float64 interpolation weights; both depend only on H*W and the two
 * fractions and are computed by the host face with numpy's own expression (core.percentile_plan). */
/* convert_to_i16 (src/core.py:44-50) of float64 values in [0, 1) (custom depth maps, src/core.py:146-174) */
int dm_convert_to_i16_f64(const double *x, long long n, uint16_t *out, void *stream);
size_t dm_normalize_u16_outliers_workspace_bytes(int B);
int dm_normalize_u16_outliers(const float *pred, int B, int H, int W, int invert, const int64_t ranks[4], double gamma_far,
                              double gamma_near, uint16_t *depth_out, int32_t *degenerate_flags, void *workspace,
                              size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * S1-S5 — stereo pair: per-row depth-driven warp + gap fill + packing.
 *            replaces  src/stereoimage_generation.py:13-74 (create_stereoimages),
 *                      :77-92 (apply_stereo_divergence), :95-159 (naive family), :162-283 (polylines), :286-307
 * depth_kind: DM_DEPTH_U16 -> `depth` is uint16; (d-min)/(max-min) is evaluated in fp64 per image on the device;
 *             DM_DEPTH_ND64 -> `depth` is float64 already-normalised depth (host face handles exotic dtypes).
 * Per eye e in {0 = left, 1 = right}: div_px[e], sep_px[e] (pixels, as the reference computes them in Python) and
 * eye_mode[e]: DM_EYE_WARP (run the algorithm), DM_EYE_IDENTITY (reference skips the warp: eye = source image),
 * DM_EYE_SKIP (eye not needed for the requested packing).
 * pack: DM_PACK_STRIDED  eye e is written to out[e] with dst_row_stride[e] / dst_img_stride[e] (bytes); covers
 *                        left-right, right-left, top-bottom, bottom-top, left-only, only-right by pointer arithmetic;
 *       DM_PACK_ANAGLYPH out[0] receives R from eye a0, G,B from eye 1-a0 where a0 = anaglyph_red_eye (0: red-cyan,
 *                        1: cyan-red-reverse); uses dst strides [0].
 * ------------------------------------------------------------------------------------------------------------- */
enum { DM_DEPTH_U16 = 0, DM_DEPTH_ND64 = 1 };
enum { DM_FILL_NONE = 0, DM_FILL_NAIVE = 1, DM_FILL_NAIVE_INTERPOLATING = 2, DM_FILL_POLYLINES_SOFT = 3,
       DM_FILL_POLYLINES_SHARP = 4 };
enum { DM_EYE_WARP = 0, DM_EYE_IDENTITY = 1, DM_EYE_SKIP = 2 };
enum { DM_PACK_STRIDED = 0, DM_PACK_ANAGLYPH = 1 };

typedef struct dm_stereo_params {
    double div_px[2];
    double sep_px[2];
    double exponent;          /* stereo_offset_exponent */
    int32_t eye_mode[2];
    int32_t fill;             /* DM_FILL_* */
    int32_t pack;             /* DM_PACK_* */
    int32_t anaglyph_red_eye; /* 0 or 1 */
    int32_t depth_kind;       /* DM_DEPTH_* */
    int32_t reserved;
    int64_t dst_row_stride[2];
    int64_t dst_img_stride[2];
} dm_stereo_params;

/* The other packings of create_stereoimages (:56-73) from a left | right pair sbs [B,H,2W,3]: mode 0 left-right, 1 right-left,
 * 2 top-bottom, 3 bottom-top, 4 red-cyan-anaglyph, 5 left-only, 6 only-right, 7 cyan-red-reverseanaglyph (a request with several
 * modes computes the eyes once and packs each mode with this). */
int dm_stereo_pack(const uint8_t *sbs, int B, int H, int W, int mode, uint8_t *out, void *stream);
/* apply_stereo_divergence's (d - min) / (max - min) (:79-81) for depth maps that are not uint16, in numpy's dtype rules
 * (dtype 0 float32, 1 float64, 2 int64) -> float64 [B, n] for DM_DEPTH_ND64; flat_out (optional): 1 where max == min */
int dm_depth_to_nd64(const void *depth, int dtype, int B, long long n, double *nd_out, int32_t *flat_out, void *stream);
size_t dm_stereo_workspace_bytes(int B, int H, int W);
int dm_stereo(const uint8_t *rgb, const void *depth, int B, int H, int W, const dm_stereo_params *params_host,
              uint8_t *out0, uint8_t *out1, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * M1 — tangent-space normal map.           replaces  src/normalmap_generation.py:5-56 (create_normalmap)
 * pre_blur / sobel / post_blur: kernel sizes, <= 0 means None (sobel <= 0 selects the np.gradient branch).
 * ------------------------------------------------------------------------------------------------------------- */
size_t dm_normalmap_workspace_bytes(int B, int H, int W, int pre_blur, int sobel, int post_blur);
int dm_normalmap(const uint16_t *depth, int B, int H, int W, int pre_blur, int sobel, int post_blur, int invert,
                 uint8_t *rgb_out, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * D2-D7 — building blocks of the depth networks (ViT backbone + DPT decoder).  The Python ModelHolder
 * (stable-diffusion-webui-depthmap-script_b200/depthmap_generation.py) strings these together per model; each call
 * is one or two kernel launches on `stream`.  fp16 operands, fp32 accumulation, fp32 residual stream.
 *   replaces: torch nn.Module.forward of DepthAnythingV2 (ddepth_anything_v2/depth_anything_v2/dpt.py:176-184,
 *   dinov2.py:297-321, dinov2_layers/{attention,block,mlp}.py), DPTDepthModel (dmidas/dpt_depth.py:110-166,
 *   dmidas/backbones/{beit,utils}.py, dmidas/blocks.py) and the surrounding numpy/cv2 pre/post-processing
 *   (dpt.py:196-221, src/depthmap_generation.py:455-499,548-559).
 * ------------------------------------------------------------------------------------------------------------- */
enum { DM_EPI_STORE_F16 = 0, DM_EPI_RESID_F32 = 1, DM_EPI_PIXSHUF = 2, DM_EPI_HEAD = 3, DM_EPI_STORE_F32 = 4 };
enum { DM_ACT_NONE = 0, DM_ACT_GELU = 1, DM_ACT_RELU = 2 };

/* C[M,N] = A[M,K] * W[N,K]^T with a fused epilogue (tcgen05 tensor cores, TMA-fed).  K % 64 == 0, N % 32 == 0. */
typedef struct dm_gemm_desc {
    int32_t M, N, K;
    int32_t epi, act;        /* DM_EPI_*, DM_ACT_* */
    const float *bias;       /* [N] fp32 or NULL */
    void *C; int32_t ldc;    /* fp16 output (STORE_F16 / PIXSHUF) */
    void *C2;                /* optional relu(C) copy, same layout */
    const void *R; int32_t ldr;    /* optional fp16 residual added before the store */
    const void *R2; int32_t ldr2;  /* optional second fp16 residual */
    float *X; int32_t ldx;   /* fp32 residual stream (RESID_F32: X += gamma*(acc+bias)) or fp32 output (STORE_F32 / HEAD) */
    const float *gamma;      /* [N] LayerScale (RESID_F32) or the fused 1x1 head weights (HEAD) */
    float head_b2;           /* HEAD: bias of the fused 1x1 conv */
    int32_t ps_s, ps_cout, ps_h, ps_w;  /* PIXSHUF: ConvTranspose2d(kernel = stride = ps_s) scatter geometry */
} dm_gemm_desc;

int dm_gemm_ex(const void *A, int lda, const void *W, int ldw, const dm_gemm_desc *desc_host, void *stream);
/* 3x3 stride-1 pad-1 conv as implicit GEMM: act NHWC fp16 [B,H,W,Cin], Wt fp16 [Cout, 9*Cin] ordered (ky,kx,cin);
 * desc->N = Cout; M and K are derived. */
int dm_conv3x3_ex(const void *act, int B, int H, int W, int Cin, const void *Wt, const dm_gemm_desc *desc_host, void *stream);
/* convenience wrappers used by the unit tests */
int dm_gemm_f16(const void *A, int lda, const void *W, int ldw, const float *bias, void *C, int ldc, int M, int N, int K,
                int act, int out_f32, void *stream);
int dm_conv3x3_f16(const void *act, int B, int H, int W, int Cin, const void *Wt, const float *bias, void *out, int Cout,
                   int relu, void *stream);
/* softmax(scale * Q K^T [+ bias]) V for head_dim 64 straight from the packed qkv activation [B*N, 3*H*64] (fp16);
 * bias: optional fp16 [H, N, bias_ld]; out: fp16 [B*N, H*64]. */
int dm_attention_f16(const void *qkv, int B, int N, int H, float scale, const void *bias, int bias_ld, void *out, void *stream);
/* Same, with the BEiT relative-position bias generated on the fly (dmidas/backbones/beit.py:29-62): rel_table_log2e is
 * fp32 [H, nrd] = the per-head bias table already resized to the gh x gw window, multiplied by log2(e);
 * nrd = (2gh-1)(2gw-1)+3, N = gh*gw+1 tokens (class token first).  No [H,N,N] bias tensor is read by the kernel.
 * rel_rowmax_log2e (fp32 [H, N], the per-query maximum of the bias) was an input of the round-1 kernel; the current kernel computes
 * exact row maxima itself and ignores it: pass NULL (the parameter stays for ABI stability). */
int dm_attention_relpos_f16(const void *qkv, int B, int gh, int gw, int H, float scale, const float *rel_table_log2e,
                            const float *rel_rowmax_log2e, int nrd, void *out, void *stream);
/* uint8 RGB [B,H,W,3] -> (cv2-style bicubic resize to net_h x net_w) -> (x/255 - mean)/std -> fp16 patch matrix
 * [B*(net_h/patch)*(net_w/patch), kpad], K ordered (c, ky, kx); network channel c reads source channel chan_map[c]. */
int dm_preprocess_patchify(const uint8_t *rgb, int B, int H, int W, int net_h, int net_w, int patch, const float *mean_host,
                           const float *std_host, const int *chan_map_host, void *out, int kpad, void *stream);
/* X[b,0,:] = cls + pos[0]; X[b,1+p,:] = pe[b*Np+p,:] + pos[1+p]  (pos may be NULL); X fp32 [B, Np+1, C] */
int dm_assemble_tokens(const void *pe, const float *cls, const float *pos, float *X, int B, int Np, int C, void *stream);
/* LayerNorm over the last dim of fp32 x [rows, C] -> fp16; drop_first != 0 skips token 0 of every image (tokens_per_img) */
int dm_layernorm_f16(const float *x, long long rows, int C, const float *gamma, const float *beta, float eps, void *out,
                     int tokens_per_img, int drop_first, void *stream);
int dm_resize_bilinear_nhwc_f16(const void *in, int B, int Hin, int Win, int C, void *out, int Hout, int Wout, void *stream);
/* mode 0: bilinear align_corners=True; mode 1: bicubic align_corners=False */
int dm_resize_f32(const float *in, int B, int Hin, int Win, float *out, int Hout, int Wout, int mode, void *stream);
int dm_im2col_s2_f16(const void *in, int B, int H, int W, int C, void *out, void *stream);
/* MiDaS ProjectReadout input: out[b*(N-1)+p, :] = [x[b,1+p,:], x[b,0,:]] (fp32 -> fp16), x fp32 [B, N, C] */
int dm_concat_readout_f16(const float *x, int B, int N, int C, void *out, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * D7 — ZoeDepth-NK / -N / -K on top of the DPT-BEiT core (csrc/zoe_kernels.cu).   replaces
 *   dzoedepth/models/depth_model.py:57-152 (pad + flip test-time augmentation), base_models/midas.py:175-186 (PrepForMidas),
 *   zoedepth_nk/zoedepth_nk_v1.py:159-243 (router, seed bins, attractors, conditional log-binomial),
 *   zoedepth/zoedepth_v1.py:120-186 (single metric head), layers/localbins_layers.py:29-68 (normed seed bins),
 *   layers/attractor.py:127-208, layers/dist_layers.py:29-121, layers/patch_transformer.py:29-92.
 * Forward index f = 2*b + flip: image b and its horizontal flip go through the network as one batch of 2B forwards.
 * `logits` is fp32 [F, lld]: columns 0 / 1 are the router's nyu / kitti logits of that forward; every head kernel picks
 * the routed head itself (argmax, first index on ties, as torch.argmax) — no host synchronisation.
 * ------------------------------------------------------------------------------------------------------------- */
/* uint8 RGB [B,H,W,3] -> /255 -> reflect pad (pad_h, pad_w) -> flip for odd f -> bilinear align_corners=True resize to
 * net_h x net_w -> (x - 0.5) / 0.5 -> fp16 patch matrix [2B * gh * gw, kpad], kpad = 3*patch^2 */
int dm_zoe_preprocess_patchify(const uint8_t *rgb, int B, int H, int W, int pad_h, int pad_w, int net_h, int net_w, int patch, void *out,
                               int kpad, void *stream);
/* x = LayerNorm(x) in place (fp32 [rows, 128]) + fp16 copy: post-norm nn.TransformerEncoderLayer of the router */
int dm_layernorm_post_f16(float *x, long long rows, int C, const float *gamma, const float *beta, float eps, void *out, void *stream);
/* self-attention of the router: qkv fp16 [F*S, 3*heads*32] (q | k | v) -> out fp16 [F*S, heads*32] */
int dm_attention_small_f16(const void *qkv, int F, int S, int heads, float scale, void *out, void *stream);
int dm_cast_f32_f16(const float *x, long long n, void *out, void *stream);
/* out[r, 0..63] = softplus(seed[r, head*64 .. head*64+63]) for the routed head of row r's forward */
int dm_zoe_select_softplus(const float *seed, int ld, const float *logits, int lld, int F, int rows_per_fwd, float *out, void *stream);
/* out = a + bilinear_align_corners(b_small -> H x W); NHWC fp16 */
int dm_resize_add_nhwc_f16(const void *a, const void *b_small, int B, int Hs, int Ws, int C, void *out, int H, int W, void *stream);
/* AttractorLayerUnnormed (inverse attractor, mean of 16): A fp32 [F*H*W, lda] pre-softplus, routed head's 16 columns at
 * head*32; b_prev fp32 [F,Hp,Wp,64] is resized (bilinear, align_corners) to H x W; b_out fp32 [F,H,W,64] */
int dm_zoe_attractor(const float *A, int lda, const float *logits, int lld, const float *b_prev, int F, int Hp, int Wp, int H, int W,
                     float *b_out, void *stream);
/* Single-head attractor layer of ZoeDepth-N / -K (inverse attractor, mean over n_attractors in {16, 8, 4, 1}).  A fp32
 * [F*H*W, lda], the layer's last 1x1 conv before its activation.  normed = 0 (AttractorLayerUnnormed): attractor i is
 * softplus(A[:, i]).  normed = 1 (AttractorLayer): attractor i is relu(A[:, 2i]) + 1e-3; with B_sorted != NULL also
 * B_sorted fp32 [F,H,W,64] = clip(sort_ascending((max - min) * b_out + min), min, max) per pixel.  b_prev / b_out as in
 * dm_zoe_attractor (b_out is the normed b_new for normed = 1) */
int dm_zoe_attractor_single(const float *A, int lda, int n_attractors, int normed, const float *b_prev, int F, int Hp, int Wp, int H, int W,
                            float min_depth, float max_depth, float *b_out, float *B_sorted, void *stream);
/* SeedBinRegressor's normed bin centres, rescaled to [0, 1] as ZoeDepth-K's first b_prev: per row r of seed fp32 [rows, ld]
 * (64 used, before the final ReLU): w = relu(seed) + 1e-3 normalised to sum max - min, edges = cumsum([min, w]),
 * out fp32 [rows, 64] = (midpoints of the edges - min) / (max - min) */
int dm_zoe_seed_normed(const float *seed, int ld, long long rows, float min_depth, float max_depth, float *out, void *stream);
/* ConditionalLogBinomial + expectation over the 64 bin centres, per net pixel.  o32: relu'd out_conv activation fp16
 * [F,nh,nw,ldo] (32 channels used); ze fp32 [F,h3,w3,ldz] = W_e . b_emb (head at column head*64, 40 used); bc fp32
 * [F,h3,w3,64] bin centres; wo [2][32][40], b0 [2][40], w2 [2][4][40], b2 [2][4] fp32 device arrays; out fp32 [F,nh,nw] */
int dm_zoe_clb_final(const void *o32, int ldo, const float *ze, int ldz, const float *bc, const float *logits, int lld, const float *wo,
                     const float *b0, const float *w2, const float *b2, int F, int nh, int nw, int h3, int w3, float min_temp, float max_temp,
                     float *out, void *stream);
/* dm_zoe_clb_final for the single metric head of ZoeDepth-N / -K: 161 inputs = out_conv (32) + relative depth (1) + bin
 * embedding (128), 80 hidden units, no router.  The relative depth is relu(w_rel . out_conv + b_rel) (w_rel fp32 [32]: the
 * core's last 1x1 conv).  ze fp32 [F,h3,w3,ldz]: W_e . b_emb at columns 0..79; wo [32][80], wr [80] (relative-depth column),
 * b0 [80], w2 [4][80], b2 [4] fp32 device arrays */
int dm_zoe_clb_final_single(const void *o32, int ldo, const float *ze, int ldz, const float *bc, const float *wo, const float *wr, const float *b0,
                            const float *w2, const float *b2, const float *w_rel, float b_rel, int F, int nh, int nw, int h3, int w3,
                            float min_temp, float max_temp, float *out, void *stream);
/* out[b] = mean(crop(bicubic(d[2b])), unflip(crop(bicubic(d[2b+1])))): d fp32 [2B,nh,nw] -> out fp32 [B,H,W] */
int dm_zoe_tta_combine(const float *d, int B, int nh, int nw, int pad_h, int pad_w, int H, int W, float *out, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * §8(f) rank 1 — video mode's cross-frame normalisation.    replaces  src/video_mode.py:103-128 (process_predicitons)
 * Frames are fp32 [count, hw] device arrays.  Each step is its own call so that, when the frames of a clip are sharded
 * over GPUs, the host can put the (tiny) collective between two steps: all-reduce MIN/MAX of lohi[2] after
 * dm_video_minmax; all-reduce SUM of the int32[1024] histograms at byte offset 32 of `workspace` between
 * dm_video_select_hist and dm_video_select_pick.  Bit-exact with numpy (float32 for 'none', float64 for 'experimental').
 * ------------------------------------------------------------------------------------------------------------- */
size_t dm_video_workspace_bytes(void);
/* 5-tap temporal blend; `frames` holds global frames [base_global, base_global+count), out gets blended [out_first, +out_count) */
int dm_video_blend(const float *frames, long long hw, int base_global, int count, int n_total, int out_first, int out_count, float *out,
                   void *stream);
int dm_video_minmax(const float *x, long long n, float *lohi_out, void *workspace, size_t workspace_bytes, void *stream);
int dm_video_scale_f32(const float *x, long long n, const float *lohi, float *out, void *stream);
int dm_video_select_init(void *workspace, const long long ranks[4], void *stream);
int dm_video_select_hist(const float *x, long long n, int pass, void *workspace, void *stream);
int dm_video_select_pick(void *workspace, int pass, void *stream);
int dm_video_select_bounds(const void *workspace, double gamma_lo, double gamma_hi, double *ab_out, void *stream);
int dm_video_scale_f64(const float *x, long long n, const double *ab, double *out, void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * §8(b) — model-level entry points (csrc/model.cu): a handle that owns the packed checkpoint, the activation buffers, the
 * resolution-dependent tables and one captured CUDA graph per shape; a forward is ONE call.
 *   replaces  the network part of ModelHolder.load_models / get_raw_prediction (src/depthmap_generation.py:76-301,375-403)
 *             for model types 1, 2 (MiDaS 3.1 DPT-BEiT-L 512 / 384), 3 (MiDaS 3.0 DPT-Large 384) and 12, 13, 14 (Depth-Anything-V2 S / B / L).
 * dm_weight: one tensor of the upstream checkpoint (state_dict key, HOST pointer, dtype 0 = fp32 / 1 = fp16 / 2 = bf16, shape);
 * the blob is only read during dm_model_create.  dtype of the model: 0 = fp16 operands, fp32 accumulation (the only one).
 * dm_depth_forward: rgb uint8 [B,H,W,3] (device) -> depth_out fp32 [B,out_h,out_w] (device), asynchronous on `stream`; the net
 * size follows the reference's Resize rule for the family from (net_w, net_h) (dm_model_net_size).  The first call of a
 * shape allocates and runs eagerly, the second captures a CUDA graph, later calls replay it (DEPTHMAP_B200_MODEL_GRAPH=0
 * disables); inside an outer stream capture the launches are simply recorded into that capture.
 * Thread-compatible: one handle per thread; handles are independent.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct dm_weight {
    const char *name;
    const void *data_host;
    int32_t dtype;
    int32_t ndim;
    int64_t shape[4];
} dm_weight;
typedef struct dm_weight_blob {
    const dm_weight *items;
    int32_t count;
} dm_weight_blob;
typedef struct dm_model dm_model_t;
/* Resolution-dependent tables exactly as the model computes them (HOST pointers, float32 arithmetic in torch's order):
 * DINOv2 interpolate_pos_encoding (dinov2.py:179-210): pos_embed [1 + n*n, C] -> out [1 + gh*gw, C];
 * BEiT _get_rel_pos_bias table half (dmidas/backbones/beit.py:29-50): table [(2w-1)^2 + 3, heads] -> out [heads, (2gh-1)(2gw-1)+3] * log2(e). */
int dm_dinov2_pos_embed(const float *pos_embed_host, int n, int C, int gh, int gw, float *out_host);
int dm_beit_rel_table(const float *table_host, int window, int heads, int gh, int gw, float *out_host);
/* MiDaS 3.0 _resize_pos_embed (dmidas/backbones/vit.py:16-31): pos_embed [1 + n*n, C] -> out [1 + gh*gw, C], bilinear */
int dm_vit_pos_embed(const float *pos_embed_host, int n, int C, int gh, int gw, float *out_host);
int dm_model_create(dm_model_t **out, int model_type, const dm_weight_blob *weights, int device, int dtype);
int dm_model_destroy(dm_model_t *model);
int dm_model_net_size(const dm_model_t *model, int W, int H, int net_w, int net_h, int *nw_out, int *nh_out);
long long dm_model_launches(const dm_model_t *model);
int dm_depth_forward(dm_model_t *model, const uint8_t *rgb, int B, int H, int W, int net_w, int net_h, float *depth_out, int out_h, int out_w,
                     void *stream);

/* ---------------------------------------------------------------------------------------------------------------
 * D8 — LeReS (ResNeXt-101 32x8d + FTB / FFM / AO decoder), csrc/leres_kernels.cu: the non-GEMM pieces.   replaces parts of
 *   estimateleres / scale_torch (src/depthmap_generation.py:406-440), lib/Resnext_torch.py:196-220, lib/network_auxi.py:95-215.
 * ------------------------------------------------------------------------------------------------------------- */
/* uint8 RGB [B,H,W,3] -> /255 -> cv2.resize(bilinear) to net_h x net_w -> (x - mean) / std -> im2col of the 7x7 stride-2 pad-3
 * stem convolution: fp16 [B*Ho*Wo, 192], taps ordered (ky, kx, c), columns 147..191 zero */
int dm_leres_stem_im2col(const uint8_t *rgb, int B, int H, int W, int net_h, int net_w, const float *mean_host, const float *std_host, void *out,
                         void *stream);
int dm_maxpool3x3s2_nhwc_f16(const void *in, int B, int H, int W, int C, void *out, void *stream);   /* kernel 3, stride 2, padding 1 */
int dm_subsample2_nhwc_f16(const void *in, int B, int H, int W, int C, void *out, void *stream);     /* x[:, ::2, ::2, :] */
int dm_add_f16(const void *a, const void *b, void *out, long long n, void *stream);
/* dm_resize_f32 reading pixel (y, x) at in[(y * Win + x) * ld] (channel 0 of an [pixels, ld] fp32 GEMM output) */
int dm_resize_f32_ld(const float *in, int ld, int B, int Hin, int Win, float *out, int Hout, int Wout, int mode, void *stream);


/* ---------------------------------------------------------------------------------------------------------------
 * D9 — BOOST (csrc/boost_kernels.cu): the device side of estimateboost / doubleestimate
 * (src/depthmap_generation.py:774-941, :1028-1050) and of the pix2pix merge U-Net (pix2pix/models/networks.py:444-543,
 * pix2pix/models/pix2pix4depth_model.py:96-116).  The U-Net keeps fp32 NHWC activations; `split` != 0 makes the column
 * builders emit [hi | lo | hi] fp16 triples (3 K columns) for the split-operand GEMM (weights packed [hi | hi | lo]).
 * Reductions leave dm_boost_partials() partial results in device memory that the consuming kernel folds itself.
 * ------------------------------------------------------------------------------------------------------------- */
int dm_boost_partials(void);
int dm_unet_first_cols(const float *x /*[H,W,2]*/, int H, int W, void *out /*fp16 [H/2*W/2, 64 (*3)]*/, int split, void *stream);
int dm_unet_down_cols(const float *x /*[H,W,C]*/, int H, int W, int C, void *out /*fp16 [H/2*W/2, 16C (*3)]*/, int split, void *stream);
int dm_unet_up_cols(const float *skip, int C1, const float *up, int C2, int H, int W, void *out /*fp16 [4][H*W, 4(C1+C2) (*3)]*/, int split,
                    void *stream);
int dm_unet_interleave(const float *tmp /*[4][H*W,N]*/, int H, int W, int N, int C, float *out /*[2H,2W,C]*/, void *stream);
int dm_unet_final(const float *tmp /*[4][H*W,N]*/, int H, int W, int N, float bias, float *out /*[2H,2W]*/, void *stream);
/* the two single-/two-channel ends of the U-Net as direct fp32 kernels (no columns, no GEMM): outermost conv 2 -> 64 (w: [64][32], columns
 * (ky, kx, cin)) and outermost transposed conv (C1 + C2) -> 1 + bias + tanh (w: [4 parities][4 taps][C1 + C2]) */
int dm_unet_first(const float *x /*[H,W,2]*/, int H, int W, const float *w, float *out /*[H/2,W/2,64]*/, void *stream);
int dm_unet_last(const float *skip, int C1, const float *up, int C2, int H, int W, const float *w, float bias, float *out /*[2H,2W]*/, void *stream);
/* out[m, n] = gamma[n] * sum over chunks c (in order) of ws[c][m, n]: the depth chunks of a split-operand GEMM */
int dm_sum_chunks_f32(const float *ws, int nchunks, long long mn, int N, const float *gamma, float *out, void *stream);
int dm_boost_minmax(const float *x, long long n, float *partial /*[partials][2]*/, void *stream);
int dm_boost_merge_input(const float *outer, const float *inner, long long n, const float *p_outer, const float *p_inner, float *out /*[n,2]*/,
                         void *stream);
int dm_boost_post(const float *t, long long n, const float *partial, int normalise, float *out, void *stream);
int dm_boost_fit_sums(const float *x, const float *y, long long n, double *partial /*[partials][4]*/, void *stream);
int dm_boost_blend(const float *mapped /*[S,S]*/, int S, const double *fit_partial, const float *profile, int n_profile, float *updated, int pitch,
                   int x1, int y1, int w, int h, void *stream);
int dm_boost_resize_cubic(const float *in, int in_pitch, long long in_plane, int Hin, int Win, float *out, int out_pitch, long long out_plane,
                          int Hout, int Wout, int planes, void *stream);
int dm_boost_u8_to_planar(const uint8_t *rgb /*[H,W,3]*/, int H, int W, float *out /*[3,H,W] = rgb / 255*/, void *stream);
int dm_leres_stem_im2col_f32(const float *img /*[3,Hi,Wi]*/, int Hi, int Wi, int x0, int y0, int w, int h, int net_h, int net_w, const float *mean,
                             const float *std, void *out, void *stream);

/* B crops of one planar image in one launch (BOOST batches its patches); rects: DEVICE int32 [B][4] = x0, y0, w, h */
int dm_leres_stem_im2col_f32_batch(const float *img, int Hi, int Wi, const int *rects_dev, int B, int net_h, int net_w, const float *mean,
                                   const float *std, void *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DEPTHMAP_B200_H */
