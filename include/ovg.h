/* libovg -- C ABI of the B200-native OmniVGGT hot path (sm_100a).
 *
 * The reference has no FFI / plugin layer (SURVEY.md section 8b): its boundary is the Python nn.Module API of
 * omnivggt/models/omnivggt.py:10-68.  The drop-in module `omnivggt-official_b200.OmniVGGT` keeps that API and
 * binds the entry points below through ctypes (INTEGRATION.md).  Every entry point
 *   - takes plain device pointers / sizes (no torch types) and a CUDA stream handle (cudaStream_t as void*),
 *   - enqueues work asynchronously on that stream and returns 0, or a negative OVG_E_* code after recording a
 *     message retrievable with ovg_last_error(),
 *   - never allocates device memory on the hot path and never falls back to the CPU.
 * Each declaration cites the reference code (file:line under /root/reference) whose arithmetic it replaces.
 */
#ifndef OVG_H_
#define OVG_H_

#ifdef __cplusplus
extern "C" {
#endif

#define OVG_OK 0
#define OVG_E_INVALID (-1) /* bad argument (shape / alignment / null pointer) */
#define OVG_E_CUDA (-2)    /* CUDA runtime or driver error; see ovg_last_error() */
#define OVG_E_NODEVICE (-3)

/* Library / device ------------------------------------------------------------------------------------- */
int ovg_version(void);               /* ABI version, currently 2 */
const char* ovg_last_error(void);    /* thread-local message of the last failing call */
int ovg_device_check(void);          /* OVG_OK iff the current device is sm_100 (B200); OVG_E_NODEVICE otherwise */
long long ovg_launch_count(void);    /* kernels launched by this library since load (bench.py "gpu_launches") */

/* Fused tcgen05 GEMM ------------------------------------------------------------------------------------
 *   acc[m, n] = sum_{t < num_taps} sum_{c < a_cols} A[m + tap_off[t], c] * B[n, t * a_cols + c]
 * A: bf16 [a_rows, a_cols] row stride lda; B: bf16 [n, num_taps * a_cols] row stride ldb (nn.Linear / flattened
 * conv weight layout).  Rows of A outside [0, a_rows) read as zero, which makes a 3x3 conv over a zero-bordered
 * NHWC map nine row-shifted GEMMs.  Epilogues (epi):
 *   OVG_EPI_BF16     out bf16 = act(acc + bias + table[m % table_rows] + skip1 + skip2), row maps below
 *                    (nn.Linear+GELU layers/mlp.py:35-36; DPT convs heads/dpt_head.py:69-126,:379-399)
 *   OVG_EPI_RESID    out fp32 [row, n] += gamma[n] * (acc + bias[n]); row = row_index ? row_index[m] : m
 *                    (proj/fc2 + LayerScale + residual: layers/block.py:82-86,:105-106, layers/layer_scale.py:26-27;
 *                     depth-token scatter-add: omnivggt_aggregator.py:199-212)
 *   OVG_EPI_QKV      bias, q/k LayerNorm(64), 2-D RoPE, q pre-scale, head-major bf16 q/k/v
 *                    (layers/attention.py:52-58, layers/rope.py:154-188)
 *   OVG_EPI_HEADTAIL ReLU, 1x1 conv 32->outc, depth/point/confidence activations, fp32 NHWC outputs
 *                    (heads/dpt_head.py:121-126,:255-260, heads/head_act.py:61-125)
 */
enum { OVG_EPI_BF16 = 0, OVG_EPI_RESID = 1, OVG_EPI_QKV = 2, OVG_EPI_HEADTAIL = 3 };
enum {
  OVG_ROWS_IDENT = 0,     /* out row = m */
  OVG_ROWS_DENSE2PAD = 1, /* m = (f, y, x) on a gh x gw grid -> zero-bordered (gh+2) x (gw+2) grid */
  OVG_ROWS_PAD = 2,       /* m already enumerates the zero-bordered grid; border rows are written as zeros */
  OVG_ROWS_PIXSHUF = 3    /* transposed conv k = s = ps: n = (ky*ps + kx)*cout + co -> pixel (y*ps+ky, x*ps+kx) */
};
enum { OVG_ACT_NONE = 0, OVG_ACT_GELU_ERF = 1, OVG_ACT_RELU = 2 };

typedef struct ovg_gemm_args {
  const void* a; long long a_rows; int a_cols; long long lda;
  const void* b; int n; long long ldb;
  int m;
  int num_taps; int tap_off[9];
  int epi;
  /* common */
  const float* bias; int act; void* out; long long ldo;
  /* OVG_EPI_BF16 */
  const float* table; int table_rows;
  const void* skip1; const void* skip2;
  int rowmap; int gh; int gw; int ps; int cout;
  /* OVG_EPI_RESID */
  const float* gamma; const int* row_index;
  /* OVG_EPI_QKV */
  void* q_out; void* k_out; void* v_out;
  int C; int ntok; int T; int nspecial; int wp; int maxpos;
  const float* qn_w; const float* qn_b; const float* kn_w; const float* kn_b;
  const float* rope_cos; const float* rope_sin; float qscale;
  /* OVG_EPI_HEADTAIL */
  const float* w2; const float* b2; int outc; int head_act; float* preds; float* conf;
  /* tuning: 0 = auto, else 64/128/256, 512 = CTA-pair kernel (256 x 256 tile per 2-SM cluster) */
  int block_n;
  /* OVG_EPI_QKV switches: q/k LayerNorm(64) and 2-D RoPE (both 1 for aggregator blocks, 0 for DINOv2 blocks) */
  int qk_norm; int rope;
  /* OVG_EPI_QKV, context parallelism (n_peers > 0): the K / V rows of this rank's tokens go to every listed rank's full-length
   * buffer [batch*heads, peer_ntok, 64] at token offset peer_tok_off (peer-mapped device memory, plain stores over NVLink);
   * k_out / v_out are then unused.  The exchange of models/aggregator.py:312-341's single SDPA over all views is thereby
   * fused into the producing GEMM's epilogue. */
  void* k_peers[8]; void* v_peers[8]; int n_peers; int peer_ntok; long long peer_tok_off;
  /* OVG_EPI_BF16 / OVG_EPI_HEADTAIL: a, b, skip1, skip2 and the 16-bit output are IEEE half (fp16) instead of bf16 -- same tensor-core
   * rate, 3 more mantissa bits; stores saturate to +-65504.  Used by the DPT heads, which the reference keeps in fp32 even under
   * autocast (models/omnivggt.py:45). */
  int f16;
} ovg_gemm_args;

int ovg_gemm(const ovg_gemm_args* args, void* stream);

/* Fused attention: out[b, i, h*64:(h+1)*64] = softmax_j(q[b,h,i,:] . k[b,h,j,:]) v[b,h,j,:], q pre-scaled by
 * log2(e)/sqrt(64).  q,k,v: bf16 [batch, heads, n, 64]; out: bf16 [batch, n, heads*64].
 * Replaces F.scaled_dot_product_attention, layers/attention.py:61-66. */
int ovg_attention(const void* q, const void* k, const void* v, void* out, int batch, int heads, int n, void* stream);
/* Same with nq query rows and nkv keys / values per (batch, head): q [batch, heads, nq, 64], k, v [batch, heads, nkv, 64],
 * out [batch, nq, heads*64] (context parallelism: a rank's own queries against the keys / values of all ranks). */
int ovg_attention_kv(const void* q, const void* k, const void* v, void* out, int batch, int heads, int nq, int nkv,
                     void* stream);
/* Same with a scratch buffer of ovg_attention_scratch_bytes() bytes (16-byte aligned): for long sequences whose 128-row query tiles
 * do not fill the last wave of resident CTAs (two per SM), the tiles of that wave are cut into 2-4 key ranges, one CTA each, and
 * a small kernel merges their (un-normalised O, softmax reference, row sum) -- e.g. 1 376 tiles on 296 slots: 4.67 instead of 5
 * waves.  Results are deterministic (fixed merge order); scratch NULL = no split. */
long long ovg_attention_scratch_bytes(void);
int ovg_attention_kv_ws(const void* q, const void* k, const void* v, void* out, int batch, int heads, int nq, int nkv,
                        void* scratch, long long scratch_bytes, void* stream);

/* LayerNorm over the last dim, fp32 or bf16 in -> bf16 (out_is_f32 = 0), fp32 (1) or fp16 (2) out, optional affine, optional row gather
 * (out row m <- in row (m / grp_out) * grp_in + grp_off + m % grp_out; grp_out = 0: identity).
 * layers/block.py:50,:67 (eps 1e-5); heads/dpt_head.py:66,:219-227. */
int ovg_layernorm(const void* in, int in_is_bf16, long long ld_in, void* out, int out_is_f32, long long ld_out, int rows,
                  int C, const float* w, const float* b, float eps, int grp_out, int grp_in, int grp_off, void* stream);

/* Token assembly + modality scatter (omnivggt_aggregator.py:155-156,:202-213; aggregator.py:343-366). */
int ovg_assemble_tokens(float* x, const float* patch, const float* cam_tok, const float* reg_tok, const float* inj0,
                        const float* placeholder, const int* has_depth, int K, int S, int T, int R, int C, int view_base,
                        void* stream);   /* view_base: index of frame 0 within its scene (0 unless the views are sharded) */

/* Per-layer camera-token injection + bf16 snapshot of the residual stream into one half of the [K*T, 2C]
 * DPT input slot + fp32 camera-token copy (omnivggt_aggregator.py:273-303,:248-251; camera_head.py:96-99). */
int ovg_inject_snapshot(float* x, const float* inj, void* slot, float* cam_out, int K, int T, int C, int coff,
                        void* stream);

/* Depth modality: masked per-scene mean over the selected views, then [depth/(mean+1e-8)*mask, mask] im2col rows
 * (2*patch*patch wide, row stride ldc) for the patch-embedding GEMM (omnivggt_aggregator.py:107-128,:189-199;
 * layers/patch_embed.py:65-77).  scratch: OVG_DEPTH_SCRATCH_DOUBLES(B) doubles of device memory. */
#define OVG_DEPTH_SCRATCH_DOUBLES(B) ((B) * (2 * 1024 + 1))
/* Same with separate view lists: the normalisation mean is taken over the views idx_stats[0..n_stats) (ALL selected views of
 * the scene, omnivggt_aggregator.py:118-126), rows are produced for the views idx_cols[0..n_cols) only (the views this rank
 * owns when a scene is sharded over ranks; n_cols may be 0). */
int ovg_depth_im2col2(const float* depth, const float* mask, const int* idx_stats, int n_stats, const int* idx_cols, int n_cols,
                      double* scratch, void* cols, int ldc, int B, int S, int H, int W, int patch, void* stream);
int ovg_depth_im2col(const float* depth, const float* mask, const int* idx, double* scratch, void* cols, int ldc,
                     int B, int S, int Sd, int H, int W, int patch, void* stream);

/* RGB patch im2col for the DINOv2 patch embedding (layers/patch_embed.py:65-77, conv k = s = patch): images fp32
 * [K,3,H,W] in [0,1] are normalised with (x - mean[c]) / std[c] (models/omnivggt_aggregator.py:143) and written as bf16
 * rows (k, py, px) x cols (c, ky, kx), zero-padded to ldc columns.  mean3 / std3 are HOST arrays of 3 floats. */
int ovg_image_im2col(const float* images, const float* mean3, const float* std3, void* cols, int ldc, int K, int H, int W,
                     int patch, void* stream);

/* im2col for the stride-2 3x3 conv (heads/dpt_head.py:93-95): bf16 NHWC [F,h,w,C] -> [F*oh*ow, 9*C]. */
int ovg_im2col3x3s2(const void* src, void* dst, int F, int h, int w, int C, void* stream);

/* Bilinear align_corners=True upsampling between zero-bordered bf16 (f16 = 0) or fp16 (f16 = 1) NHWC maps
 * (heads/dpt_head.py:242-247,:466,:472-497) with the optional UV position embedding of heads/dpt_head.py:249-250 given in
 * separable form: tx fp32 [W, C/2] for channels [0, C/2), ty fp32 [H, C/2] for channels [C/2, C) (both NULL: no embedding). */
int ovg_upsample_bilinear(const void* src, void* dst, const float* tx, const float* ty, int F, int h, int w, int H, int W,
                          int C, int f16, void* stream);

/* Fused DPT output tail (heads/dpt_head.py:242-260, heads/head_act.py:61-125): bilinear resize (align_corners=True) of the
 * zero-bordered 16-bit NHWC map src [F, h+2, w+2, 128] to H x W, + UV position embedding (tx fp32 [W, 64], ty fp32 [H, 64], or both
 * NULL), 3x3 conv 128 -> 32 (w3x3: 16-bit [32, 9*128], K order (ky, kx, c); bias fp32 [32]), ReLU, 1x1 conv 32 -> outc (w2 fp32
 * [outc, 32], b2), activations (head_act 0: exp, 1: inverse-log; confidence 1 + exp) -> preds fp32 [F, H, W, outc-1], conf fp32
 * [F, H, W].  The H x W x 128 map is never materialised: the resized rows go straight into the tensor-core operand (rounded to 16
 * bits), and the position embedding enters through its own image under the 3x3 kernel, added in fp32 (the convolution is linear).
 * f16: src / w3x3 are fp16 (else bf16).  scratch: ovg_dpt_tail_scratch_bytes(H, W) bytes, 16-byte aligned (unused when tx is NULL).
 * ovg_dpt_tail_supported: 1 if the geometry fits the kernel (C == 128, upsampling, <= 80 source pixels under a 130-pixel strip). */
int ovg_dpt_tail_supported(int h, int w, int H, int W, int C);
long long ovg_dpt_tail_scratch_bytes(int H, int W);
int ovg_dpt_tail(const void* src, const float* tx, const float* ty, const void* w3x3, const float* bias, const float* w2,
                 const float* b2, int outc, int head_act, float* preds, float* conf, int F, int h, int w, int H, int W, int f16,
                 void* scratch, void* stream);

/* GPU input pipeline (SURVEY.md section 8f rank 4): the per-view work of visual_util.py:719-841 (load_images_and_cameras) on
 * decoded pixels.  The tap / index tables are small per-image-size arrays computed by the host with the libraries' own arithmetic
 * (Pillow Resample.c precompute_coeffs + normalize_coeffs_8bpc; OpenCV resizeNN).
 * ovg_preprocess_image: uint8 RGB [h, w, 3] -> Pillow-exact bicubic resize to [nh, nw] (two passes, uint8 rounding after each) ->
 * rows [crop, crop + fh) -> fp32 [3, fh, nw] = uint8 / 255 (ToTensor).  (hmin, hcnt, hk[nw, hksize]) / (vmin, vcnt, vk[nh, vksize]):
 * first source index, tap count and 22-bit fixed-point taps per output column / row; an axis that keeps its size passes NULLs.
 * tmp: uint8 [h, nw, 3] scratch (unused when w == nw).   visual_util.py:731-751 */
int ovg_preprocess_image(const unsigned char* src, int h, int w, int nw, int nh, int crop, int fh, const int* hmin, const int* hcnt,
                         const int* hk, int hksize, const int* vmin, const int* vcnt, const int* vk, int vksize,
                         unsigned char* tmp, float* out, void* stream);
/* ovg_preprocess_depth: validity filter (non-finite, > max_depth, < 1e-5 -> 0) + nearest-neighbour resize through the index tables
 * sy[nh], sx[nw] + crop -> depth fp32 [fh, nw], mask fp32 [fh, nw] (depth > 1e-5).  src element (r, c) at
 * src[r * row_stride + c * col_stride] (the reference transposes PNG depth maps: swap the strides).   visual_util.py:768-791 */
int ovg_preprocess_depth(const float* src, long long row_stride, long long col_stride, const int* sy, const int* sx, int crop,
                         int fh, int nw, float max_depth, float* depth, float* mask, void* stream);
/* ovg_prepare_cameras: camera-to-world [K,3,4] -> world-to-camera (closed-form SE3 inverse); intrinsics [K,3,3] rescaled by
 * geom[k] = (scale_x, scale_y, crop_y or < 0) ; views with has[k] == 0 get the reference's zero placeholders.  visual_util.py:807-824 */
int ovg_prepare_cameras(const float* c2w, const float* kin, const float* geom, const int* has, float* w2c, float* kout, int K,
                        void* stream);

/* On-device post-processing (SURVEY.md section 8f rank 3): what inference.py does on the host right after the forward.
 * ovg_pose_decode: pose_enc fp32 [K,9] = [t, quat xyzw, fov_h, fov_w] -> extrinsic [K,3,4] (world->camera, [R|t]),
 * intrinsic [K,3,3] (fx = (W/2)/tan(fov_w/2), fy = (H/2)/tan(fov_h/2), principal point at the image centre; may be NULL) and
 * cam2world [K,3,4] = closed-form SE3 inverse (may be NULL).
 * utils/pose_enc.py:65-130, utils/rotation.py:14-44, utils/geometry.py:269-318. */
int ovg_pose_decode(const float* pose_enc, float* extrinsic, float* intrinsic, float* cam2world, int K, int H, int W,
                    void* stream);

/* ovg_unproject_depth: world[k,v,u,:] = R_c2w ((u-cu) d/fu, (v-cv) d/fv, d) + t_c2w; depth fp32 [K,H,W], world fp32 [K,H,W,3].
 * utils/geometry.py:151-180 (unproject_depth_map_to_point_map), :183-264; visual_util.py:42-73. */
int ovg_unproject_depth(const float* depth, const float* intrinsic, const float* cam2world, float* world, int K, int H, int W,
                        void* stream);

/* ovg_conf_percentile_mask: threshold = numpy.percentile(conf, percent) (exact, linear interpolation),
 * mask[i] = conf[i] >= threshold && conf[i] > floor (inference.py:132-133: floor = 0.1).  workspace: device scratch of
 * OVG_PERCENTILE_WORKSPACE_BYTES; threshold_out: device float; count_out: device u64 (kept elements) or NULL. */
#define OVG_PERCENTILE_WORKSPACE_BYTES (6 * 8 + 512 * 4 + 4 * 4)
int ovg_conf_percentile_mask(const float* conf, long long n, float percent, float floor_, void* workspace,
                             unsigned char* mask, float* threshold_out, unsigned long long* count_out, void* stream);

/* ======================================================================================================================
 * Runtime: the launch SEQUENCES of the hot path behind handles, so that a host in any language runs the path with three
 * calls and raw device pointers (SURVEY.md section 8b).  Weight pointers refer to device memory in kernel layout (bf16
 * [N, K] matrices, fp32 vectors) owned by the caller and must stay valid for the life of the handle; descriptors are copied.
 * No entry point allocates device memory: the caller passes a 256-byte aligned workspace of ovg_*_workspace_bytes().
 * ====================================================================================================================== */
typedef struct ovg_block_weights {           /* one pre-LN transformer block, reference layers/block.py:27-107 */
  const float* ln1_w; const float* ln1_b;
  const void* w_qkv; const float* b_qkv;     /* bf16 [3C, C] */
  const float* qn_w; const float* qn_b; const float* kn_w; const float* kn_b;   /* q/k LayerNorm(64); all NULL for DINOv2 blocks */
  const void* w_proj; const float* b_proj; const float* g1;                     /* bf16 [C, C]; LayerScale gamma */
  const float* ln2_w; const float* ln2_b;
  const void* w_fc1; const float* b_fc1; const void* w_fc2; const float* b_fc2; const float* g2;
} ovg_block_weights;

/* Aggregator: token assembly, depth / camera modality injection, depth x (frame block, global block), kept intermediates.
 * reference models/omnivggt_aggregator.py:130-305, models/aggregator.py:312-341. */
typedef struct ovg_aggregator_desc {
  int C; int registers; int depth; int patch;
  const ovg_block_weights* frame_blocks;     /* host array [depth] */
  const ovg_block_weights* global_blocks;    /* host array [depth] */
  const float* cam_tok; const float* reg_tok; const float* placeholder;          /* [2,C], [2,registers,C], [C] */
  const void* depth_w; const float* depth_b;                                      /* bf16 [C, 2*patch*patch], fp32 [C] */
  const float* ones_c;                                                            /* fp32 [C] of ones */
  int keep_layers[4];                                                             /* layers whose outputs feed the DPT heads */
} ovg_aggregator_desc;
typedef struct ovg_aggregator ovg_aggregator;
int ovg_aggregator_create(const ovg_aggregator_desc* desc, ovg_aggregator** out);
void ovg_aggregator_destroy(ovg_aggregator* h);
long long ovg_aggregator_workspace_bytes(const ovg_aggregator* h, int B, int S, int H, int W, int n_depth);
/* Supported image sizes: H and W multiples of the patch size with at most OVG_MAX_PATCHES_PER_SIDE patches per side (2 044 px at
 * patch 14), and B*S*T token rows below 2^31.  The RoPE tables then need max(H, W) / patch + 1 <= OVG_ROPE_MAX_POSITIONS rows. */
#define OVG_MAX_PATCHES_PER_SIDE 146
#define OVG_ROPE_MAX_POSITIONS (OVG_MAX_PATCHES_PER_SIDE + 1)
/* patch_tokens fp32 [B*S, P, C]; inj fp32 [depth+1, B*S, C] (camera injection vectors, omnivggt_aggregator.py:172-179,:273-287);
 * depth / mask fp32 [B,S,H,W] and depth_idx device int[n_depth] (n_depth = 0: no depth aux); rope tables fp32 [maxpos, 16];
 * slots: host array of 4 device pointers, bf16 [B*S, T, 2C] each (frame half | global half); cam_out fp32 [B*S, 2C]. */
int ovg_aggregator_forward(ovg_aggregator* h, const float* patch_tokens, const float* inj, const float* depth, const float* mask,
                           const int* depth_idx, int n_depth, const float* rope_cos, const float* rope_sin, int maxpos, int B,
                           int S, int H, int W, void* workspace, long long workspace_bytes, void* const* slots, float* cam_out,
                           void* stream);

/* Frozen DINOv2 patchifier on the same kernels: reference layers/vision_transformer.py:214-271. */
typedef struct ovg_dino_desc {
  int C; int registers; int depth; int patch; int kpad;      /* kpad: 3*patch*patch rounded up to a multiple of 8 */
  const ovg_block_weights* blocks;                           /* host array [depth] */
  const void* w_patch; const float* b_patch;                 /* bf16 [C, kpad] (zero padded), fp32 [C] */
  const float* norm_w; const float* norm_b; const float* ones_c;
} ovg_dino_desc;
typedef struct ovg_dino ovg_dino;
int ovg_dino_create(const ovg_dino_desc* desc, ovg_dino** out);
void ovg_dino_destroy(ovg_dino* h);
long long ovg_dino_workspace_bytes(const ovg_dino* h, int K, int H, int W);
/* images fp32 [K,3,H,W] in [0,1]; base_tokens fp32 [1+registers+P, C] = [cls + pos0, registers, pos_patches];
 * mean3 / std3: HOST float[3]; patch_tokens_out fp32 [K, P, C] (x_norm_patchtokens). */
int ovg_dino_forward(ovg_dino* h, const float* images, const float* base_tokens, const float* mean3, const float* std3, int K,
                     int H, int W, void* workspace, long long workspace_bytes, float* patch_tokens_out, void* stream);

/* One DPT head (depth or point): reference heads/dpt_head.py:128-304, heads/head_act.py:61-125. */
typedef struct ovg_dpt_fusion {
  const void* rcu1[4];     /* resConfUnit1: conv1 w (bf16 [f, 9f]), conv1 b (fp32), conv2 w, conv2 b; all NULL for refinenet4 */
  const void* rcu2[4];     /* resConfUnit2 */
  const void* oc_w; const float* oc_b;   /* out_conv 1x1: bf16 [f, f], fp32 [f] */
} ovg_dpt_fusion;
typedef struct ovg_dpt_desc {
  int C2; int feat; int patch; int outc;                     /* 2*embed_dim, features (256), 14, 2 (depth) / 4 (points) */
  int oc[4];                                                  /* projection widths (256, 512, 1024, 1024) */
  const void* proj_w[4]; const float* proj_b[4];              /* 1x1 projections with the LayerNorm affine folded in */
  const void* up_w[2]; const float* up_b[2];                  /* ConvTranspose k4s4 / k2s2 as [(ky,kx,cout), cin] */
  const void* down_w; const float* down_b;                    /* Conv k3 s2 p1: bf16 [oc3, 9*oc3] */
  const void* rn_w[4];                                        /* layerN_rn 3x3, no bias: bf16 [feat, 9*oc] */
  ovg_dpt_fusion fus[4];                                      /* refinenet1..4 */
  const void* oc1_w; const float* oc1_b;                      /* output_conv1 3x3 feat -> feat/2 */
  const void* oc2_w; const float* oc2_b;                      /* output_conv2[0] 3x3 feat/2 -> 32 */
  const float* w2; const float* b2;                           /* output_conv2[2] 1x1 32 -> outc (fp32) */
  int f16;                                                    /* 1: every 16-bit weight above and every intermediate map is fp16
                                                                 (11-bit significand, saturating stores) instead of bf16 */
} ovg_dpt_desc;
typedef struct ovg_dpt ovg_dpt;
int ovg_dpt_create(const ovg_dpt_desc* desc, ovg_dpt** out);
void ovg_dpt_destroy(ovg_dpt* h);
long long ovg_dpt_workspace_bytes(const ovg_dpt* h, int Fc, int H, int W);
/* One chunk of Fc frames starting at frame f0.  slots: host array of 4 device pointers, bf16 [K, T, C2]; tables: host array of 4
 * device pointers, fp32 [P, oc[l]] UV position embeddings x0.1 (heads/dpt_head.py:262-272); tx fp32 [W, feat/4], ty fp32
 * [H, feat/4] separable embedding of the full-resolution stage; head_act 0: exp (depth), 1: inverse-log (points);
 * preds fp32 [K, H, W, outc-1], conf fp32 [K, H, W] (written for frames f0 .. f0+Fc-1). */
int ovg_dpt_forward(ovg_dpt* h, const void* const* slots, int T, int nspecial, int f0, int Fc, int H, int W,
                    const float* const* tables, const float* tx, const float* ty, int head_act, float* preds, float* conf,
                    void* workspace, long long workspace_bytes, void* stream);

/* Camera head: iterative pose refinement on the camera tokens; reference heads/camera_head.py:83-154.  The weight-streaming
 * GEMMs run on the tcgen05 GEMM; AdaLN, the S-token attention (head_dim D / heads) and the 9-wide pose update are small fp32
 * kernels. */
typedef struct ovg_camera_desc {
  int D; int heads; int trunk_depth;                           /* 2*embed_dim (2048), 16, 4 */
  const ovg_block_weights* trunk;                              /* host array [trunk_depth]; qn_w .. kn_b NULL */
  const float* token_norm_w; const float* token_norm_b; const float* trunk_norm_w; const float* trunk_norm_b;
  const float* empty_pose;                                     /* fp32 [9] */
  const float* embed_w; const float* embed_b;                  /* embed_pose: fp32 [D, 9], [D] */
  const void* mod_w; const float* mod_b;                       /* poseLN_modulation[1]: bf16 [3D, D], fp32 [3D] */
  const void* fc1_w; const float* fc1_b;                       /* pose_branch.fc1: bf16 [D/2, D], fp32 [D/2] */
  const float* fc2_w; const float* fc2_b;                      /* pose_branch.fc2: fp32 [9, D/2], [9] */
} ovg_camera_desc;
typedef struct ovg_camera ovg_camera;
int ovg_camera_create(const ovg_camera_desc* desc, ovg_camera** out);
void ovg_camera_destroy(ovg_camera* h);
long long ovg_camera_workspace_bytes(const ovg_camera* h, int K);
/* cam_tokens fp32 [B*S, D]; out fp32 [iters, B*S, 9]: the activated pose encoding after each iteration. */
int ovg_camera_forward(ovg_camera* h, const float* cam_tokens, int B, int S, int iters, float* out, void* workspace,
                       long long workspace_bytes, void* stream);

/* Cross-GPU barrier on peer-mapped flags (no NCCL, no host): the rank bumps its private device counter `epoch_counter`,
 * writes the new value into slot `rank` of every peer's flag array (int[world], peer-mapped, zero-initialised) and waits until
 * all slots of its own array have reached it.  Orders the peer stores of the kernels launched before it on this stream against
 * the peers' reads launched after their barrier.  All ranks must execute the same sequence of barriers. */
int ovg_peer_barrier(int* const* flag_peers, int* epoch_counter, int rank, int world, void* stream);

/* Context-parallel aggregator (SURVEY.md section 8f rank 2): ONE scene whose views are sharded over `world` GPUs of a node.
 * Every rank runs the per-token work (LayerNorm, QKV / proj / MLP GEMMs, frame attention) on its own S views; in the global
 * blocks (models/aggregator.py:312-341: one SDPA over all views) the QKV epilogue stores the K / V rows of the rank's tokens
 * straight into every rank's full-length K / V buffer over NVLink (ovg_gemm_args.k_peers), a flag barrier follows, and the
 * rank's own queries attend to all keys (ovg_attention_kv).  No collective library call on the data path; K / V buffers are
 * double buffered so that one barrier per global block suffices. */
typedef struct ovg_context_parallel {
  int rank; int world;
  int views_total;                    /* views of the whole scene; this rank holds views [rank*S, rank*S + S), S = views_total / world */
  void* k_peers[2][8];                /* [buffer][rank]: bf16 [heads, views_total*T, 64] in rank's memory, peer mapped */
  void* v_peers[2][8];
  int* flag_peers[8];                 /* [rank]: int[world], peer mapped, zero-initialised once */
  int* epoch_counter;                 /* private device int, zero-initialised once */
  float* cam_peers[8];                /* [rank]: fp32 [views_total, 2C] camera tokens of ALL views (the camera head attends across
                                         views, heads/camera_head.py:104-154); every rank stores its rows into every peer */
} ovg_context_parallel;
/* As ovg_aggregator_forward with B = 1 and S = the LOCAL view count, except for the depth modality, whose normalisation is
 * global over the scene: depth / mask are the FULL tensors [1, views_total, H, W], depth_idx lists ALL selected views (scene
 * indices, n_depth of them) and depth_idx_local the selected views this rank owns (scene indices, n_depth_local of them). */
int ovg_aggregator_forward_cp(ovg_aggregator* h, const ovg_context_parallel* cp, const float* patch_tokens, const float* inj,
                              const float* depth, const float* mask, const int* depth_idx, int n_depth,
                              const int* depth_idx_local, int n_depth_local, const float* rope_cos, const float* rope_sin,
                              int maxpos, int S, int H, int W, void* workspace, long long workspace_bytes, void* const* slots,
                              float* cam_out, void* stream);   /* cam_out: this rank's rows [S, 2C]; all views: cp->cam_peers[rank] */

/* Timing hook for bench.py: when enabled, every global-attention launch of ovg_aggregator_forward is bracketed by CUDA events
 * on its stream; after a synchronize, ovg_runtime_attention_times() returns the elapsed ms of the launches since the enable. */
void ovg_runtime_time_attention(int enable);
/* Process-wide switch (default on): the block runtimes hand ovg_attention_kv_ws their scratch, so long sequences may split the
 * tiles of the last CTA wave over the keys.  Off: every tile is computed by one CTA -- the summation order of a tile then does not
 * depend on how many tiles the launch has, which is what makes a context-parallel forward BIT-identical to the single-GPU one
 * (tests/test_cp_gpu.py checks that with the switch off, and agreement within 5e-3 of the dense outputs with it on). */
void ovg_runtime_attention_split(int enable);
int ovg_runtime_attention_times(float* ms, int max_n);

#ifdef __cplusplus
}
#endif
#endif /* OVG_H_ */
