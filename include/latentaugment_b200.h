/* latentaugment_b200 -- C ABI of the B200-native LatentAugment hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every pointer
 * named `d_*` is a DEVICE pointer to fp32 data owned by the caller (the Python host keeps
 * them in torch tensors); the library allocates nothing on the device except what it carves
 * out of the caller-provided workspace (and one transient scratch in la_set_latent_bank).
 * All calls are asynchronous on the given stream unless stated; return value 0 = success,
 * otherwise an error code whose text is la_last_error().
 *
 * Reference interfaces replaced (paths relative to the reference repository root):
 *   la_engine_create      <- LatentAug.__init__/load_stylegan   augments/utils/util_latent_aug.py:70-121,466-484
 *                            (+ the parameter contract models/stylegan3/legacy.py:122-203)
 *   la_set_latent_bank    <- register_buffer('W') from compute_stats('latent')   util_latent_aug.py:140-148,503-563
 *   la_set_image_bank     <- register_buffer('X') from compute_stats('img')      util_latent_aug.py:150-158
 *   la_mapping            <- G.mapping(z, None, truncation_psi) in z_to_w / forward_ganrand   util_latent_aug.py:202-205,459-464
 *   la_synthesis          <- G.synthesis(ws, noise_mode=...) / synthetize         util_latent_aug.py:227,486-489
 *                            (ops: torch_utils/ops/{conv2d_resample,upfirdn2d,bias_act,fma}.py)
 *   la_augment            <- LatentAug.forward: the N-step Adam loop, criteria, gate, final synthesis
 *                                                                                util_latent_aug.py:207-310
 *   la_set_discriminator  <- self.D (the unpickled StyleGAN2 discriminator, parameter contract legacy.py:220-289) and the
 *                            realism term calc_loss_disc: softplus(-D(x, c=None)).mean() * w_disc   util_latent_aug.py:363-371
 *   la_pairwise_sqdist    <- l2_loss_vectorized(X, Y, compute_mean=False)         util_latent_aug.py:315-361
 *   la_nearest_codes      <- (north_star extension, SURVEY.md F3) argmin / top-k of that matrix
 *   la_project            <- StyleGAN2-ADA projector.py::project, batched, producing the inverted codes of --init_w inv
 *                            (DESIGN.md "Projection")
 *   la_detector_features  <- the VGG16 fc7 embedding StyleGAN3's precision / recall feeds to compute_pr (pinned to
 *                            torchvision's vgg16; DESIGN.md §13)
 */
#ifndef LATENTAUGMENT_B200_H
#define LATENTAUGMENT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LA_MAX_BLOCKS 12          /* resolutions 4 .. 8192 */
#define LA_MAX_CONV (2 * LA_MAX_BLOCKS)
#define LA_MAX_MAPPING 8
#define LA_MAX_STEPS 64            /* steps whose loss values are logged (the loop itself is not capped) */
#define LA_LOSS_COLS 5             /* loss-log row: latent, pixel, total, discriminator, perceptual */
#define LA_ABI_VERSION 203

typedef struct la_engine la_engine;
typedef struct la_detector la_detector;
typedef void* la_stream;          /* cudaStream_t */

enum la_precision {
    LA_PRECISION_BF16 = 0,        /* one bf16 tensor-core pass, fp32 accumulate (tolerance: rel-L2 1e-2) */
    LA_PRECISION_FP32_PARITY = 1  /* split-bf16 (hi/lo) operands, 3 passes, fp32 accumulate (rel-L2 1e-3) */
};

enum la_noise_mode { LA_NOISE_NONE = 0, LA_NOISE_CONST = 1, LA_NOISE_RANDOM = 2 };

/* One 3x3 modulated-conv layer: names per legacy.py:178-195. */
typedef struct la_conv_params {
    const float* d_weight;         /* [cout, cin, 3, 3] */
    const float* d_bias;           /* [cout] */
    const float* d_noise_const;    /* [res, res] */
    float noise_strength;
    const float* d_affine_weight;  /* [cin, w_dim] */
    const float* d_affine_bias;    /* [cin] */
} la_conv_params;

/* One toRGB layer: legacy.py:196-199. */
typedef struct la_torgb_params {
    const float* d_weight;         /* [img_channels, cin, 1, 1] */
    const float* d_bias;           /* [img_channels] */
    const float* d_affine_weight;  /* [cin, w_dim] */
    const float* d_affine_bias;    /* [cin] */
} la_torgb_params;

/* StyleGAN2 generator (skip architecture) description; constructor kwargs per legacy.py:122-144. */
typedef struct la_generator_desc {
    int img_resolution;            /* power of two >= 8 */
    int img_channels;              /* 1..3 */
    int w_dim, z_dim;
    int num_blocks;                /* log2(res) - 1 */
    int channels[LA_MAX_BLOCKS];   /* feature maps of block 4, 8, ... (multiples of 64) */
    float conv_clamp;              /* < 0: no clamp */
    const float* d_const;          /* synthesis.b4.const [channels[0], 4, 4] */
    const float* d_resample_filter;/* [4, 4] (setup_filter([1,3,3,1])) */
    la_conv_params conv[LA_MAX_CONV];     /* b4.conv1, b8.conv0, b8.conv1, b16.conv0, ... (2*num_blocks - 1) */
    la_torgb_params torgb[LA_MAX_BLOCKS]; /* b4.torgb, b8.torgb, ... */
    int mapping_layers;            /* 0: no mapping network given */
    float mapping_lr_multiplier;
    const float* d_mapping_weight[LA_MAX_MAPPING];   /* fc{i}.weight [out, in] */
    const float* d_mapping_bias[LA_MAX_MAPPING];
    const float* d_w_avg;          /* [w_dim] */
} la_generator_desc;

/* Options of one augmentation call: the opt.* fields LatentAug.forward reads
 * (augments/latent_aug.py:45-98, util_latent_aug.py:84-112). */
typedef struct la_augment_options {
    int num_steps;                 /* opt_num_epochs */
    float lr;                      /* opt_lr */
    float w_latent, w_pix;         /* criteria weights */
    int soft_aug;                  /* 0: hard_aug, 1: smooth_aug */
    float alpha;
    int final_noise_mode;          /* la_noise_mode of the last synthesis (reference default: random) */
    int n_modalities;              /* number of leading image channels the pixel criterion covers */
    float w_disc;                  /* weight of the discriminator realism term; > 0 needs la_set_discriminator */
    float w_lpips;                 /* weight of the perceptual term; > 0 needs la_set_lpips + la_set_feature_bank */
    int lpips_crop_x, lpips_crop_y;/* origin of this call's crop window, absolute image coordinates (util_dataset.py:284-296: one draw per forward) */
    int lpips_norm_mode;           /* 0: lpips_script form (pair mean), 1: forward_tr form (pair sum / bank size) */
} la_augment_options;

/* One residual block of the StyleGAN2 'resnet' discriminator at resolution res (names per legacy.py:267-287). */
typedef struct la_disc_block_params {
    const float* d_fromrgb_weight; /* [ch, img_channels, 1, 1]  (top block only, else null) */
    const float* d_fromrgb_bias;   /* [ch] */
    const float* d_conv0_weight;   /* [ch, ch, 3, 3] */
    const float* d_conv0_bias;     /* [ch] */
    const float* d_conv1_weight;   /* [ch_next, ch, 3, 3]   (down 2) */
    const float* d_conv1_bias;     /* [ch_next] */
    const float* d_skip_weight;    /* [ch_next, ch, 1, 1]   (down 2, no bias) */
} la_disc_block_params;

/* StyleGAN2 discriminator description (c_dim = 0, architecture 'resnet', mbstd_num_channels = 1). */
typedef struct la_disc_desc {
    int img_resolution, img_channels;
    int num_blocks;                /* log2(res) - 2 residual blocks: res, res/2, ..., 8 */
    int channels[LA_MAX_BLOCKS];   /* feature maps at res, res/2, ..., 8, 4  (num_blocks + 1 entries, multiples of 64) */
    float conv_clamp;              /* < 0: no clamp */
    int mbstd_group_size;          /* 4 upstream */
    const float* d_resample_filter;/* [4, 4] (setup_filter([1,3,3,1])) */
    la_disc_block_params block[LA_MAX_BLOCKS];
    const float* d_b4_conv_weight; /* [ch4, ch4 + 1, 3, 3] */
    const float* d_b4_conv_bias;   /* [ch4] */
    const float* d_b4_fc_weight;   /* [ch4, ch4 * 16] */
    const float* d_b4_fc_bias;     /* [ch4] */
    const float* d_b4_out_weight;  /* [1, ch4] */
    const float* d_b4_out_bias;    /* [1] */
} la_disc_desc;

/* VGG16 feature extractor + LPIPS linear layers of the perceptual term (reference augments/criteria/lpips/networks.py:87-97,
 * 22-32; torchvision vgg16.features parameter order).  Taps are the ReLU outputs relu1_2, relu2_2, relu3_3, relu4_3, relu5_3
 * (1-based layer indices 4, 9, 16, 23, 30 of BaseNet.forward, networks.py:52-64); a tap is used iff its lin weight is given.
 * The in-tree LPIPS uses taps 16/23/30 (networks.py:94), the NVIDIA TorchScript model of the lpips_script path all five. */
#define LA_VGG_CONVS 13
#define LA_VGG_TAPS 5
typedef struct la_vgg_desc {
    const float* d_conv_weight[LA_VGG_CONVS];  /* [cout, cin, 3, 3]: 3-64-64 | 128-128 | 256-256-256 | 512-512-512 | 512-512-512 */
    const float* d_conv_bias[LA_VGG_CONVS];    /* [cout] */
    const float* d_lin_weight[LA_VGG_TAPS];    /* [C_tap] (the 1x1 conv C -> 1 without bias), or null = tap not used */
    float mean[3], std[3];                     /* z-score of the replicated grey crop (networks.py:41-50) */
    int crop_size;                             /* crop_size_aug: 64 (power of two >= 64) */
    int per_sample_targets;                    /* 1: also plan fp32 per-sample target features for la_set_projection_targets
                                                  (crop_size must be min(res, 256), res <= 512); 0: bank mode only */
} la_vgg_desc;

/* VGG16 detector of precision / recall (DESIGN.md §13): torchvision vgg16 `features` (same parameters as la_vgg_desc), the
 * NCHW flatten, classifier.0 (fc6) + ReLU and classifier.3 (fc7) + ReLU. */
typedef struct la_detector_desc {
    const float* d_conv_weight[LA_VGG_CONVS];  /* [cout, cin, 3, 3] */
    const float* d_conv_bias[LA_VGG_CONVS];    /* [cout] */
    const float* d_fc6_weight;                 /* [4096, 25088] (input index c * 49 + h * 7 + w) */
    const float* d_fc6_bias;                   /* [4096] */
    const float* d_fc7_weight;                 /* [4096, 4096] */
    const float* d_fc7_bias;                   /* [4096] */
    float mean[3], std[3];                     /* per-channel normalisation of the 0..255 input: (v - mean) / std */
} la_detector_desc;

const char* la_last_error(void);
/* ABI version (LA_ABI_VERSION) and sizeof of the structs passed by pointer, in the order la_generator_desc,
 * la_augment_options, la_disc_desc, la_conv_params, la_torgb_params, la_disc_block_params, la_vgg_desc, la_detector_desc
 * (returns how many were written, at most `max`): a binding checks both before the first call. */
int la_version(void);
int la_struct_sizes(size_t* out, int max);

/* Discriminator of the realism term; it runs in the engine's precision (`precision` below must equal the engine's).
 * The workspace is caller-owned like the engine's.  la_disc_logits / la_disc_loss_grad are the stand-alone forms
 * of what la_augment does every step when w_disc > 0 (tests, criteria plugin). */
int la_disc_workspace_bytes(const la_disc_desc* d, int batch, int precision, size_t* bytes);
int la_set_discriminator(la_engine* e, const la_disc_desc* d, void* d_workspace, size_t workspace_bytes, la_stream stream);
/* d_img [batch, img_channels, res, res] fp32 -> d_logits [batch] */
int la_disc_logits(la_engine* e, const float* d_img, float* d_logits, la_stream stream);
/* loss = w_disc * mean softplus(-D(img)) -> d_loss [1];  d loss / d img -> d_grad [batch, img_channels, res, res] */
int la_disc_loss_grad(la_engine* e, const float* d_img, float w_disc, float* d_loss, float* d_grad, la_stream stream);

/* Perceptual term (reference calc_loss_lpips_torchscript / calc_loss_lpips_tr, util_latent_aug.py:387-424, + LPIPS.forward,
 * criteria/lpips/lpips.py:44-56).  la_set_lpips installs the network (caller-owned workspace, engine precision);
 * la_set_feature_bank takes the real crops [M, img_channels, crop, crop] fp32 in [-1, 1] (the reference builds its feature
 * bank from one random window per real image, util_latent_aug.py:564-579) and keeps only the bank moments;
 * la_lpips_loss_grad is the stand-alone form of what la_augment does every step when w_lpips > 0:
 * crop window with origin (crop_x, crop_y) in absolute image coordinates (the reference draws the position inside the
 * centre crop, util_dataset.py:284-309: add the centre-crop offset), loss [1] = w_lpips * mean over modalities of the normalised pair
 * distance (norm_mode 0: / (n * m), 1: / m), grad [batch, C, res, res] = d loss / d img. */
int la_lpips_workspace_bytes(const la_vgg_desc* v, int batch, int img_channels, int precision, size_t* bytes);
int la_set_lpips(la_engine* e, const la_vgg_desc* v, void* d_workspace, size_t workspace_bytes, la_stream stream);
int la_set_feature_bank(la_engine* e, const float* d_crops, int M, la_stream stream);
int la_lpips_loss_grad(la_engine* e, const float* d_img, int crop_x, int crop_y, float w_lpips, int norm_mode, float* d_loss,
                       float* d_grad, la_stream stream);
/* norm_mode 2 (needs la_set_projection_targets): the projection's distance of every sample to its OWN target over the whole
 * image (crop_x = crop_y = 0; area-pooled 2x2 when res = 2 * crop_size), d_loss [batch] per sample (w_lpips is ignored),
 * d_grad = d (sum of d_loss) / d img. */
/* Test hook: normalised activations of used tap k (0-based among the used taps) from the last la_lpips_loss_grad /
 * la_augment step: fp32 [batch * img_channels, h, w, C] (NHWC); *count receives the element count (d_out may be null). */
int la_lpips_tap(la_engine* e, int k, float* d_out, size_t* count, la_stream stream);

/* filtered_lrelu (reference torch_utils/ops/filtered_lrelu.py:56-153; the StyleGAN3 synthesis-layer op, SURVEY.md row a23):
 * y = decimate_down( FIR_fd( clamp( lrelu( FIR_fu( pad( zero_insert_up( x + b ) ) ) * up^2 ) * gain ) ) ).
 * d_x [N, C, H, W] fp32 -> d_y [N, C, out_h, out_w] with mid = H*up + py0 + py1 - (fu_taps - 1),
 * out_h = ceil((mid - (fd_taps - 1)) / down).  h_fu / h_fd are HOST arrays of separable taps (null = identity).
 * d_mask_out (int8 [N*C, mid_h, mid_w], or null) receives the activation-derivative class per intermediate pixel
 * (0 clamped, 1 positive, 2 negative); with d_mask_in the activation is replaced by gain * that derivative -- the
 * backward pass is this same call with the filters' roles swapped (latentaugment_b200/ops_sg3.py).  mask_o / mask_h /
 * mask_w place the mask tensor inside the intermediate (0 sizes = it covers the intermediate exactly). */
int la_filtered_lrelu(const float* d_x, int N, int C, int H, int W, const float* h_fu, int fu_taps, const float* h_fd, int fd_taps,
                      const float* d_b, int up, int down, int px0, int px1, int py0, int py1, float gain, float slope, float clamp,
                      int flip_filter, const signed char* d_mask_in, signed char* d_mask_out, int mask_oy, int mask_ox, int mask_h,
                      int mask_w, float* d_y, la_stream stream);

/* Bytes of device workspace an engine of this shape needs. */
int la_engine_workspace_bytes(const la_generator_desc* g, int batch, int precision, size_t* bytes);

/* Builds an engine over caller-owned workspace.  Weight preparation kernels are enqueued on
 * `stream`; the generator parameter tensors must stay alive for the engine's lifetime (biases,
 * noise constants are read in place). */
int la_engine_create(const la_generator_desc* g, int batch, int precision, void* d_workspace, size_t workspace_bytes,
                     la_stream stream, la_engine** out);
void la_engine_destroy(la_engine* e);

/* Real-code bank W [M, num_ws, w_dim] and real-image bank X [M, C, res, res] in [-1, 1].
 * Only their moments are kept (SURVEY.md App. B); the tensors are not referenced afterwards. */
int la_set_latent_bank(la_engine* e, const float* d_W, int M, la_stream stream);
int la_set_image_bank(la_engine* e, const float* d_X, int M, la_stream stream);

/* w[n, :] = mapping(z[n, :]) with truncation; n <= engine batch.  One row per sample (the
 * reference broadcasts it to num_ws rows). */
int la_mapping(la_engine* e, const float* d_z, int n, float truncation_psi, float* d_w, la_stream stream);

/* img [batch, C, res, res] (NCHW fp32) = G.synthesis(ws).  ws element (n, i, k) is read at
 * d_ws[n*stride_n + i*stride_i + k] (stride_i = 0 broadcasts one row per sample).
 * noise: LA_NOISE_CONST uses the layers' noise_const; LA_NOISE_RANDOM reads unit normal noise
 * from d_noise, laid out layer after layer as [batch, res_l, res_l] (conv order of la_generator_desc). */
int la_synthesis(la_engine* e, const float* d_ws, long long stride_n, long long stride_i, int noise_mode,
                 const float* d_noise, float* d_img, la_stream stream);
size_t la_noise_floats(const la_engine* e);

/* The hot path.  d_w0 [batch, w_dim] initial codes; outputs: d_img [batch, C, res, res],
 * d_w_aug [batch, w_dim] (one row per sample), d_loss_log [min(num_steps, LA_MAX_STEPS), LA_LOSS_COLS] =
 * (latent, pixel, total, discriminator, perceptual) or NULL.  d_final_noise as in la_synthesis (may be NULL unless final_noise_mode == RANDOM). */
int la_augment(la_engine* e, const float* d_w0, const la_augment_options* opt, const float* d_final_noise, float* d_img,
               float* d_w_aug, float* d_loss_log, la_stream stream);

/* Projection of real images into W (StyleGAN2-ADA projector.py::project, batched; DESIGN.md "Projection").
 * la_set_projection_targets: d_img [batch, C, res, res] fp32 in [-1, 1]; needs la_set_lpips with per_sample_targets = 1.
 * la_project: num_steps Adam steps (betas 0.9 / 0.999, eps 1e-8) from d_w0 [batch, w_dim]; step t synthesises (const noise)
 * from w_opt + d_sigma[t] * d_wnoise[t] (d_wnoise [num_steps, batch, w_dim] unit normal, or NULL for none), takes the
 * summed per-sample LPIPS distance to the targets over all used taps, and steps with learning rate d_lr[t].
 * d_lr, d_sigma: DEVICE arrays [num_steps].  Outputs: d_w_out [batch, w_dim] = w_opt after the last step (no noise);
 * d_loss_log [num_steps] (or NULL) = the summed loss of every step.  All device arrays must stay alive until the call
 * has completed on the stream. */
int la_set_projection_targets(la_engine* e, const float* d_img, la_stream stream);
int la_project(la_engine* e, const float* d_w0, int num_steps, const float* d_lr, const float* d_sigma, const float* d_wnoise,
               float* d_w_out, float* d_loss_log, la_stream stream);

/* D[j, i] = |Y_j|^2 + |X_i|^2 - 2 <Y_j, X_i>  ([bank, batch] orientation, fp32, the reference's
 * association order).  X [n, K], Y [m, K]. */
int la_pairwise_sqdist(const float* d_X, int n, const float* d_Y, int m, int K, float* d_D, la_stream stream);

/* k nearest bank rows per query under that distance, ties to the lowest index.  Candidates are
 * selected by ONE bf16 tensor-core GEMM pass with a fused per-tile top-k and re-ranked exactly (fp64 dot, one
 * rounding, the reference's association order); the re-rank margin bounds the bf16 error and tiles whose candidate
 * list may be incomplete are rescanned, so the result equals the exhaustive search for any data.
 * la_bank_prepare fills d_bank_bf16 [m, K] bf16 and d_bank_sqnorm [m + 1] fp32 (the squared norms followed by their
 * maximum).  index_offset is added to the returned indices (bank shards).  Outputs: d_dist [n, k] fp32, d_idx [n, k] int64. */
int la_bank_prepare(const float* d_Y, int m, int K, void* d_bank_bf16, float* d_bank_sqnorm, la_stream stream);
int la_nearest_codes(const float* d_X, int n, const float* d_Y, const void* d_bank_bf16, const float* d_bank_sqnorm, int m, int K,
                     int k, long long index_offset, void* d_workspace, size_t workspace_bytes, float* d_dist, long long* d_idx,
                     la_stream stream);
int la_nearest_codes_workspace_bytes(int n, int m, int K, int k, size_t* bytes);
/* Merges per-shard (dist, idx) lists [shards, n, k] into the global k best. */
int la_merge_topk(const float* d_dist, const long long* d_idx, int shards, int n, int k, float* d_out_dist, long long* d_out_idx,
                  la_stream stream);
/* Same, shard s read at d_dist + s * dist_shard_stride (floats) / d_idx + s * idx_shard_stride (int64s): lets one
 * all-gather of a packed per-rank record (dist block, idx block) feed the merge without unpacking. */
int la_merge_topk_strided(const float* d_dist, const long long* d_idx, int shards, int n, int k, long long dist_shard_stride,
                          long long idx_shard_stride, float* d_out_dist, long long* d_out_idx, la_stream stream);

/* Precision / recall of feature sets (StyleGAN3 compute_pr; DESIGN.md §12).  The manifold Y [m, K] and the queries hold
 * fp16-valued fp32 features; d2 is the distance above.  la_pr_manifold_prepare fills d_planes [2, m, K] bf16 (hi | lo: an fp16
 * value is exactly hi + lo) and d_sqnorm [m + 1] (squared norms followed by their maximum).  Candidates are scored by three
 * bf16 tensor-core passes over the planes, (hi,hi) + (lo,hi) + (hi,lo); exact rechecks make both results exact for any data.
 *   la_pr_radii:  d_r2[i] = the (nhood + 1)-th smallest d2(X_i, Y_j) over all j (a point of the manifold counts itself and
 *                 duplicates count).  X [n, K] are the rows whose radii are wanted (normally rows of Y).  1 <= nhood <= 7,
 *                 m >= nhood + 1.
 *   la_pr_member: d_member[i] = 1 when, for some j, h(d2(X_i, Y_j)) <= h(d_r2[j]) with h(v) = fp16(sqrt(max(v, 0)))
 *                 (round to nearest even, saturating to +inf), else 0.  X [n, K] are the probes.
 * Each adds to *d_fallback (device int, the caller zeroes it; NULL = not counted) the number of queries that were scanned
 * exhaustively because their candidate list overflowed.  K must be a multiple of 64; workspaces 1024-byte aligned. */
int la_pr_manifold_prepare(const float* d_Y, int m, int K, void* d_planes, float* d_sqnorm, la_stream stream);
int la_pr_radii_workspace_bytes(int n, int m, int K, int nhood, size_t* bytes);
int la_pr_radii(const float* d_X, int n, const float* d_Y, const void* d_planes, const float* d_sqnorm, int m, int K, int nhood,
                void* d_workspace, size_t workspace_bytes, float* d_r2, int* d_fallback, la_stream stream);
int la_pr_member_workspace_bytes(int n, int m, int K, size_t* bytes);
int la_pr_member(const float* d_X, int n, const float* d_Y, const void* d_planes, const float* d_sqnorm, const float* d_r2, int m, int K,
                 void* d_workspace, size_t workspace_bytes, unsigned char* d_member, int* d_fallback, la_stream stream);

/* VGG16 detector embeddings (DESIGN.md §13).  A detector is independent of any engine: it owns a caller-provided workspace
 * (1024-byte aligned) planned for at most `batch` images per call in `precision`; creation prepares the weights on `stream`
 * (the weight tensors are not referenced afterwards; the bias tensors are read in place and must stay alive).
 * la_detector_features: d_img [n, C, res, res] fp32 in [-1, 1], 1 <= n <= batch, 16 <= res <= 1024; per image, channel
 * `modality` is quantised to 0..255 as StyleGAN3 saves images (clamp(x * 127.5 + 128, 0, 255) truncated), replicated to three
 * channels, area-resized to 224^2, normalised, and embedded -> d_out [n, 4096] fp32 (the ReLU of fc7). */
int la_detector_workspace_bytes(const la_detector_desc* d, int batch, int precision, size_t* bytes);
int la_detector_create(const la_detector_desc* d, int batch, int precision, void* d_workspace, size_t workspace_bytes, la_stream stream,
                       la_detector** out);
void la_detector_destroy(la_detector* det);
int la_detector_features(la_detector* det, const float* d_img, int n, int C, int res, int modality, float* d_out, la_stream stream);

/* Test hooks: run every tap-GEMM of the engine once through the SIMT twin as well and report
 * the largest deviation (debug cross-check of the tensor-core path; not a product path). */
int la_debug_set_simt(la_engine* e, int use_simt);
int la_debug_check(la_engine* e, la_stream stream);
/* Times each tap-GEMM launch of one optimisation step alone (CUDA events, `reps` launches each).
 * h_ms: HOST array [4*L + 1] = forward GEMM[0..L), data-gradient GEMM[0..L), FIR pass forward[0..L),
 * FIR pass backward[0..L) (0 where the layer has none), backward seed.  Synchronous. */
int la_debug_time_gemms(la_engine* e, int reps, float* h_ms, int* n_layers);   /* synchronises; non-zero if a pipeline wait timed out */
long long la_debug_launch_count(const la_engine* e);
/* Copies an internal quantity of the LAST optimisation step to d_out (fp32; null = only report *count): what = 0 style
 * gradients (layer-blocked [batch * soff_l + n * cin_l + i], conv layers then toRGB layers), 1 styles (same layout),
 * 2 demodulation coefficients, 3 d loss / d w of the synthesis path [batch, w_dim], 4 the per-layer block offsets. */
int la_debug_get(la_engine* e, int what, float* d_out, size_t* count, la_stream stream);

#ifdef __cplusplus
}
#endif
#endif
