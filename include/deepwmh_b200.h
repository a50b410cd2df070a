/* deepwmh_b200.h -- C ABI of the B200-native DeepWMH / nnU-Net 3d_fullres inference path.
 *
 * The reference (lchdl/DeepWMH) reaches this path through a process boundary:
 *   deepwmh/main/predict.py:153-156            run_shell('nnUNet_predict -i .. -o .. -tr nnUNetTrainerV2 ...')
 *   deepwmh/pipeline/DCNN_multistage.py:331-344,531-535   (same CLI, --save_softmax / --disable_tta)
 * and, inside that process, through the Python predictor surface of the un-vendored nnunet fork
 *   nnUNetTrainerV2.predict_preprocessed_data_return_seg_and_softmax / SegmentationNetwork.predict_3D
 * (SURVEY.md section 8a rows a6/a7).  There is no FFI in the reference for it; these entry points
 * are what a ctypes binding placed at that seam binds (INTEGRATION.md shows the stub).
 *
 * Conventions: every function returns 0 on success, non-zero on failure; dwmh_last_error() gives
 * the thread-local message.  One dwmh_ctx per GPU, not re-entrant; distinct contexts are
 * independent.  Device pointers are plain CUDA device addresses owned by the caller; `stream` is
 * a cudaStream_t passed as void* (NULL = default stream).  Volumes are C-ordered [X][Y][Z]
 * (Z fastest); inputs of M = in_channels modalities are channel-major [M][X][Y][Z] and class maps
 * [C][X][Y][Z] with C = num_classes, exactly the (c, x, y, z) numpy arrays nnU-Net hands to and
 * returns from predict_3D.  DeepWMH's own model has M = 1 and C = 2.
 * No torch types, no exceptions and no Python objects cross this line.
 */
#ifndef DEEPWMH_B200_H_
#define DEEPWMH_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DWMH_MAX_POOL 7
#define DWMH_MAX_IN_CHANNELS 4   /* modalities: the multi-modality first conv keeps 4 input slices per modality and one
                                    weight tile per modality in one SM's shared memory */
#define DWMH_MAX_CLASSES 8       /* classes (incl. background): the head keeps every class's logit of two voxels in registers */

typedef struct dwmh_ctx dwmh_ctx;

/* Generic_UNet hyper-parameters, i.e. what nnUNetTrainerV2.process_plans reads from plans.pkl
 * (SURVEY.md Appendix A1/A6).  Replaces nnUNetTrainerV2.initialize_network [U]. */
typedef struct dwmh_net_desc {
  int32_t in_channels;                        /* plans['num_modalities']: 1 .. DWMH_MAX_IN_CHANNELS  */
  int32_t num_classes;                        /* network outputs, 2 .. DWMH_MAX_CLASSES: plans['num_classes'] + 1 for a
                                               * softmax model, the number of regions for a sigmoid one          */
  int32_t base_num_features;                  /* 32                                                  */
  int32_t max_num_features;                   /* 320                                                 */
  int32_t num_pool;                           /* len(pool_op_kernel_sizes)                           */
  int32_t patch_size[3];                      /* plans_per_stage[..]['patch_size']  (x, y, z)        */
  int32_t pool_op_kernel_sizes[DWMH_MAX_POOL][3];      /* each entry 1 or 2                          */
  int32_t conv_kernel_sizes[DWMH_MAX_POOL + 1][3];     /* each entry 1 or 3                          */
  int32_t act_dtype;                          /* 0 = fp16 operands/storage (default), 1 = bf16       */
  int32_t max_batch;                          /* patch forwards per batch (multiple of the mirror count), 0 = default 8 */
  int32_t head_nonlin;                        /* the model's inference_apply_nonlin: 0 = softmax over classes (default),
                                               * 1 = sigmoid per output (region-based trainers, e.g. nnUNetTrainerV2BraTSRegions) */
  int32_t struct_size;                        /* MUST be sizeof(dwmh_net_desc): dwmh_create rejects any other value, so a
                                               * binding built against another layout of this struct fails loudly instead
                                               * of being read past its end                                           */
} dwmh_net_desc;

const char* dwmh_last_error(void);
/* 101: the separate two-class argmax entry point is gone; dwmh_argmax takes two classes like any other count.
 * 102: dwmh_net_desc.head_nonlin (sigmoid-head models) and dwmh_region_labels. */
int dwmh_version(void);

/* --- life cycle (replaces load_model_and_checkpoint_files + trainer.initialize(False)) ----------
 * dwmh_create fails for in_channels or num_classes outside the bounds above, for head_nonlin other than 0 or 1, and for
 * in_channels > 1 with base_num_features > 32. */
int dwmh_create(dwmh_ctx** out, int device, const dwmh_net_desc* desc);
int dwmh_destroy(dwmh_ctx* ctx);
/* A further model on the same device that BORROWS the activation workspaces of `parent` (k resident models of the
 * checkpoint ensemble, predict_cases' `for p in params` loop / DCNN_multistage.py:320-345: ~60 MB of packed weights per
 * model instead of another set of activation buffers).  Same dwmh_net_desc as the parent.  The parent's weights must be
 * committed first, the parent must outlive the borrower, and contexts sharing workspaces run on ONE stream at a time. */
int dwmh_create_like(dwmh_ctx** out, dwmh_ctx* parent);

/* trainer.load_checkpoint_ram: one call per state_dict entry, nnU-Net key names
 * ("conv_blocks_context.0.blocks.0.conv.weight", "tu.3.weight", "seg_outputs.4.weight", ...),
 * fp32 host data in PyTorch layout.  Unknown keys of the deep-supervision heads 0..num_pool-2 are
 * accepted and ignored (discarded at inference).  dwmh_commit_weights repacks to device layouts and
 * fails if a required tensor is missing. */
int dwmh_set_weight(dwmh_ctx* ctx, const char* nnunet_key, const float* data, const int64_t* shape, int32_t ndim);
int dwmh_commit_weights(dwmh_ctx* ctx);

/* --- a2: GenericPreprocessor.resample_and_normalize, non-CT scheme [U] -------------------------
 * In place on a device fp32 volume of n voxels: ONE modality (nnU-Net normalises each modality on its own,
 * so a multi-modality input takes one call per channel, each channel 16-byte aligned).
 * mask_mode 0: use_mask_for_norm False -> statistics over all voxels, all voxels normalised.
 * mask_mode 1: mask = (seg[i] >= 0), seg = device int8 array (nnU-Net's nonzero mask); outside -> 0.
 * mask_mode 2: mask = (vol[i] != 0)   (the benchmark's definition, SURVEY.md section 8d).
 * x = (x - mean) / (std + 1e-8), population std.  stats_out (host, may be NULL) receives {mean, std, count}. */
int dwmh_zscore(dwmh_ctx* ctx, float* vol_dev, const int8_t* seg_dev, int64_t n, int32_t mask_mode,
                double* stats_out, void* stream);

/* --- a8/a9 host helpers -------------------------------------------------------------------------
 * _compute_steps_for_sliding_window: writes up to max_steps entries per axis, returns counts.
 * _get_gaussian(patch, 1/8): closed form of scipy's separable filter of a unit impulse. */
int dwmh_compute_steps(const int32_t patch[3], const int32_t image[3], double step_size,
                       int32_t* steps_x, int32_t* steps_y, int32_t* steps_z, int32_t max_steps, int32_t counts[3]);
int dwmh_gaussian_map(const int32_t patch[3], double sigma_scale, float* out_host);
/* Optional: install a caller-computed importance map (host fp32 [px][py][pz]) instead of the closed form. */
int dwmh_set_importance_map(dwmh_ctx* ctx, const float* map_host);

/* --- a7/a11/a12: SegmentationNetwork.predict_3D, tiled branch -----------------------------------
 * vol_dev: normalised fp32 [M][X][Y][Z], each extent >= patch (caller pads, a10).
 * Accumulates into agg_dev fp32 [C][X][Y][Z] and wgt_dev fp32 [X][Y][Z] (caller zero-initialises):
 *   agg[:, tile] += gaussian * sum_m (1/M) unflip_m(nonlin(net(flip_m(tile)))),  wgt[tile] += gaussian
 * with nonlin the model's inference nonlinearity (softmax over classes, or a sigmoid per output for head_nonlin = 1; the
 * latter rounds the product before the add, as the reference's `*=` then `+=` do)
 * for the tiles with linear index in [tile_begin, tile_end) in x-outer / y / z-inner order
 * (tile_end < 0 = all).  mirror_axes_mask: bit a set = axis a in mirror_axes; do_mirroring = 0 -> M = 1.
 * use_gaussian = 0 (or a single tile) -> weights of 1.  Tile-sharded multi-GPU runs reduce agg and
 * wgt across ranks between this call and dwmh_finalize. */
int dwmh_predict_3d(dwmh_ctx* ctx, const float* vol_dev, int32_t X, int32_t Y, int32_t Z,
                    double step_size, int32_t do_mirroring, int32_t mirror_axes_mask, int32_t use_gaussian,
                    float* agg_dev, float* wgt_dev, int32_t tile_begin, int32_t tile_end, void* stream);

/* The weight buffer the complete tile set leaves behind (wgt of dwmh_predict_3d over all tiles, bit-identical: the
 * importance map of the covering tiles added per voxel in tile order).  It does not depend on the data, so a rank of a
 * tile-sharded run computes it locally and only agg crosses NVLink.  Overwrites wgt_dev fp32 [X][Y][Z]. */
int dwmh_weight_map(dwmh_ctx* ctx, int32_t X, int32_t Y, int32_t Z, double step_size, int32_t use_gaussian,
                    float* wgt_dev, void* stream);

/* class_probabilities = agg / wgt ; seg = argmax over classes (first maximum wins).
 * softmax_dev fp32 [C][X][Y][Z] (may alias agg_dev), seg_dev uint8 [X][Y][Z] with values 0 .. C-1; either may be NULL.
 * The same for a sigmoid-head model (upstream's regions_class_order = None); its region labels come from
 * dwmh_region_labels on the probabilities, with seg_dev NULL here. */
int dwmh_finalize(dwmh_ctx* ctx, const float* agg_dev, const float* wgt_dev, float* softmax_dev,
                  uint8_t* seg_dev, int32_t X, int32_t Y, int32_t Z, void* stream);

/* a13 ensemble: acc += softmax / k  (k-model mean of predict_cases), n floats. */
int dwmh_axpy(dwmh_ctx* ctx, float* acc_dev, const float* x_dev, float alpha, int64_t n, void* stream);
/* seg = argmax over num_classes (1 .. 255) of softmax_dev fp32 [num_classes][nvox]; the first maximum wins (ties go to the
 * lower class, as numpy.argmax). */
int dwmh_argmax(dwmh_ctx* ctx, const float* softmax_dev, int32_t num_classes, uint8_t* seg_dev, int64_t nvox, void* stream);
/* Labels of a region-based model (nnU-Net v1 with regions_class_order): seg = 0, then for r = 0 .. num_regions-1 in order
 * seg[probs[r] > 0.5] = region_class_order_host[r] -- a later region overwrites an earlier one, exactly 0.5 and NaN are
 * outside.  probs_dev fp32 [num_regions][nvox] (the sigmoid probabilities), region_class_order_host HOST int32
 * [num_regions], seg_dev uint8 [nvox].  Refused before any device work: a null pointer, num_regions outside
 * 1 .. DWMH_MAX_CLASSES, a label outside 0 .. 255, nvox <= 0. */
int dwmh_region_labels(dwmh_ctx* ctx, const float* probs_dev, int32_t num_regions, const int32_t* region_class_order_host,
                       uint8_t* seg_dev, int64_t nvox, void* stream);

/* --- SURVEY 8f-3: checkpoint ensemble with softmax masking (deepwmh/pipeline/DCNN_multistage.py:102-125,317-394).
 * dwmh_ensemble_masked_add: acc += 1 - m (1 - x) for one checkpoint's BACKGROUND probability x (the fork's
 * `<case>_0.nii.gz`), valid mask m (NULL = all ones), with the reference's rounding (float32 arrays from load_nifti_simple: one rounding per operation).
 * dwmh_ensemble_refine: acc /= k (the ensembled field, in place) and label = acc < 0.5 (label_dev may be NULL). */
int dwmh_ensemble_masked_add(dwmh_ctx* ctx, float* acc_dev, const float* bg_softmax_dev, const float* valid_mask_dev,
                             int64_t n, void* stream);
int dwmh_ensemble_refine(dwmh_ctx* ctx, float* acc_dev, int32_t k, uint8_t* label_dev, int64_t n, void* stream);

/* --- SURVEY 8f-2: `remove_sparks` (deepwmh/analysis/image_ops.py:325-344; called from predict.py:19-26,158-163) on the
 * device: 6-connected components of seg_dev > 0 (scipy.ndimage.label's default), components with fewer than
 * min_volume voxels are discarded, the rest become 1.  seg_dev / out_dev: uint8 [X][Y][Z], may alias.  The
 * voxel-size rule of remove_3mm_sparks (:346-367) stays on the host (deepwmh_b200/preprocess.py). */
int dwmh_remove_sparks(dwmh_ctx* ctx, const uint8_t* seg_dev, int32_t X, int32_t Y, int32_t Z, int32_t min_volume,
                       uint8_t* out_dev, void* stream);

/* nnU-Net v1 postprocessing, one entry of postprocessing.json: mask = label is in the class set (bit c of class_mask, bit 0 must be
 * clear); 6-connected components of mask; the components with the largest voxel count are kept, every other one is set to 0
 * unless min_valid_mm3 >= 0 and count * volume_per_voxel >= min_valid_mm3 (fp64).  No host synchronisation.
 * seg_dev: uint8 [X][Y][Z], modified in place; voxels outside the mask are never written.  Five launches, all on `stream`.
 * Refused before any device work: null ctx / seg_dev, an empty volume, X*Y*Z >= 2^31, class_mask == 0 or with bit 0 set,
 * volume_per_voxel <= 0 or not finite, min_valid_mm3 NaN.  Applying a whole for_which_classes list is one call per entry,
 * in order (deepwmh_b200/postprocessing.py). */
int dwmh_keep_largest_components(dwmh_ctx* ctx, uint8_t* seg_dev, int32_t X, int32_t Y, int32_t Z, uint32_t class_mask,
                                 double volume_per_voxel, double min_valid_mm3, void* stream);

/* --- SURVEY 8f-4: stage-1 NLL anomaly map (deepwmh/analysis/lesion_analysis.py:84-176) ---------------------------
 * Context-free (no network involved): `device` is the CUDA ordinal; every buffer is a caller-owned device pointer,
 * volumes fp32 [X][Y][Z], masks fp32 with the reference's `> 0.5` convention.  fp64 arithmetic per voxel, fp32 storage.
 * Every call runs on `device`, enqueues on `stream` and restores the calling thread's current CUDA device on return.
 *
 * dwmh_s1_zscore: z_score (deepwmh/analysis/image_ops.py:172-179, masked_mean/std :13-21) in place:
 *   x = (x - mean_mask) / max(std_mask, 1e-5) for ALL voxels (mask NULL = statistics over everything).
 *   fill_outside != 0 additionally applies lesion_analysis.py:150-151: voxels with mask < 0.5 <- min of z inside.
 *   workspace: >= 64 bytes of device memory.  stats_out (host, may be NULL) = {mean, std, count} (synchronises). */
int dwmh_s1_zscore(int32_t device, float* x_dev, const float* mask_dev, int64_t n, int32_t fill_outside, void* workspace_dev,
                   double* stats_out, void* stream);
/* The same for nvol <= 33 volumes sharing one mask in ONE launch pair (target + registered references of a case):
 * xs = HOST array of nvol device pointers; workspace >= 64 * nvol bytes. */
int dwmh_s1_zscore_batch(int32_t device, float* const* xs, int32_t nvol, const float* mask_dev, int64_t n, int32_t fill_outside,
                         void* workspace_dev, void* stream);
/* mean_std_grid(data, patch_size, order=1, mask) (image_ops.py:56-170): mean / std of the half-overlapping patch blocks
 * of the zero-padded volume, zero-bordered, linearly zoomed by the step (scipy.ndimage.zoom, order 1) and cropped.
 * mask_dev NULL = the unmasked branch; std_out_dev may be NULL.  workspace: dwmh_s1_mean_std_grid_workspace() bytes. */
int dwmh_s1_mean_std_grid_workspace(int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], int64_t* bytes);
int dwmh_s1_mean_std_grid(int32_t device, const float* x_dev, const float* mask_dev, int32_t X, int32_t Y, int32_t Z,
                          const int32_t patch_size[3], float* mean_out_dev, float* std_out_dev, void* workspace_dev, void* stream);
/* lesion_analysis.py:163-169 fused for a whole case: local mean of the target and of the k references (k <= 32, may be 0;
 * refs = HOST array of device pointers), then every reference aligned in place, x_i = x_i - x_i_local_mu + x_prime_local_mu,
 * evaluated from the coarse grids (the references' local-mean volumes are never written).  target_local_mu_out_dev
 * (may be NULL) receives x_prime_local_mu.  Three launches in total. */
int dwmh_s1_local_mean_align_workspace(int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], int32_t k, int64_t* bytes);
int dwmh_s1_local_mean_align(int32_t device, const float* target_dev, float* const* refs, int32_t k, const float* mask_dev,
                             int32_t X, int32_t Y, int32_t Z, const int32_t patch_size[3], float* target_local_mu_out_dev,
                             void* workspace_dev, void* stream);
/* x = x - local_mu + target_local_mu, in place (lesion_analysis.py:166-169: align a reference to the target). */
int dwmh_s1_align_local_mean(int32_t device, float* x_dev, const float* local_mu_dev, const float* target_local_mu_dev, int64_t n, void* stream);
/* nll(x_prime, x_refs, min_std, side, return_all) (lesion_analysis.py:84-113, use_mask=False) with group_mean / group_std
 * (image_ops.py:197-231) fused: refs = HOST array of k device pointers (k <= 32); min_std < 0 selects the `sigma += 1e-6`
 * branch; side +1 / -1 / 0 = '+' / '-' / None; mul_mask_dev (may be NULL) multiplies the score (`anomaly * m_valid_score`);
 * anomaly / mu / sigma outputs may each be NULL. */
int dwmh_s1_group_nll(int32_t device, const float* x_prime_dev, const float* const* refs, int32_t k, double min_std, int32_t side,
                      const float* mul_mask_dev, float* anomaly_dev, float* mu_out_dev, float* sigma_out_dev, int64_t n, void* stream);
/* The same with one mask per reference (group_mean / group_std with masks, image_ops.py:197-231; the Otsu branch of nll,
 * lesion_analysis.py:87-92): reference k counts at a voxel only where ref_masks[k] >= 0.5; a voxel no reference covers gets
 * mu = sigma = NaN and anomaly 0 (np.nan_to_num). */
int dwmh_s1_group_nll_masked(int32_t device, const float* x_prime_dev, const float* const* refs, const float* const* ref_masks, int32_t k,
                             double min_std, int32_t side, const float* mul_mask_dev, float* anomaly_dev, float* mu_out_dev,
                             float* sigma_out_dev, int64_t n, void* stream);
/* scipy.ndimage.median_filter(size=kernel_size, mode='constant', cval=0) as used by median_3mm (image_ops.py:181-183,
 * 378-421; kernel-size rule on the host: deepwmh_b200/stage1.py).  Sizes 1..9 per axis, in != out.  Bit-exact. */
int dwmh_s1_median_filter(int32_t device, const float* in_dev, float* out_dev, int32_t X, int32_t Y, int32_t Z,
                          const int32_t kernel_size[3], void* stream);

/* component_filtering(mask, voxel_size) (image_ops.py:253-306): per slice of every filtered orientation, 2-D erosion and the
 * largest 4-connected component (first label on ties); thin-slice data filters all three orientations, thick-slice data
 * (max / min voxel size > 3) only across the thick axis while the other two orientations add the mask itself; out = sum > 0.5
 * as 0 / 1 floats.  Integer work, bit-exact.  workspace: dwmh_s1_component_filtering_workspace() bytes; mask != out. */
int dwmh_s1_component_filtering_workspace(int32_t X, int32_t Y, int32_t Z, int64_t* bytes);
int dwmh_s1_component_filtering(int32_t device, const float* mask_dev, int32_t X, int32_t Y, int32_t Z, const double voxel_size[3],
                                float* out_dev, void* workspace_dev, void* stream);

/* Otsu support (skimage.filters.threshold_otsu as called at lesion_analysis.py:145-146, image_ops.py:308-323; skimage is not
 * vendored: its published 256-bin algorithm is restated, the 256-entry scan runs on the host -- deepwmh_b200/stage1.py).
 * dwmh_s1_minmax: min / max over mask > 0.5 (NULL = all voxels) -> host out[2]; workspace >= 8 bytes; synchronises.
 * dwmh_s1_histogram: numpy.histogram binning for nbins equal-width bins given their nbins + 1 edges (device, float64):
 *   bin i holds edges[i] <= v < edges[i+1], last bin closed, exact edge corrections.  Voxels with mask < 0.5 are skipped
 *   (fill_outside = 0) or counted as fill_value (np.where(mask < 0.5, fill, x)).  counts_dev: uint64 [nbins].
 * dwmh_s1_threshold_mask: out = (x > threshold) * mul_mask   (mul_mask may be NULL). */
int dwmh_s1_minmax(int32_t device, const float* x_dev, const float* mask_dev, int64_t n, void* workspace_dev, float out_minmax[2], void* stream);
int dwmh_s1_histogram(int32_t device, const float* x_dev, const float* mask_dev, int64_t n, int32_t fill_outside, float fill_value,
                      const double* edges_dev, int32_t nbins, uint64_t* counts_dev, void* stream);
int dwmh_s1_threshold_mask(int32_t device, const float* x_dev, float threshold, const float* mul_mask_dev, float* out_dev, int64_t n, void* stream);

/* Histogram-curve and tissue-prior steps of nll_analysis (lesion_analysis.py:52-82,188-243).
 * dwmh_s1_masked_sums: {sum, sum of squares, count} of nvol <= 33 volumes over mask > 0.5 (and v > 0 if positive_only), one
 *   launch; out_host: double [nvol][3]; workspace >= 64 * nvol bytes; synchronises.  (bin width of histogram_analysis :64-66)
 * dwmh_s1_label_vote: average_contiguous_labels (image_ops.py:23-38; per-voxel argmax of the label histogram over the k maps,
 *   first maximum wins, label ids < num_labels <= 16) and tissue_majority = (#maps with label > 0.5) > k / 2 (:238-242);
 *   labels = HOST array of k device pointers to fp32 label maps; either output may be NULL.
 * dwmh_s1_apply_priors: stage 1: anomaly *= (averaged_label > 0.5) (:216);
 *   stage 2: anomaly = (1.5 < averaged_label < 2.5 ? anomaly_median : anomaly) * tissue_majority (:232-243).  In place. */
int dwmh_s1_masked_sums(int32_t device, const float* const* xs, int32_t nvol, const float* mask_dev, int64_t n, int32_t positive_only,
                        void* workspace_dev, double* out_host, void* stream);
int dwmh_s1_label_vote(int32_t device, const float* const* labels, int32_t k, int32_t num_labels, float* averaged_label_dev,
                       float* tissue_majority_dev, int64_t n, void* stream);
int dwmh_s1_apply_priors(int32_t device, float* anomaly_dev, const float* anomaly_median_dev, const float* averaged_label_dev,
                         const float* tissue_majority_dev, int32_t stage, int64_t n, void* stream);

/* --- SURVEY 8f-1: spacing resample (resample_data_or_seg [U:preprocessing/preprocessing.py]; the resample-back of
 * save_segmentation_nifti_from_softmax [U:inference/segmentation_export.py]) on the device, context-free.
 * skimage.transform.resize(order, mode='edge', anti_aliasing=False, clip=True) semantics, fp64 arithmetic:
 *   src_dev fp32 [in_shape] -> dst_dev [out_shape]; order 3 (image data), 1 (crop mask, softmax) or 0;
 *   separate_axis >= 0: nnU-Net's "separate z" rule -- the resize runs per slice orthogonal to that axis and the axis
 *   itself is resampled nearest-neighbour (order_z = 0); -1: full 3-D resize.
 *   out_mode 0: dst fp32.  out_mode 1: dst int8 = (value >= 0.5 ? 0 : -1), i.e. resize_segmentation of nnU-Net's
 *   {-1, 0} crop mask when src is the 0/1 indicator of label 0.
 * workspace_dev: dwmh_resample_workspace() bytes of device memory. */
int dwmh_resample_workspace(const int32_t in_shape[3], int32_t order, int32_t separate_axis, int64_t* bytes);
int dwmh_resample(int32_t device, const float* src_dev, const int32_t in_shape[3], void* dst_dev, const int32_t out_shape[3],
                  int32_t order, int32_t separate_axis, int32_t out_mode, void* workspace_dev, void* stream);

/* --- nnU-Net's CT intensity normalisation [U:GenericPreprocessor.resample_and_normalize] of one modality, in place on the
 * device, context-free.  vol_dev fp32 [n]; lb / ub = intensityproperties' percentile_00_5 / percentile_99_5.  Every constant
 * is rounded to fp32 and the arithmetic is fp32 with IEEE division:
 *   DWMH_NORM_CT:  x = (clip(x, lb, ub) - mean) / sd, mean / sd from the plans (> 0).  No synchronisation; any alignment
 *                  (128-bit accesses when vol is 16-byte and seg 4-byte aligned).  stats_host must be NULL.
 *   DWMH_NORM_CT2: mask = lb < x < ub on the unclipped values; x = (clip(x, lb, ub) - mn) / sd with mn / sd the mean and
 *                  population std of x over the mask, accumulated in fp64 (deterministic, one cooperative launch; mean / sd
 *                  are ignored).  vol 16-byte, seg 4-byte aligned; workspace_dev: DWMH_CT_WORKSPACE_BYTES of 8-byte aligned
 *                  device memory, not shared with a call in flight.  stats_host (may be NULL) = {mn, sd, mask count} in fp64,
 *                  which synchronises the stream; an empty mask leaves NaN in vol and a count of 0.
 * seg_dev (may be NULL): int8 crop mask [n]; x = 0 where seg < 0 (use_mask_for_norm).  Refused before any device work: a
 * null vol, n <= 0, another scheme, a non-finite lb / ub (or, for CT, mean / sd), lb > ub, sd <= 0 for CT.
 * "noNorm" needs no call; "nonCT" is dwmh_zscore.  The host-buffer calls (dwmh_predict_volume_host*) normalise with the
 * z-score only. */
#define DWMH_NORM_CT 1
#define DWMH_NORM_CT2 2
#define DWMH_CT_WORKSPACE_BYTES 65536
int dwmh_ct_normalize(int32_t device, float* vol_dev, const int8_t* seg_dev, int64_t n, int32_t scheme, double lb, double ub,
                      double mean, double sd, double* stats_host, void* workspace_dev, void* stream);

/* --- The 3d_cascade_fullres input [U:inference/predict.py::preprocess_save_to_queue], context-free: labels_dev uint8
 * [in_shape] (the previous stage's labels after transpose_forward, values 0 .. num_classes-1) -> resize_segmentation(labels,
 * out_shape, order=1) -> one-hot over classes 1 .. num_classes-1 as fp32 0 / 1 planes dst_dev [num_classes-1][out_shape]
 * (the network input's channels after the modalities).  Bit-exact: the order-1 taps of dwmh_resample in fp64.  Refused
 * before any device work: a null pointer, an extent <= 0, num_classes outside 2 .. DWMH_MAX_CLASSES. */
int dwmh_cascade_onehot(int32_t device, const uint8_t* labels_dev, const int32_t in_shape[3], float* dst_dev,
                        const int32_t out_shape[3], int32_t num_classes, void* stream);

/* --- N4 bias-field correction (the `N4BiasFieldCorrection -d 3 -c [50x50x50x50,0.0] -s 2` step of DeepWMH_predict,
 * deepwmh/main/predict.py:117-126) on the device, context-free.  Restated from Tustison et al. 2010 with 200 bins, FWHM 0.15,
 * Wiener noise 0.01, cubic B-splines on an initial 1 x 1 x 1 mesh doubled per level, convergence threshold 0
 * (oracle/n4_oracle.py, DESIGN.md).  in_dev fp32 [X][Y][Z]; voxels <= 0 take no part in the fit.  Shrink by `shrink` per axis
 * (floor(N / shrink) points, at least 2 per axis), num_levels <= 8 fitting levels with iterations_host[level] iterations each
 * (HOST array).  out_dev = in / exp(B); log_field_dev (may be NULL) = B.  in_dev may alias out_dev.  Deterministic: two calls
 * are bit-identical.  No host synchronisation.  workspace_dev: dwmh_n4_workspace() bytes of device memory. */
int dwmh_n4_workspace(int32_t X, int32_t Y, int32_t Z, int32_t shrink, int32_t num_levels, int64_t* bytes);
int dwmh_n4(int32_t device, const float* in_dev, int32_t X, int32_t Y, int32_t Z, int32_t shrink, int32_t num_levels,
            const int32_t* iterations_host, float* out_dev, float* log_field_dev, void* workspace_dev, void* stream);

/* --- a6 end to end with HOST buffers (what predict_preprocessed_data_return_seg_and_softmax does):
 * raw fp32 volume [M][X][Y][Z] in host memory -> (optional z-score of every modality, mask_mode as above, <0 = skip)
 * -> tiled prediction -> host softmax fp32 [C][X][Y][Z] and seg uint8 [X][Y][Z].  H2D/D2H inside.  The probabilities are
 * those of the model's inference nonlinearity; seg is always the argmax (region labels: dwmh_region_labels on device
 * buffers). */
int dwmh_predict_volume_host(dwmh_ctx* ctx, const float* vol_host, int32_t X, int32_t Y, int32_t Z,
                             int32_t zscore_mask_mode, double step_size, int32_t do_mirroring,
                             int32_t mirror_axes_mask, int32_t use_gaussian,
                             float* softmax_host, uint8_t* seg_host, void* stream);

/* The same with nnU-Net's own normalisation mask (mask_mode 1): seg_mask_host int8 [X][Y][Z], >= 0 inside the
 * hole-filled non-zero crop mask (crop_to_nonzero [U:preprocessing/cropping.py]), -1 outside; one mask for all modalities. */
int dwmh_predict_volume_host_masked(dwmh_ctx* ctx, const float* vol_host, const int8_t* seg_mask_host,
                                    int32_t X, int32_t Y, int32_t Z, double step_size, int32_t do_mirroring,
                                    int32_t mirror_axes_mask, int32_t use_gaussian,
                                    float* softmax_host, uint8_t* seg_host, void* stream);

/* --- test / profiling hooks ----------------------------------------------------------------------
 * Generic_UNet.forward + the model's inference nonlinearity (softmax, or sigmoid for head_nonlin = 1) on n patches:
 * patches_dev fp32 [n][M][px][py][pz] -> probs_dev fp32 [n][C][px][py][pz]. */
int dwmh_forward_patches(dwmh_ctx* ctx, const float* patches_dev, int32_t n, float* probs_dev, void* stream);
/* Copy the (normalised, activated) output of layer `layer_index` of the last forward, converted to
 * fp32 NCDHW, into out_dev (capacity in floats); dims_out = {n, c, d, h, w}.  Layer order = execution order. */
int dwmh_debug_layer_output(dwmh_ctx* ctx, int32_t layer_index, float* out_dev, int64_t capacity, int32_t dims_out[5], void* stream);
/* The same for samples first, first + 1, ... of the last forward (dims_out[0] = how many were copied). */
int dwmh_debug_layer_output_from(dwmh_ctx* ctx, int32_t layer_index, int32_t first, float* out_dev, int64_t capacity,
                                 int32_t dims_out[5], void* stream);
int dwmh_num_layers(dwmh_ctx* ctx);
/* What the launch of layer `layer_index` at batch nb (1 .. max_batch) would run, computed by the functions the launch itself
 * uses; read-only.  Valid after dwmh_commit_weights.  out[DWMH_PLAN_KIND] is one of DWMH_PLAN_FIRST / CONV / TCONV /
 * CUDA_CORE; for a CUDA-core layer only KIND, KD, the strides and ACT are set (the rest is 0).  G is the tile pipelines per
 * CTA after the launch's pairing rule, ITEMS = nb * ncb * nzb * tiles, GRID = CTAs. */
enum {
  DWMH_PLAN_KIND = 0, DWMH_PLAN_KD, DWMH_PLAN_SD, DWMH_PLAN_SH, DWMH_PLAN_SW,
  DWMH_PLAN_KC, DWMH_PLAN_KSTEPS, DWMH_PLAN_CB, DWMH_PLAN_NCB, DWMH_PLAN_RESIDENT, DWMH_PLAN_SA, DWMH_PLAN_NB, DWMH_PLAN_R,
  DWMH_PLAN_G, DWMH_PLAN_ZB, DWMH_PLAN_NZB, DWMH_PLAN_TILES, DWMH_PLAN_ITEMS, DWMH_PLAN_GRID,
  DWMH_PLAN_XFORM, DWMH_PLAN_S222, DWMH_PLAN_ACT,
  DWMH_LAYER_PLAN_FIELDS
};
enum { DWMH_PLAN_FIRST = 0, DWMH_PLAN_CONV = 1, DWMH_PLAN_TCONV = 2, DWMH_PLAN_CUDA_CORE = 3 };
int dwmh_layer_plan(dwmh_ctx* ctx, int32_t layer_index, int32_t nb, int32_t out[DWMH_LAYER_PLAN_FIELDS]);
/* Kernel variant used by a layer: 0 = direct (CUDA cores), 1 = tcgen05 implicit GEMM. */
int dwmh_layer_kernel_kind(dwmh_ctx* ctx, int32_t layer_index);
/* 1 when the layer's InstanceNorm + LeakyReLU are applied by its consumer on load (no separate pass, the layer's buffer keeps
 * the raw conv output), 0 otherwise, -1 for a bad index.  Valid after dwmh_commit_weights. */
int dwmh_layer_norm_on_load(dwmh_ctx* ctx, int32_t layer_index);
/* Force the generic kernels everywhere (1) or restore automatic selection (0) - for cross-checking. */
int dwmh_set_force_generic(dwmh_ctx* ctx, int32_t on);
/* Counters since creation: kernels launched by this library, conv FLOPs issued. */
int dwmh_get_counters(dwmh_ctx* ctx, int64_t* kernel_launches, double* conv_flops);
/* Device time (ms, CUDA events on `stream`) the last dwmh_predict_3d spent per stage:
 * out[0]=conv stack (all kernels of the forwards), out[1]=aggregate, out[2]=sum of the tcgen05 conv kernel launches
 * (CUDA events around every launch), out[3]=TFLOP those launches computed.  Only filled when enabled (adds syncs). */
int dwmh_set_stage_timing(dwmh_ctx* ctx, int32_t on);
int dwmh_get_stage_timing(dwmh_ctx* ctx, float out_ms[4]);
/* Per kernel class of the last timed dwmh_predict_3d: out[3k + {0,1,2}] = {device ms, algorithmic bytes, launches} for
 * k = 0 conv3_tc_kernel (bytes not counted here), 1 instnorm_lrelu_kernel, 2 head_softmax_kernel (any class count). */
int dwmh_get_kernel_timing(dwmh_ctx* ctx, double out[9]);

#ifdef __cplusplus
}
#endif
#endif /* DEEPWMH_B200_H_ */
