/*
 * humanrf_b200 -- C ABI of the B200-native (sm_100a) HumanRF per-ray hot path.
 *
 * Drop-in boundary for the reference's three pybind11 torch extensions and the two
 * third-party CUDA packages its hot path calls (SURVEY.md section 8b).  Every entry point
 * takes plain DEVICE pointers (unless the name says host) + sizes + a CUDA stream handle
 * (cudaStream_t passed as void*, NULL = legacy default stream); no torch types.  All
 * functions return 0 on success and a non-zero code on failure; hrf_last_error() gives the
 * message (the reference throws std::runtime_error from CHECK_CONTIGUITY_AND_DEVICE,
 * actorshq/toolbox/native/utils.cuh:5-19; the Python host mirror raises RuntimeError).
 * Launches are asynchronous on the given stream; nothing here synchronises except the
 * functions documented as doing so.
 */
#ifndef HUMANRF_B200_H_
#define HUMANRF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HRF_N_LEVELS 16        /* humanrf/args/model_args.py:26 n_levels            */
#define HRF_N_FEATURES 32      /* n_levels * n_features_per_level (2)               */
#define HRF_MLP_WIDTH 64       /* model_args.py:12 n_neurons                        */
#define HRF_GEO_DIM 15         /* model_args.py:10 geometry_feature_dim             */
#define HRF_MLP_BLOB_BYTES 22528 /* packed bf16 weights: sigma 64x32,16x64; colour 64x(32|48),64x64,16x64 */
#define HRF_MAX_CAMERA_EMBEDDING_DIM 17 /* 16 SH + 15 geo + E <= 48 */

const char* hrf_last_error(void);
int hrf_version(void);
/* device properties the host mirror needs: out[0]=SM count, out[1]=cc major, out[2]=cc minor */
int hrf_device_info(int* out3);

/* ------------------------------------------------------------------------------------------
 * Occupancy grid ring.  Replaces occupancy_grid_native.OccupanyGrid
 * (actorshq/dataset/native/occupancy_grid.cu:8-95): a ring of `buffer_size` G^3 occupancy
 * volumes; add_grid copies a uint8 [G][G][G] (z,y,x) device tensor into the next slot and
 * returns an int64 handle the sampler understands (the reference returns a
 * cudaTextureObject_t; here it is the device address of a bit-packed G^3 volume).
 * ---------------------------------------------------------------------------------------- */
typedef struct hrf_occgrid hrf_occgrid;
int hrf_occgrid_create(uint64_t grid_resolution, int buffer_size, hrf_occgrid** out);
int hrf_occgrid_destroy(hrf_occgrid* g);
int hrf_occgrid_add(hrf_occgrid* g, const uint8_t* grid_u8, uint64_t res0, uint64_t res1, uint64_t res2,
                    void* stream, int64_t* handle_out);
/* test hook: evaluates the emulated `tex3D(handle, p) > 0` for n points (xyz normalised) */
int hrf_occgrid_lookup(int64_t handle, int grid_resolution, const float* points_xyz, int64_t n,
                       uint8_t* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Ray sampler.  Replaces ray_sampler_native.get_{rays,samples}_{aabb,occupancy}_minmax
 * (actorshq/dataset/native/ray_sampler.cu:196-325).  Three phases, no host round trip inside:
 *   hrf_sampler_rays   : compute_minmax_kernel (:80-147) for all R candidate rays, ray mask
 *                        (optionally AND NOT light_mask, :254-257), device-side compaction,
 *                        per-ray gathers (:258-266) and per-ray sample counts/offsets
 *                        (:283-290, occupancy filter of :183-189 already applied).
 *                        counters[0]=R' (kept rays), counters[1]=N' (kept samples).
 *   hrf_sampler_samples: compute_sample_distances_kernel (:149-194) + final compaction
 *                        (:322-323) written directly at the scanned offsets.
 * rgba_pool / light_mask are DEVICE-resident pools here (the reference indexes a CPU pool and
 * bounces through the host, :262); the Python mirror keeps the CPU-pool call signature.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  const int32_t* frame_numbers;      /* [B] */
  const int32_t* camera_numbers;     /* [B] */
  const int64_t* grid_handles;       /* [B] from hrf_occgrid_add (unused for aabb mode) */
  const uint8_t* landscape_modes;    /* [B] bool */
  const float*   inverse_krs;        /* [B,3,3], stored transposed as the reference does (data_loader.py:194-207) */
  const float*   camera_origins;     /* [B,3] */
  const float*   aabb;               /* [2,3] */
  const uint8_t* rgba_pool;          /* [P,4] uint8 or NULL */
  const uint8_t* light_mask;         /* [P] bool, indexed by pool pixel, or NULL */
  const uint8_t* light_mask_rays;    /* [R] bool, indexed by candidate ray (host-pool callers), or NULL */
  int32_t grid_resolution, image_width, image_height;
  float step;
  int32_t occupancy;                 /* 1: occupancy minmax + filter, 0: aabb only */
  int32_t filter_light_bloom;
  int32_t want_samples;              /* 0: get_rays_* variants (counts are all zero) */
} hrf_sampler_params;

int hrf_sampler_rays(const hrf_sampler_params* p, const int64_t* all_ray_indices, int64_t num_rays,
                     /* full-size outputs [R] */
                     uint8_t* ray_mask,
                     /* compacted outputs, capacity R */
                     float* ray_origins, float* ray_directions, float* rgba, int32_t* frame_numbers,
                     int32_t* camera_numbers, float* minmaxes, int64_t* kept_ray_indices,
                     int32_t* sample_offsets /* [R+1] exclusive scan of kept-sample counts */,
                     int64_t* counters /* [2] device */, void* workspace, int64_t workspace_bytes, void* stream);
int64_t hrf_sampler_workspace_bytes(int64_t num_rays);
int hrf_sampler_samples(const hrf_sampler_params* p, int64_t num_kept_rays, const int64_t* kept_ray_indices,
                        const float* ray_origins, const float* ray_directions, const float* minmaxes,
                        const int32_t* sample_offsets, float* distances /* [N'] */,
                        int32_t* relative_ray_indices /* [N'] */, void* stream);

/* ------------------------------------------------------------------------------------------
 * Radiance field.  Replaces HumanRF.density / HumanRF.forward
 * (humanrf/scene_representation/humanrf.py:158-208): 4 tcnn HashGrids per segment
 * (decomposition4d.py:79-129), compose_tensors (tensor_composition.cu:9-55), sigma MLP +
 * truncated_exp (humanrf.py:181-186), SH/identity colour MLP (:188-206) in ONE kernel.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  const uint32_t* grid[4];           /* bf16x2 entries: xyz, xyt, yzt, xzt encodings     */
  const float*    vectors;           /* [4, vec_res, 32] fp32 (decomposition4d.py:76-78) */
  uint32_t level_offset[HRF_N_LEVELS]; /* entry offset of each level                      */
  uint32_t level_size[HRF_N_LEVELS];   /* hashmap_size of each level (entries)            */
  uint32_t hashed_mask;              /* bit l: level l uses the spatial hash             */
  uint32_t n_entries;                /* entries per grid                                 */
  /* Optional transposed fp32 copy of `vectors`, [4 axes][16 levels][vec_res][2] (hrf_transpose_vectors; kept current by
   * hrf_adam_multi / hrf_dp_reduce_adam through hrf_adam_tensor.vectors_t): the gradient scatter reads one level's
   * feature pair of consecutive rows from consecutive addresses.  NULL: the scatter reads `vectors` itself. */
  const float*    vectors_t;
} hrf_segment;

typedef struct {
  const hrf_segment* segments;       /* device array [num_segments]                      */
  const int32_t* frame_to_segment;   /* device [lut_size]   (humanrf.py:99)              */
  const float*   frame_to_tlocal;    /* device [lut_size]   (humanrf.py:100-103)         */
  const void*    mlp_blob;           /* device, HRF_MLP_BLOB_BYTES, see hrf_pack_layout   */
  float    level_scale[HRF_N_LEVELS];
  uint32_t level_res[HRF_N_LEVELS];
  int32_t  num_segments, lut_size, vec_res;
  float    density_scale;
  /* camera embeddings (humanrf.py:75-76,194-204): fp32 [num_cameras, camera_embedding_dim], or NULL / 0 */
  const float* camera_embeddings;
  int32_t  camera_embedding_dim, num_cameras;
  int32_t  color_in_width;           /* 32 (no embedding) or 48: width of the padded colour-net input */
} hrf_field;

/* Sample source: either explicit per-sample queries (QueryInput, query_io.py:6-13) or the
 * ray-batch form used by prune_samples/render (volume_rendering.py:66-72,110-119). */
typedef struct {
  /* query form (ray_origins == NULL) */
  const float* positions;            /* [N,3] in [-0.5,0.5] */
  const float* directions;           /* [N,3] or NULL for density-only */
  const int32_t* frame_numbers;      /* [N] */
  /* ray-batch form */
  const float* ray_origins;          /* [R,3] */
  const float* ray_directions;       /* [R,3] */
  const int32_t* ray_frame_numbers;  /* [R] */
  const float* sample_distances;     /* [N] */
  const int64_t* ray_indices;        /* [N] sorted ascending */
  int64_t num_samples;
  /* camera numbers, only read when the field has camera embeddings and use_camera_embeddings != 0
   * (is_training; at evaluation the embedding is all zeros, humanrf.py:196-204) */
  const int32_t* camera_numbers;     /* query form: [N] */
  const int32_t* ray_camera_numbers; /* ray-batch form: [R] */
  int32_t use_camera_embeddings;
  /* Sync-free pipelines: when non-NULL the kernels read the LIVE number of samples from this device scalar and
   * num_samples is the capacity of the per-sample arrays (grid sizing, strides of the [..][N] buffers).  This is what
   * lets a training step prune on the device and keep going without reading the survivor count back
   * (the reference reads it implicitly through boolean-mask indexing, volume_rendering.py:83-84). */
  const int64_t* num_samples_dev;
} hrf_samples;

/* mode: 0 = density only (sigma, geo), 1 = density + radiance.  Any output may be NULL.
 * mlp_impl: 0 = tcgen05 tensor-core path (the product); 1 = SIMT fp32 debug path used only by
 * tests to localise tensor-core descriptor faults. */
int hrf_field_forward(const hrf_field* f, const hrf_samples* s, int mode, int mlp_impl,
                      float* sigma /* [N] */, void* geo_bf16 /* [N,16] (col 0 = raw h0) */,
                      float* rgb /* [N,3] */, void* feat_bf16 /* [N,32] composed features saved for backward, or NULL */,
                      void* grid_feat_bf16 /* [64,N] bf16x2 per-(level,grid) interpolated features for backward, or NULL */,
                      void* stream);

/* The MLP half of hrf_field_forward for samples whose composed features already exist (the density-only pass of
 * prune_samples encodes every candidate; the render pass of the survivors does not have to encode them again):
 * feat_in_bf16 [M,32] as written by a previous pass, feat_index[i] = its row for sample i (NULL = identity).
 * `s` must be in ray-batch form (view directions / camera numbers are read through ray_indices). */
int hrf_field_forward_from_features(const hrf_field* f, const hrf_samples* s, const void* feat_in_bf16,
                                    const int32_t* feat_index, float* sigma /* [N] */, float* rgb /* [N,3] */,
                                    void* stream);

/* Inference render in ONE field kernel (humanrf/volume_rendering.py:87-150 without gradients): encode -> sigma MLP ->
 * colour MLP -> per-ray compositing, w_i = exp(-sum_{j<i} sigma_j dt_j) (1 - exp(-sigma_i dt_i)), colour = sum w rgb +
 * background (1 - sum w).  Per-sample sigma / rgb never leave the SM; a small second kernel chains the rays that
 * straddle 128-sample tile borders and writes the background for rays without samples.  Samples must be sorted by
 * ray (ray_offsets[r] = first sample of ray r).  feat_in / feat_index: optional composed features of an earlier
 * pass (hrf_field_forward_from_features semantics; then nothing is encoded here).  s->num_samples_dev is honoured.
 * workspace: hrf_render_fused_workspace_bytes(s->num_samples) bytes of device scratch. */
int64_t hrf_render_fused_workspace_bytes(int64_t num_samples_capacity);
int hrf_render_fused(const hrf_field* f, const hrf_samples* s /* ray-batch form */, const int32_t* ray_offsets /* [R+1] */,
                     int64_t num_rays, float step, const float* background /* [R,3] or NULL */, const void* feat_in_bf16,
                     const int32_t* feat_index, float* color /* [R,3] */, float* weights_sum /* [R] */, void* workspace,
                     void* stream);

/* Density-only pass of prune_samples (volume_rendering.py:66-84) with an exact early stop: ray chunks are
 * evaluated front to back; once a ray's accumulated optical depth makes every later sample fail nerfacc's
 * transmittance test (T < 1e-4) those samples are reported with sigma = 0 without being evaluated.  The kept
 * set of hrf_prune on this sigma equals the one on the fully evaluated sigma.  workspace: device scratch of
 * hrf_density_early_stop_workspace_bytes(num_rays) bytes. */
int64_t hrf_density_early_stop_workspace_bytes(int64_t num_rays);
int hrf_field_density_early_stop(const hrf_field* f, const hrf_samples* s /* ray-batch form */,
                                 const int32_t* ray_offsets /* [R+1] */, int64_t num_rays, float step,
                                 float stop_depth /* > -ln(1e-4); 9.4 recommended */, float* sigma /* [N] */,
                                 void* feat_bf16 /* [N,32] composed features of every evaluated sample, or NULL */,
                                 void* grid_feat_bf16 /* [64,N] per-(level,grid) features, or NULL */,
                                 void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * Compositing.  Replaces nerfacc.render_visibility / render_weight_from_density /
 * accumulate_along_rays as called from humanrf/volume_rendering.py:75-84,123-145.
 * ---------------------------------------------------------------------------------------- */
/* ray_offsets[r] = first sample of ray r in the sorted ray_indices; ray_offsets[R] = N */
int hrf_ray_offsets(const int64_t* ray_indices, int64_t num_samples, int64_t num_rays,
                    int32_t* ray_offsets /* [R+1] */, void* stream);
/* prune: keep_i = (T_i >= 1e-4) & (alpha_i >= 1e-4), alpha = 1-exp(-sigma*step); writes the
 * kept samples compacted; counters[0] = kept count.  kept_offsets [R+1] workspace. */
int hrf_prune(const float* sigma, const float* sample_distances, const int64_t* ray_indices,
              const int32_t* ray_offsets, int64_t num_rays, float step, float early_stop_eps, float alpha_thre,
              uint8_t* keep_mask /* [N] or NULL */, int32_t* kept_offsets /* [R+1] */,
              float* out_distances, int64_t* out_ray_indices, int32_t* out_source_index /* [N] index of each kept sample
              in the input arrays, or NULL */, int64_t* counters, void* stream);
/* render: w_i = exp(-sum_{j<i} sigma_j*dt_j) * (1-exp(-sigma_i*dt_i)), dt=(t+step)-t;
 * color = sum w*rgb (+ background*(1-sum w)), weights_sum = sum w. background: [R,3] or NULL. */
int hrf_composite_forward(const float* sigma, const float* rgb, const float* sample_distances,
                          const int32_t* ray_offsets, int64_t num_rays, float step, const float* background,
                          float* color /* [R,3] */, float* weights_sum /* [R] */,
                          float* weights /* [N] or NULL */, void* stream);
/* backward of the above w.r.t. sigma and rgb given d_color [R,3], d_weights_sum [R] */
int hrf_composite_backward(const float* sigma, const float* rgb, const float* sample_distances,
                           const int32_t* ray_offsets, int64_t num_rays, float step, const float* background,
                           const float* d_color, const float* d_weights_sum,
                           float* d_sigma /* [N] */, float* d_rgb /* [N,3] */, void* stream);

/* ------------------------------------------------------------------------------------------
 * Backward of the radiance field (autograd of humanrf.py:158-208): recomputes the forward per
 * 128-sample tile, runs MLP dgrad/wgrad on the tensor cores, scatters table / vector gradients.
 * Gradients are ACCUMULATED (+=) into the fp32 buffers; the caller zeroes them.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
  float* grid[4];                    /* [n_entries,2] fp32, same order as hrf_segment.grid */
  float* vectors;                    /* [4, vec_res, 32] fp32 */
} hrf_segment_grads;

int hrf_field_backward(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads /* device array */,
                       const float* d_sigma /* [N] */, const float* d_rgb /* [N,3] or NULL */,
                       const float* d_geo /* [N,15] gradient of the geometry features, or NULL */,
                       const void* feat_bf16 /* composed features from a forward pass, or NULL to re-encode */,
                       const void* grid_feat_bf16 /* [64,stride] from a forward pass, or NULL to re-gather the tables */,
                       const int32_t* feat_index /* row of sample i in feat / grid_feat (NULL = identity) */,
                       int64_t grid_feat_stride /* row length of grid_feat (0 = num_samples) */,
                       float* d_mlp /* fp32 [3072 + 64*color_in_width + 5120]: sigma W1,W2, colour W1,W2,W3 row-major [out,in] */,
                       float* d_camera_embeddings /* fp32 [num_cameras, dim] accumulated into, or NULL */,
                       void* workspace /* 160 bytes per sample (16-byte aligned): d(features) level-major, positions, segment ids */, void* stream);
/* The same backward in two phases, so that a data-parallel trainer can start reducing one table's gradient while the
 * next table's scatter still runs: hrf_field_backward == hrf_field_backward_mlp + hrf_field_backward_tables(0, 4).
 * Table k's gradient is complete after the launch covering grid k; the vector gradients after the last launch. */
int hrf_field_backward_mlp(const hrf_field* f, const hrf_samples* s, const float* d_sigma, const float* d_rgb,
                           const float* d_geo, const void* feat_bf16, const int32_t* feat_index, float* d_mlp,
                           float* d_camera_embeddings, void* workspace, void* stream);
int hrf_field_backward_tables(const hrf_field* f, const hrf_samples* s, const hrf_segment_grads* seg_grads,
                              const void* grid_feat_bf16, const int32_t* feat_index, int64_t grid_feat_stride,
                              const void* workspace, int grid_first, int grid_count, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training loss on the per-ray outputs, forward and backward in one launch (trainer.py:205-215,229-238,
 * utils/loss.py:4-10): gt = rgb*mask + background*(1-mask); HuberLoss(delta, mean) over [R,3] +
 * bce_weight * mean(BCE(clamp(weights_sum,0,1), mask)) with eps 1e-10.  loss_out[0] += loss (caller zeroes);
 * d_color / d_weights_sum are d(loss * *loss_scale_dev) (loss_scale_dev NULL = 1: data-parallel ranks weight their
 * share of the union batch with it).
 * ---------------------------------------------------------------------------------------- */
int hrf_train_loss(const float* color /* [R,3] */, const float* weights_sum /* [R] */, const float* rgba /* [R,4] */,
                   const float* background /* [R,3] */, int64_t num_rays, float huber_delta, float bce_weight,
                   const float* loss_scale_dev, float* d_color /* [R,3] */, float* d_weights_sum /* [R] */,
                   float* loss_out /* [1], accumulated */, void* stream);

/* ------------------------------------------------------------------------------------------
 * tensor_composition_native parity (tensor_composition.cu:120-219): stand-alone fwd/bwd of
 * sum_k feat3D_k * lerp(vector_k, coord_k) on fp16 features, as the reference's extension.
 * ---------------------------------------------------------------------------------------- */
int hrf_compose_tensors_forward(const void* xyz, const void* xyt, const void* yzt, const void* xzt /* half [N,F] */,
                                const float* vectors /* [4,VR,F] */, const float* coords /* [N,4] */,
                                int64_t n, int feature_dim, int vec_res, void* out /* half [N,F] */, void* stream);
int hrf_compose_tensors_backward(const void* xyz, const void* xyt, const void* yzt, const void* xzt,
                                 const float* vectors, const float* coords, const void* d_out, int64_t n,
                                 int feature_dim, int vec_res, void* d_xyz, void* d_xyt, void* d_yzt, void* d_xzt,
                                 float* d_vectors /* zero-initialised by the callee */, void* stream);

/* ------------------------------------------------------------------------------------------
 * Optimiser: fused Adam (run.py:101-104: betas (0.9,0.99), eps 1e-15) over a flat fp32 buffer,
 * optionally refreshing the bf16 shadow copy the forward reads.  grad_scale multiplies the
 * gradient first (1/global_ray_count for data-parallel means).
 * ---------------------------------------------------------------------------------------- */
int hrf_adam_step(float* param, float* exp_avg, float* exp_avg_sq, const float* grad, void* shadow_bf16 /* or NULL */,
                  int64_t n, float lr, float beta1, float beta2, float eps, int step, float grad_scale,
                  void* stream);
int hrf_cast_bf16(const float* src, void* dst_bf16, int64_t n, void* stream);
/* vectors [4, vec_res, 32] -> vectors_t [4, 16, vec_res, 2] (hrf_segment.vectors_t) */
int hrf_transpose_vectors(const float* vectors, float* vectors_t, int vec_res, void* stream);

/* All parameter tensors of a model in ONE launch (the per-tensor entry point above costs one launch per tensor: 23
 * for a single segment).  tensors: device array of descriptors; a tensor whose *active flag is 0 is skipped entirely
 * -- parameters, moments AND its step counter -- which is what torch.optim.Adam does with a parameter whose .grad is
 * None (the reference gives untouched temporal segments no gradient, humanrf.py:162-179, trainer.py:174).  Step
 * counters live on the device (int32 per tensor, incremented here), so a step needs no host decision.  After reading
 * a gradient element the kernel writes 0 back when zero_grad != 0 (the bucket is then clean for the next backward).
 * blob_perm: for the MLP tensors, element i of the tensor is also written as bf16 to shadow[blob_perm[i]] (the packed
 * tcgen05 weight blob) instead of shadow[i]. */
typedef struct {
  float* param; float* exp_avg; float* exp_avg_sq; float* grad;
  void* shadow_bf16;                 /* or NULL */
  const int32_t* blob_perm;          /* or NULL */
  const int32_t* active;             /* device flag (segment used by this step) or NULL = always active */
  int32_t* step;                     /* device step counter of this tensor */
  int64_t n;
  int64_t first_block;               /* exclusive prefix of ceil(n / HRF_ADAM_BLOCK_ELEMS) over the tensors */
  float* vectors_t;                  /* `vectors` tensors only: the transposed copy to refresh (hrf_segment.vectors_t), or NULL */
  int32_t vec_res;
} hrf_adam_tensor;
#define HRF_ADAM_BLOCK_ELEMS 4096
int hrf_adam_multi(const hrf_adam_tensor* tensors /* device */, int num_tensors, int64_t total_blocks, float lr, float beta1,
                   float beta2, float eps, float grad_scale, int zero_grad, void* stream);

/* ------------------------------------------------------------------------------------------
 * Data-parallel training (SURVEY 8e; the reference is single-GPU, the step wrapped is trainer.py:250-253).
 * One process per GPU.  Gradient buckets and bf16 shadow tables live in peer-visible device memory
 * (hrf_peer_alloc + CUDA IPC handles exchanged by the host side); hrf_dp_reduce_adam is the whole exchange step in one
 * kernel over NVLink peer memory: for this rank's 1/world slice of every sharded tensor it sums the gradient slices of
 * all ranks (P2P loads, rank order), runs Adam on the local fp32 master / moments and stores the refreshed bf16 shadow
 * entries into every rank's shadow buffer (P2P stores); replicated (small) tensors are reduced on every rank.  The
 * caller brackets it with two cross-rank barriers (all gradients complete before; all shadows written / all buckets
 * read after) and clears its own bucket afterwards.
 * ---------------------------------------------------------------------------------------- */
#define HRF_DP_MAX_WORLD 8
int hrf_peer_alloc(int64_t bytes, void** ptr_out);        /* zero-filled, exportable (not from a pooled allocator) */
int hrf_peer_free(void* ptr);
int hrf_peer_export(void* ptr, void* handle_out64 /* 64 bytes, host */);
int hrf_peer_open(const void* handle64, void** ptr_out);  /* a handle exported by ANOTHER process */
int hrf_peer_close(void* ptr);
typedef struct {
  float* grad[HRF_DP_MAX_WORLD];     /* every rank's gradient bucket (own entry = local pointer) */
  void*  shadow[HRF_DP_MAX_WORLD];   /* every rank's flat bf16 shadow buffer */
  int32_t world, rank;
} hrf_dp_peers;
typedef struct {
  float* param; float* exp_avg; float* exp_avg_sq;   /* local tensors, full size (a sharded tensor only touches its slice) */
  int64_t grad_offset;               /* element offset of the tensor inside every gradient bucket */
  int64_t shadow_offset;             /* element offset inside every shadow buffer (sharded tensors), or -1 */
  void* local_shadow_bf16;           /* replicated tensors: local bf16 copy / packed MLP blob, or NULL */
  const int32_t* blob_perm;          /* as hrf_adam_tensor */
  const int32_t* active;
  int32_t* step;
  int64_t n;
  int64_t shard_begin, shard_end;    /* this rank's element range; [0, n) for replicated tensors */
  int64_t first_block;               /* exclusive prefix of ceil((shard_end - shard_begin) / HRF_ADAM_BLOCK_ELEMS) */
  int32_t sharded;
  int32_t vec_res;
  float* vectors_t;                  /* as hrf_adam_tensor */
} hrf_dp_tensor;
/* block_first / block_count: the range of blocks (in the first_block numbering of the descriptor table) this launch
 * covers -- the whole table, or the tensors of one hash grid so that its exchange runs while the next grid's gradient is
 * still being scattered.  advance_steps != 0 on the first launch of a step (it advances the step counters of the active
 * tensors, once). */
int hrf_dp_reduce_adam(const hrf_dp_peers* peers /* host */, const hrf_dp_tensor* tensors /* device */, int num_tensors,
                       int64_t block_first, int64_t block_count, int advance_steps, float lr, float beta1, float beta2,
                       float eps, float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Pre-processing that feeds the hot path (SURVEY 8f-4).
 * hrf_occupancy_from_masks: visual-hull carving, replaces occupancy_grid_generation_native.generate_from_masks
 * (actorshq/toolbox/native/occupancy_grid_generation.cu:16-123).  projection_matrices [C,4,4] are stored transposed
 * exactly as the reference passes them (GLM is column-major).
 * hrf_occupancy_union_count: cluster |= (grid == 255); *count_dev = popcount(cluster) -- equations (2)-(4) of
 * humanrf/adaptive_temporal_partitioning.py:11-26 on a bit-packed union (grid_u8 may be NULL to only count).
 * ---------------------------------------------------------------------------------------- */
int hrf_occupancy_from_masks(const uint8_t* masks /* [C, H*W] */, const float* projection_matrices /* [C,4,4] */,
                             const uint8_t* landscape_modes /* [C] bool */, int num_cameras, int camera_coverage_threshold,
                             int grid_resolution, int width, int height, uint8_t* occupancy_grid /* [G,G,G] */, void* stream);
int hrf_occupancy_union_count(void* cluster_bits /* ceil(n/32) u32, caller-zeroed per cluster */, const uint8_t* grid_u8 /* [n] */,
                              int64_t num_voxels, int64_t* count_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Validation metrics (humanrf/trainer.py:373-419 and actorshq/evaluation/evaluate.py:76-85 without LPIPS), all on the
 * device with no host read.
 * hrf_mask_bbox: box = cv2.boundingRect(mask > 0) as int32 (x, y, w, h); an empty mask gives (0, 0, 0, 0).
 * hrf_image_metrics: im1 / im2 are [height, width, 3] images (fp32, or uint8 when is_uint8), rows row_stride elements
 * apart, read as value / data_range.  what bit 0: SSIM over the ROI (roi = device (x, y, w, h) clipped to the image,
 * NULL = whole image) with skimage's defaults as the reference calls structural_similarity: 7x7 uniform window,
 * sample covariance, K1 = 0.01, K2 = 0.03, map cropped by 3 pixels, mean of the channel means; a ROI narrower or
 * shorter than 7 gives NaN.  what bit 1: PSNR over the whole image, -10 log10 of the per-pixel channel-mean squared
 * error averaged over the pixels with psnr_mask != 0 (psnr_mask [height, width] or NULL = all; needs
 * row_stride == 3 * width).  out[4] (device): SSIM, PSNR, summed squared error, pixel count; what is not computed is
 * NaN.  workspace: hrf_image_metrics_workspace_bytes(height, width) bytes; results are bitwise reproducible.
 * ---------------------------------------------------------------------------------------- */
int hrf_mask_bbox(const uint8_t* mask /* [height, width] */, int height, int width, int32_t* box /* [4] */, void* stream);
int64_t hrf_image_metrics_workspace_bytes(int height, int width);
int hrf_image_metrics(const void* im1, const void* im2, int is_uint8, int height, int width, int64_t row_stride,
                      const int32_t* roi, float data_range, const uint8_t* psnr_mask, int what, double* out,
                      void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------
 * Self tests (used by tests/ only): one 128xN x K tcgen05 MMA with caller-chosen descriptor
 * fields, to pin the shared-memory descriptor encoding on real hardware.
 * ---------------------------------------------------------------------------------------- */
int hrf_selftest_umma(const void* a_bf16 /* [M,K] row-major */, const void* b_bf16 /* [N,K] row-major */,
                      float* d /* [M,N] */, int m /* 64 or 128 */, int n, int k,
                      /* physical placement of the 8x8 core matrices in shared memory (bytes) */
                      uint32_t a_kstride, uint32_t a_mstride, uint32_t b_kstride, uint32_t b_nstride,
                      /* descriptor fields (bytes) */
                      uint32_t a_lbo, uint32_t a_sbo, uint32_t b_lbo, uint32_t b_sbo,
                      int mn_major /* bit 0: A is MN-major, bit 1: B is MN-major */, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HUMANRF_B200_H_ */
