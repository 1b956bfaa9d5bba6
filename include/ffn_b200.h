/*
 * ffn_b200.h — C ABI of libffn_b200.so, the B200-native flood-filling inference engine.
 *
 * This is the boundary a maintainer of google/ffn binds (ctypes stub in INTEGRATION.md) to replace
 * the TensorFlow/JAX executor *and* the numpy flood-fill loop of the inference hot path.  Every
 * entry point names the reference interface it stands in for (paths relative to the reference
 * checkout).  Conventions:
 *
 *   - plain C types only; all coordinates/shapes are (z, y, x), arrays are C-order zyx;
 *   - the caller owns every host buffer, the engine owns every device buffer; handles are opaque;
 *   - every function returns 0 on success, non-zero on failure; ffn_last_error() (thread-local)
 *     describes the failure;
 *   - calls are synchronous; one in-flight call per engine (the Python host serialises);
 *   - there is NO CPU fallback: creation fails if no sm_100 device is usable.
 */
#ifndef FFN_B200_H_
#define FFN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct FfnEngine FfnEngine;
typedef struct FfnCanvas FfnCanvas;

/* Arithmetic of the 3x3x3 convolutions. */
enum {
  FFN_COMPUTE_FP16_TC = 0, /* fp16 operands, fp32 accumulate on tcgen05 tensor cores; fp32 residual stream */
  FFN_COMPUTE_FP32 = 1,    /* fp32 FMA on CUDA cores ("precise" parity mode) */
  FFN_COMPUTE_FP16X2_TC = 2 /* near-fp32 on the tensor cores: every operand split into fp16 hi + lo parts,
                             * a*w = a_hi*w_hi + a_lo*w_hi + a_hi*w_lo as three tcgen05 MMAs into the same fp32
                             * accumulator (weights pre-scaled by 2^10 so that w_lo stays normal) */
};

enum { FFN_IMAGE_U8 = 0, FFN_IMAGE_F32 = 1 };

enum { FFN_ARRAY_SEED = 0, FFN_ARRAY_SEGMENTATION = 1, FFN_ARRAY_QPROB = 2, FFN_ARRAY_IMAGE = 3 };

enum { FFN_MASK_MOVEMENT = 0, FFN_MASK_SEED = 1 };

/* Geometry of ConvStack3DFFNModel — ffn/training/models/convstack_3d.py:59-81 (fov_size, deltas,
 * depth, features) with ModelInfo's xyz triples (ffn/training/model.py:25-46) already reversed. */
typedef struct {
  int32_t fov_zyx[3];
  int32_t deltas_zyx[3];
  int32_t depth;    /* residual modules; 2*depth 3x3x3 convolutions + conv_lom */
  int32_t features; /* must be 32 */
} FfnModelDesc;

/* InferenceOptions (ffn/inference/inference.proto:131-168) after Canvas.__init__ converted the
 * probabilities to logits and stored them back as float32 (ffn/inference/inference.py:186-195),
 * plus the float64 movement-policy threshold of movement.get_policy_fn (movement.py:241-242). */
typedef struct {
  float init_activation;        /* logit */
  float pad_value;              /* logit */
  float move_threshold;         /* logit, float32 — Canvas.is_valid_pos / disco test */
  float segment_threshold;      /* logit */
  float disco_seed_threshold;   /* probability-space fraction; < 0 disables (inference.py:416) */
  double policy_score_threshold;/* FaceMaxMovementPolicy.score_threshold (float64 logit) */
  int32_t min_boundary_dist_zyx[3];
  int32_t min_segment_size;
} FfnOptions;

/* Result of one Canvas.segment_at (ffn/inference/inference.py:460-533). */
typedef struct {
  int64_t iters;            /* return value of segment_at */
  int32_t min_pos[3];       /* Canvas._min_pos */
  int32_t max_pos[3];       /* Canvas._max_pos */
  int32_t seed_got_too_weak;
  int32_t queue_len;        /* entries left in the movement-policy deque */
  int32_t finished;         /* 0 if max_steps was hit before the queue drained (call again to resume) */
  int32_t reserved;
} FfnSegStats;

/* storage.OriginInfo (ffn/inference/storage.py:35) per accepted segment. */
typedef struct {
  int32_t id;
  int32_t start_zyx[3];
  int64_t iters;
  double walltime_sec;
} FfnOrigin;

/* One (segment, overlapped id, voxel count) triple of Canvas.overlaps (inference.py:624-632,668). */
typedef struct {
  int32_t id;
  int32_t other_id;
  int64_t count;
} FfnOverlap;

/* Counters named as in ffn/inference/inference.py (counters['...']). */
typedef struct {
  int64_t inference_calls;      /* 'inference-calls' == FoV steps */
  int64_t segment_at_calls;     /* 'segment_at-loop-calls' */
  int64_t seeds_examined;       /* seeds that reached Canvas (after the border filter of seed.py:81-88) */
  int64_t skip_threshold;
  int64_t skip_invalid_pos;
  int64_t skip_restricted_pos;  /* 'skip_restriced_pos' (sic) */
  int64_t seed_got_too_weak;
  int64_t voxels_segmented;
  int64_t voxels_overlapping;
  int64_t invalid_weak;         /* segments rejected: weak seed */
  int64_t invalid_small;        /* segments rejected: too small */
  int64_t invalid_other;        /* segments rejected: num_iters <= 0 */
  int64_t segments;             /* accepted */
  int64_t max_id;               /* Canvas._max_id */
  double device_seconds;        /* sum of kernel time (CUDA events) of this call */
  int64_t kernel_launches;
} FfnCounters;

const char* ffn_last_error(void);

/* ---- engine: owns device context, packed weights, workspace ------------------------------
 * Replaces Runner._init_tf_model + Saver.restore (ffn/inference/runner.py:98-163).
 * weights_dhwio[i]: float32 [3,3,3,Cin,32] in TF DHWIO order for i < 2*depth (Cin = 2 for i == 0),
 * weights_dhwio[2*depth]: conv_lom [1,1,1,32,1]; biases[i]: [32] (conv_lom: [1]).
 * Geometry limits (an error, not a crash, when exceeded): every FoV size odd and >= 3; x extent <= 33 (the
 * operand staging of one tile must fit the 227 KB of shared memory: x = 35 needs 233 072 B); depth 1..16;
 * deltas in [0, fov // 2]; at most 10 tiles of 126 FoV rows per CTA (the fp32 residual stream of every tile lives
 * in TMEM), i.e. ceil(tiles / SMs) <= 10 — (65,65,33) has 1124 tiles and needs at least 113 SMs.  The more tiles
 * a CTA owns, the fewer chains fit (ffn_engine_set_chains): 10 / tiles-per-CTA, at most 4. */
int ffn_engine_create(int device, const FfnModelDesc* model, const float* const* weights_dhwio,
                      const float* const* biases, int compute_mode, FfnEngine** out);
/* Canvases created from the engine may outlive this call: the engine is then released by the last
 * ffn_canvas_destroy (until then those canvases stay fully usable). */
void ffn_engine_destroy(FfnEngine* engine);
int ffn_engine_set_compute_mode(FfnEngine* engine, int compute_mode);
/* Flood-fill chains time-multiplexed over the SMs by ONE persistent kernel (1..4; 0 = default 4): objects of a
 * canvas in flight at once in ffn_canvas_segment_all (committed in seed order — the results are those of the
 * sequential reference loop, inference.py:538-683, for any value), and patches of a batch sharing a round in
 * ffn_predict (the reference batches FoVs into one session.run, executor.py:266-340).  1 = strictly one
 * object / patch at a time. */
int ffn_engine_set_chains(FfnEngine* engine, int max_chains);
/* Number of SMs (CTAs of the cooperative grid) this engine's kernel occupies; 0 = all.  Several engines
 * with disjoint SM budgets (e.g. 3 x 49) driven from different host threads run their persistent kernels
 * CONCURRENTLY on one GPU: the B200 form of the reference's batching across canvases
 * (InferenceRequest.batch_size / concurrent_requests, doc/manual.md:89-97). */
int ffn_engine_set_grid(FfnEngine* engine, int num_ctas);
/* sm count, cooperative grid size, shared memory per CTA, tiles per FoV: info[0..3]. */
int ffn_engine_info(FfnEngine* engine, int64_t info[8]);

/* Device-side cycle counters of CTA 0 (out[0..15]) and the last CTA (out[16..31]): slot 0 grid-barrier
 * wait, 1 activation TMA wait, 2 weight wait, 3 UMMA issue, 4 epilogue wait-for-MMA, 5 epilogue body,
 * 6 stage, 7 paste, 8 leader, 9 steps, 10 kernel, 11 conv layers, 12-14 leader parts, 15 layer-end sync.
 * Off by default (reading the clock perturbs the critical CTA): ffn_engine_profile(e, NULL, 1) switches
 * the counters on, (e, NULL, 0) off; with out != NULL the counters are returned (and reset if reset). */
int ffn_engine_profile(FfnEngine* engine, int64_t out[32], int reset);
/* Tile timeline of one CTA (CTA 1) recorded while the counters are on: out[e * 2048 + i] = SM clock when event e
 * happened to that role's i-th tile since kernel start (0 producer saw the chain barrier, 1 copies issued, 2 UMMA
 * issuer saw the operands, 3 got an accumulator slot, 4 UMMAs issued, 5 epilogue saw the accumulators, 6 epilogue
 * done, 7 i-th barrier release by the signal warp); 0 = not recorded.  n <= 8 * 2048.  Debug / profiles only. */
int ffn_engine_trace(FfnEngine* engine, int64_t* out, int64_t n, int reset);

/* ---- L0 drop-in: ExecutorClient.predict (ffn/inference/executor.py:134-139, 266-340) -------
 * seed, image: host float32 [batch, Z, Y, X]; logits_out: host float32 [batch, Z, Y, X]
 * (the 'logits' fetch without the trailing channel axis).  Copies in, runs, copies out. */
int ffn_predict(FfnEngine* engine, const float* seed, const float* image, int batch,
                float* logits_out);

/* ---- canvas: HBM-resident state of ffn.inference.inference.Canvas (inference.py:129-310) ---
 * image: host [Z,Y,X] uint8 (normalised on the fly as (x - mean) / stddev in float32, exactly
 * runner.py:383-385) or float32 (already normalised; mean/stddev ignored). */
int ffn_canvas_create(FfnEngine* engine, const void* image, int image_dtype,
                      const int32_t shape_zyx[3], float image_mean, float image_stddev,
                      const FfnOptions* options, int keep_probability_maps, FfnCanvas** out);
void ffn_canvas_destroy(FfnCanvas* canvas);
/* MovementRestrictor.mask / .seed_mask (movement.py:290-314); mask: host uint8 [Z,Y,X] or NULL. */
int ffn_canvas_set_mask(FfnCanvas* canvas, int which, const uint8_t* mask);

/* Canvas.segment_at (inference.py:460-533).  reset == 1: init_seed + reset_state first
 * (partial_segment_iters == 0 path); reset == 2: reset_state only — the seed and the extents are kept
 * (Canvas.reset_seed_per_segment == False, inference.py:486-490); reset == 0 resumes the current object.  Runs at most
 * max_steps FoV steps (<= 0: unlimited) inside ONE persistent kernel launch per ~budget. */
int ffn_canvas_segment_at(FfnCanvas* canvas, const int32_t start_zyx[3], int reset,
                          int64_t max_steps, FfnSegStats* out);

/* Canvas.segment_all (inference.py:538-683) over an explicit seed list (the coords a seed policy
 * produced, seed.py:63-95).  origins_out / overlaps_out: caller arrays with the given capacities;
 * n_origins / n_overlaps receive the counts (ids are assigned as ++max_id in seed order). */
int ffn_canvas_segment_all(FfnCanvas* canvas, const int32_t* seeds_zyx, int64_t n_seeds,
                           FfnOrigin* origins_out, int64_t origins_cap, int64_t* n_origins,
                           FfnOverlap* overlaps_out, int64_t overlaps_cap, int64_t* n_overlaps,
                           FfnCounters* counters_out);

/* Canvas.update_at (inference.py:386-441): one FoV step at pos, no movement policy.
 * pred_out: host float32 [Z,Y,X] of the FoV (the merged logits pasted into the seed). */
int ffn_canvas_update_at(FfnCanvas* canvas, const int32_t pos_zyx[3], float* pred_out);

/* Canvas.init_seed (inference.py:443-450). */
int ffn_canvas_init_seed(FfnCanvas* canvas, const int32_t pos_zyx[3]);

/* Lazy views of Canvas.seed / .segmentation / .seg_prob (and the image as float32): copy a box. */
int ffn_canvas_read(FfnCanvas* canvas, int which, const int32_t lo_zyx[3],
                    const int32_t size_zyx[3], void* dst);
int ffn_canvas_write(FfnCanvas* canvas, int which, const int32_t lo_zyx[3],
                     const int32_t size_zyx[3], const void* src);

/* Movement-policy state for .cpoint compatibility (movement.py:180-184): deque entries as
 * (score, z, y, x) float64 quadruples, done-set as int32 lattice triples, start position. */
int ffn_canvas_policy_state_size(FfnCanvas* canvas, int64_t* queue_len, int64_t* done_len);
int ffn_canvas_policy_state_get(FfnCanvas* canvas, double* queue_szyx, int32_t* done_zyx,
                                int32_t start_zyx[3]);
int ffn_canvas_policy_state_set(FfnCanvas* canvas, const double* queue_szyx, int64_t queue_len,
                                const int32_t* done_zyx, int64_t done_len,
                                const int32_t start_zyx[3]);
/* Resume of an in-flight object restored from a .cpoint (Canvas.restore_checkpoint returning
 * partial_segment_iters > 0, inference.py:728-778): after ffn_canvas_policy_state_set and the
 * seed/segmentation writes, the next ffn_canvas_segment_all first finishes this object (with
 * the given iteration count and extents) and commits it, then continues with its seed list. */
int ffn_canvas_set_resume(FfnCanvas* canvas, int64_t iters, const int32_t min_pos[3],
                          const int32_t max_pos[3]);
/* Event log of the device loop (debugging, Canvas.history export).  Call with capacity > 0 and
 * events_out == NULL to (re)start logging, capacity == 0 to stop; call with events_out != NULL to
 * fetch: rows of (type, z, y, x), type 1 push, 2 pop valid, 3 pop invalid, 4 pop below threshold,
 * 5 pop already done, 6 FoV step, 7 seed invalid, 8 object start, 9 (count, 0, 0) = Canvas.history_deleted of the step just
 * executed (inference.py:420-422).  *n_events = events produced (may exceed capacity). */
int ffn_canvas_trace(FfnCanvas* canvas, int64_t capacity, int32_t* events_out, int64_t* n_events);
/* PolicyPeaks on the device (ffn/inference/seed.py:142-199): Sobel magnitude -> gaussian(sigma 49/6)
 * adaptive threshold -> exact Euclidean distance transform (anisotropy = voxel size) -> local maxima
 * (min_distance 3) with the tie-break noise `noise` (host float64 [Z,Y,X] = RandomState(42).rand, or
 * NULL).  Uses the canvas' resident image, segmentation and masks.  coords_out receives up to `cap`
 * (z, y, x) triples in arbitrary order (sort them for the policy); *n_out = number of peaks found. */
int ffn_canvas_seed_peaks(FfnCanvas* canvas, const float voxel_size_zyx[3], const double* noise,
                          int32_t* coords_out, int64_t cap, int64_t* n_out);
/* Canvas._max_id / counters carried across calls (checkpoint restore, init segmentation). */
int ffn_canvas_set_max_id(FfnCanvas* canvas, int64_t max_id);
int ffn_canvas_get_counters(FfnCanvas* canvas, FfnCounters* out);
/* Bookkeeping of the last ffn_canvas_segment_all: out[0] objects started ahead of their turn, out[1] of
 * those discarded (re-run in turn or rejected by the in-order gating), out[2] FoV steps of the discarded runs,
 * out[3] FoV steps executed in total (FfnCounters.inference_calls counts only what the reference counts),
 * out[4] rounds of the persistent kernel, out[5] / out[6] chain-rounds spent without an object / waiting for the
 * turn to commit, out[7] chains used. */
int ffn_canvas_spec_stats(FfnCanvas* canvas, int64_t out[8]);

/* Multi-GPU merge helpers (SURVEY.md 8e): raw device pointers for NCCL, and the HBM-bound
 * relabel kernel that adds a rank's ID offset to every label > 0. */
int ffn_canvas_device_ptr(FfnCanvas* canvas, int which, void** ptr, int64_t* bytes);
int ffn_canvas_add_id_offset(FfnCanvas* canvas, int32_t offset);

/* Self tests / micro-benchmarks of the sm_100a building blocks (results in out[]; see
 * ffn_b200/csrc/selftest.cuh).  Used by tests and profiles/, not by the product path. */
int ffn_selftest_umma(int device, int variant, double* out, int n_out);

#ifdef __cplusplus
}
#endif
#endif /* FFN_B200_H_ */
