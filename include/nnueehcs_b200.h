/*
 * nnueehcs_b200 -- C ABI of the B200-native uncertainty-estimation hot path.
 *
 * The reference (cjlauer16/NNUEEHCS) is pure Python and has no FFI layer; the boundary this
 * library replaces is the body of three Python methods and two metric functions.  Each entry
 * point below names the reference interface it stands in for (paths relative to the reference
 * root).  All pointers are raw device (or, where stated, host) pointers, all sizes are plain
 * integers; no torch / C++ types cross this boundary.  INTEGRATION.md shows the ctypes binding
 * a maintainer of the reference would add.
 *
 * Threading / streams: every call enqueues work on the CUDA stream passed as `stream`
 * (a cudaStream_t cast to void*; NULL = legacy default stream) on the current device and
 * returns without synchronising unless stated otherwise.  Errors never abort(): a non-zero
 * status is returned and uq_last_error() (thread-local) describes it, so the Python side can
 * raise ValueError (UQ_ERR_INVALID / UQ_ERR_UNSUPPORTED) or RuntimeError (UQ_ERR_CUDA), the
 * two exception kinds the reference's callers handle (examples/bo_driven/bo.py:469-497).
 */
#ifndef NNUEEHCS_B200_H
#define NNUEEHCS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UQ_ABI_VERSION 3

/* status codes */
#define UQ_OK 0
#define UQ_ERR_INVALID 1     /* bad argument / configuration  -> ValueError   */
#define UQ_ERR_CUDA 2        /* CUDA runtime failure          -> RuntimeError */
#define UQ_ERR_UNSUPPORTED 3 /* shape/precision not built     -> ValueError   */
#define UQ_ERR_WORKSPACE 4   /* workspace too small           -> RuntimeError */

/* which wrapper's forward is being evaluated */
#define UQ_MODE_ENSEMBLE 0   /* EnsembleModel.forward      nnueehcs/models.py:99-108  */
#define UQ_MODE_MC_DROPOUT 1 /* MCDropoutModel.forward     nnueehcs/models.py:147-163 */
#define UQ_MODE_DELTA_UQ 2   /* DeltaUQMLP.forward         nnueehcs/models.py:313-341 */
#define UQ_MODE_PAGER 3      /* PAGERMLP._score_samples    nnueehcs/models.py:396-429: roles of
                                sample and anchor swapped, P[n][k] = net(cat(a_k - x_n, x_n));
                                out0 = mean_k P[n][k], out1 = max_k |P[n][k] - Y_k|, raised to
                                score_floor[n] when given (torch.maximum at models.py:389-390) */

/* arithmetic the MLP stack runs in */
#define UQ_PREC_FP32 0 /* the 1e-5 parity mode.  Runs on the tensor cores as a scaled fp16 x 2 split
                          (three tcgen05 kind::f16 MMAs per K step into fp32 TMEM accumulators,
                          per-product error <= 7e-7) when uq_model_supports_fp32_tc(), else as
                          UQ_PREC_FP32_FFMA                                                  */
#define UQ_PREC_BF16 1 /* tcgen05 bf16 x bf16 -> fp32 TMEM accumulators: the throughput mode */
#define UQ_PREC_FP32_FFMA 2 /* CUDA-core FFMA, fp32 accumulate, one grouped SGEMM per layer: any
                               layer shape; the cross-check of the two modes above           */

/* what uq_forward writes */
#define UQ_OUT_MEAN_STD 0 /* out0 = mean, out1 = unbiased std (what evaluation.py consumes)   */
#define UQ_OUT_MOMENTS 1  /* out0 = mean, out1 = M2, count returned in *out_count (K-shards) */

typedef struct uq_model uq_model_t; /* opaque: packed weights of K members */

/*
 * One Linear (+ optional eval-mode BatchNorm1d, ReLU, Dropout) block of the nn.Sequential that
 * nnueehcs/model_builder.py:30-73 (build_network) produces.  Device pointers, float32,
 * `weight` is [out_features, in_features] row-major exactly as torch stores nn.Linear.weight.
 * Null bn_* pointers mean "no BatchNorm after this Linear".
 */
typedef struct uq_layer_desc {
  int32_t in_features;
  int32_t out_features;
  const float* weight;
  const float* bias;      /* [out] or NULL */
  const float* bn_weight; /* gamma, [out] or NULL */
  const float* bn_bias;   /* beta */
  const float* bn_mean;   /* running_mean */
  const float* bn_var;    /* running_var */
  float bn_eps;
  int32_t relu;    /* 1: ReLU follows (after BN if present) */
  int32_t dropout; /* 1: an nn.Dropout follows this block's activation (MC dropout only) */
} uq_layer_desc;

typedef struct uq_forward_args {
  int32_t mode;         /* UQ_MODE_*  */
  int32_t precision;    /* UQ_PREC_*  */
  int32_t output;       /* UQ_OUT_*   */
  int32_t member_begin; /* K-axis shard: members / passes / anchors [begin, begin+count) */
  int32_t member_count; /*   of this call; full range = [0, K)                            */
  int32_t total_members; /* K of the whole job (Philox pass ids and anchors index by global id) */
  int32_t dropout_active; /* 0: "dropout-off" parity case (P identical passes) */
  int32_t row_base;     /* native Philox masks only: global index of x's first row, so that a rank
                           that runs a slice [row_base, row_base + n) of the samples draws the same
                           bits as the unsharded call (0 for a whole-batch call)              */
  double dropout_p;     /* MCDropoutModel.dropout_percent (models.py:132-134) */
  uint64_t philox_seed; /* native masks: Philox4x32-10 keyed by seed, counter =     */
  uint64_t philox_offset; /*   (global pass id, dropout layer, sample, feature group)  */
  const uint8_t* masks; /* injected keep-masks or NULL. Layout: for dropout layer l (in module
                           order) a block [total_members][n][width_l] of bytes (0/1), blocks
                           concatenated in layer order. */
  const float* anchors; /* Delta-UQ anchors [total_members][d_in] (d_in = net input / 2) */
  const float* anchor_targets; /* PAGER: anchors_Y [total_members][d_out] (models.py:440-449) */
  const float* score_floor;    /* PAGER: [n][d_out] or NULL -- the Delta-UQ std the conformal
                                  score is maximised with */
} uq_forward_args;

/* -- library ------------------------------------------------------------------------------ */
int uq_abi_version(void);
const char* uq_last_error(void);
/* number of kernels this library launched on this thread since the last reset (bench.py's
   gpu_launches) */
uint64_t uq_launch_count(void);
void uq_launch_count_reset(void);
/* diagnostics: microseconds the five phases (statistics, fine-bin pass, fold, grid evaluation,
   JS terms) of this thread's last single-launch uq_kde_jsd took on the current device */
int uq_kde_jsd_phase_us(double* out5);

/* -- model packing: replaces the weight walk the wrappers do implicitly through
      nn.Sequential.__call__ (models.py:103,156-158).  `layers` is
      [n_members][n_layers] (host array of descriptors holding device pointers).  The library
      copies/folds what it needs (fp32 weights + eval-BN scale/shift; bf16 UMMA-swizzled image
      with BN folded) into its own device buffers; the caller may free its tensors after the
      call's stream work has completed. */
int uq_model_create(uq_model_t** out, int32_t n_members, int32_t n_layers,
                    const uq_layer_desc* layers, void* stream);
/*    Same with flags.  UQ_MODEL_ANCHOR_FIRST: in UQ_MODE_DELTA_UQ / UQ_MODE_PAGER the network input
      of a sample x and an anchor a is cat([a, x - a]) -- the channel order of the public `deltauq`
      package (deltaUQ_MLP.create_anchored_batch: torch.cat([A, diff], axis=1)) that the reference
      subclasses (nnueehcs/models.py:288) -- instead of cat([x - a, a]) (flags = 0, what
      uq_model_create packs).  The two differ by a swap of the first Linear's column halves; a
      checkpoint trained with the reference stack needs the flag.  Other modes ignore it. */
#define UQ_MODEL_ANCHOR_FIRST 1
int uq_model_create_ex(uq_model_t** out, int32_t n_members, int32_t n_layers,
                       const uq_layer_desc* layers, int32_t flags, void* stream);
int uq_model_destroy(uq_model_t* model);
/* 1 if the bf16 tcgen05 path supports this model's shapes, else 0 (reason in uq_last_error) */
int uq_model_supports_bf16(const uq_model_t* model);
/* 1 if UQ_PREC_FP32 runs on the tensor cores for this model (equal hidden widths, multiple of 64,
   <= 512, at most 16 network inputs -- for UQ_MODE_DELTA_UQ / UQ_MODE_PAGER that is the doubled
   width, so at most 8 sample features), else 0 (reason in uq_last_error) and UQ_PREC_FP32 is the
   CUDA-core path */
int uq_model_supports_fp32_tc(const uq_model_t* model);

/* -- the forward: K x net(x) -> stack -> mean(0), std(0), fused.
      x: [n, d_in] float32 row-major on device.  out0/out1: [n, d_out] float32 on device.
      workspace: device scratch of at least uq_forward_workspace_bytes(...) bytes (may be NULL
      when that returns 0).  *out_count (host, may be NULL) receives member_count. */
size_t uq_forward_workspace_bytes(const uq_model_t* model, int64_t n, const uq_forward_args* args);
int uq_forward(const uq_model_t* model, const float* x, int64_t n, const uq_forward_args* args,
               float* out0, float* out1, void* workspace, size_t workspace_bytes,
               double* out_count, void* stream);

/* same call with HOST buffers (pinned or pageable): H2D of x, forward, D2H of both outputs,
   synchronises `stream` before returning.  This is the end-to-end path bench.py times. */
int uq_forward_host(const uq_model_t* model, const float* x_host, int64_t n,
                    const uq_forward_args* args, float* out0_host, float* out1_host,
                    void* stream);

/* -- K-axis shards: Chan merge of per-shard (count, mean, M2), then unbiased std.
      means/m2s: [n_shards][len] float32 device (e.g. the NCCL all-gather buffer),
      counts: host array [n_shards].  Writes mean/std [len]. */
int uq_moments_merge(const float* means, const float* m2s, const double* counts,
                     int32_t n_shards, int64_t len, float* out_mean, float* out_std,
                     void* stream);

/*    Same merge for shards that are not packed back to back: shard s has its means at
      means + s * shard_stride and its M2 at m2s + s * shard_stride (e.g. the receive buffer of the
      all-to-all in nnueehcs_b200/distributed.py, [shard][mean | M2][slice]).  Shards with count 0
      are skipped.  output = UQ_OUT_MEAN_STD writes (mean, unbiased std), UQ_OUT_MOMENTS (mean, M2). */
int uq_moments_merge_ex(const float* means, const float* m2s, int64_t shard_stride,
                        const double* counts, int32_t n_shards, int64_t len, float* out_mean,
                        float* out_second, int32_t output, void* stream);

/* -- native dropout masks: writes the Philox keep-masks uq_forward would draw for dropout layer
      `dropout_layer` as bytes [total_members][n][width] (the injected-mask layout), so a
      native-RNG MC-dropout run can be replayed bit-for-bit through the CPU oracle. */
int uq_philox_keep_masks(uint8_t* out, int64_t n, int32_t width, int32_t total_members,
                         int32_t dropout_layer, double dropout_p, uint64_t seed, uint64_t offset,
                         void* stream);

/* -- metrics -------------------------------------------------------------------------------
      uq_wasserstein_1d replaces scipy.stats.wasserstein_distance as called from
      WassersteinEvaluation._evaluate_uncertainties (nnueehcs/evaluation.py:182).
      u, v: float32 device arrays; result (float64) written to *out_host after the call
      synchronises `stream`.  workspace from uq_wasserstein_workspace_bytes. */
size_t uq_wasserstein_workspace_bytes(int64_t nu, int64_t nv);
int uq_wasserstein_1d(const float* u, int64_t nu, const float* v, int64_t nv, double* out_host,
                      void* workspace, size_t workspace_bytes, void* stream);

/*    Same integral with the method spelled out (uq_wasserstein_1d = UQ_WASSERSTEIN_AUTO):
      BINNED reads each sample once, resolves every key bin on which F_u - F_v keeps one sign from
      the bin's (count, integer offset sum) alone and sorts only the values of the other bins;
      SORT radix-sorts both samples (scipy's own route); AUTO = BINNED unless more than half of
      the values sit in ambiguous bins or a value is inf/NaN.  info_host (may be NULL) receives
      {method used, u values sorted, v values sorted}. */
#define UQ_WASSERSTEIN_AUTO 0
#define UQ_WASSERSTEIN_SORT 1
#define UQ_WASSERSTEIN_BINNED 2
int uq_wasserstein_1d_ex(const float* u, int64_t nu, const float* v, int64_t nv, int32_t method,
                         double* out_host, int64_t* info_host, void* workspace,
                         size_t workspace_bytes, void* stream);

/*    Enqueue / finish forms of the two distribution metrics: the same results without a stream
      synchronisation inside the call, so that a caller that needs several metrics of the same
      score vectors (the reference's evaluate() loop over its metric list,
      nnueehcs/evaluation.py:122-144) pays ONE synchronisation for all of them.
      enqueue: the single-launch method's memset + kernel on `stream`; `record` is caller-owned
      MAPPED PINNED host memory of UQ_METRIC_RECORD_BYTES (cudaHostAlloc / torch pin_memory) that
      the kernel's last block fills in.  The inputs must stay untouched until finish; the
      workspace may be handed to further enqueue calls on the SAME stream (each call zeroes what
      it needs, in stream order).  finish (after the caller has synchronised `stream`): reads the
      record; where the single-launch method does not apply (ambiguous bins, inf / NaN, a range
      beyond ~4000 bandwidths) it runs the synchronous call from scratch. */
#define UQ_METRIC_RECORD_BYTES 256
int uq_wasserstein_1d_enqueue(const float* u, int64_t nu, const float* v, int64_t nv, void* record,
                              void* workspace, size_t workspace_bytes, void* stream);
int uq_wasserstein_1d_finish(const float* u, int64_t nu, const float* v, int64_t nv,
                             const void* record, double* out_host, int64_t* info_host,
                             void* workspace, size_t workspace_bytes, void* stream);
int uq_kde_jsd_enqueue(const float* u, int64_t nu, const float* v, int64_t nv, int32_t grid_pts,
                       void* record, void* workspace, size_t workspace_bytes, void* stream);
int uq_kde_jsd_finish(const float* u, int64_t nu, const float* v, int64_t nv, int32_t grid_pts,
                      const void* record, double* out_host, int32_t* method_used, void* workspace,
                      size_t workspace_bytes, void* stream);

/*    uq_kde_jsd replaces JensenShannonEvaluation.pdf_jsd (nnueehcs/evaluation.py:268-276):
      Scott-bandwidth Gaussian KDE of each sample on a shared `grid_pts`-point linspace between
      the joint min and max, then the Jensen-Shannon distance of the two pdf vectors. */
size_t uq_kde_jsd_workspace_bytes(int64_t nu, int64_t nv, int32_t grid_pts);
int uq_kde_jsd(const float* u, int64_t nu, const float* v, int64_t nv, int32_t grid_pts,
               double* out_host, void* workspace, size_t workspace_bytes, void* stream);
/*    Same with the method spelled out (uq_kde_jsd = UQ_KDE_AUTO).  WINDOW: the samples are
      sorted and every chunk adds exp() terms to the grid points within 9 bandwidths (every term of
      scipy's sum above 3e-18 of the peak).  MOMENTS: bins of width h/4, six moments per bin from one
      pass over the sample, Hermite series on the grid -- independent of N x grid work, JS distance
      within 1e-9 relative of WINDOW; needs (max - min) / (h/4) <= 8192.  AUTO = MOMENTS when it
      applies.  *method_used (host, may be NULL) receives what ran. */
#define UQ_KDE_AUTO 0
#define UQ_KDE_WINDOW 1
#define UQ_KDE_MOMENTS 2
int uq_kde_jsd_ex(const float* u, int64_t nu, const float* v, int64_t nv, int32_t grid_pts,
                  int32_t method, double* out_host, int32_t* method_used, void* workspace,
                  size_t workspace_bytes, void* stream);

/*    The ascending sort underneath the SORT method, uq_score_metrics and the WINDOW KDE, on its
      own: what np.sort does inside scipy's _cdf_distance (behind nnueehcs/evaluation.py:182) and
      np.percentile (evaluation.py:292-381).  Stable 4-pass LSD radix sort of the float32 bit
      patterns (-0.0 before +0.0; every NaN last, as np.sort puts them, returned as 0x7FFFFFFF).  x, out: [n] float32 device,
      16-byte aligned, out == x allowed; asynchronous on `stream`. */
size_t uq_sort_workspace_bytes(int64_t n);
int uq_sort_f32(const float* x, int64_t n, float* out, void* workspace, size_t workspace_bytes,
                void* stream);

/* -- score consumers (SURVEY.md section 8f row 1): the rest of what nnueehcs/evaluation.py derives
      from the two score vectors, from one pair of device sorts.  Replaces MeanScoreEvaluation /
      MaxScoreEvaluation / PercentileScoreEvaluation (evaluation.py:292-381, numpy on the host),
      TNRatTPX._evaluate_scores (:538-580, a Python loop over every unique score), AUROC (:614-624,
      sklearn on the host) and PercentileBasedClassifier (:637-662 over classification.py:103-143,
      torch.quantile + four counts).  id / ood: float32 device arrays. ------------------------ */
typedef struct uq_score_request {
  double percentile_q;          /* PercentileScoreEvaluation.percentile, in [0, 100]        */
  double target_tpr;            /* TNRatTPX.target_tpr, in [0, 1]                            */
  double classifier_percentile; /* PercentileBasedIdOodClassifier.percentile, in [0, 1]      */
  int32_t tnr_reversed;         /* TNRatTPX.reversed                                         */
  int32_t classifier_reversed;  /* PercentileBasedClassifier.reversed (scores negated first) */
} uq_score_request;
typedef struct uq_score_result {
  double mean_score, max_score, percentile_score; /* of the ID scores */
  double auroc;                                   /* OOD = positive class */
  double tnr_at_tpr;
  double sensitivity, specificity, fpr, fnr;
} uq_score_result;
size_t uq_score_metrics_workspace_bytes(int64_t n_id, int64_t n_ood);
int uq_score_metrics(const float* id_scores, int64_t n_id, const float* ood_scores, int64_t n_ood,
                     const uq_score_request* req, uq_score_result* out_host, void* workspace,
                     size_t workspace_bytes, void* stream);

/* -- sharded metrics (one process per GPU; SURVEY.md section 8e).  The reference is
      single-process scipy (nnueehcs/evaluation.py:182, :268-276) and has no counterpart; these are
      the per-rank steps that nnueehcs_b200/distributed.py strings together with one all-reduce /
      all-to-all each. ------------------------------------------------------------------------ */

/*    (min, max, mean, M2 = sum (x - mean)^2) of one shard, float64, written to out_host[4] after
      synchronising `stream`.  Shards are merged on the host with Chan's formula. */
size_t uq_sample_stats_workspace_bytes(void);
int uq_sample_stats(const float* x, int64_t n, double* out_host, void* workspace,
                    size_t workspace_bytes, void* stream);

/*    Adds one shard's Gaussian kernel sums to `grid` (float64 [grid_pts], device, accumulated in
      place) for the grid linspace(lo, hi, grid_pts) and the given kernel bandwidth (both global
      quantities).  All-reduce the grids of the two samples, then uq_jsd_from_grids. */
size_t uq_kde_grid_workspace_bytes(int64_t n);
int uq_kde_grid_accumulate(const float* x, int64_t n, double lo, double hi, double bandwidth,
                           int32_t grid_pts, double* grid, void* workspace,
                           size_t workspace_bytes, void* stream);
/*    scipy.spatial.distance.jensenshannon of two raw kernel-sum vectors, grids = [2][grid_pts]
      float64 on device; result to *out_host after synchronising `stream`. */
int uq_jsd_from_grids(const double* grids, int32_t grid_pts, double* out_host, void* stream);

/*    Histogram of the values over uq_key_bins() order-preserving coarse key bins (added to
      `hist`, uint32 [bins], device): all-reduced to choose balanced value-range splitters. */
int32_t uq_key_bins(void);
int uq_key_histogram(const float* x, int64_t n, uint32_t* hist, void* stream);
/*    Scatter a shard into per-destination segments: value with key bin b goes to part
      bin_to_part[b] (uint8 [bins], device).  cursors (uint64 [n_parts], device) hold each
      segment's start offset in `out` on entry and its end offset on return. */
int uq_partition_by_bin(const float* x, int64_t n, const uint8_t* bin_to_part, int32_t n_parts,
                        float* out, unsigned long long* cursors, void* stream);
/*    One value range of the sample-sorted Wasserstein: every u and v value of this rank's range,
      with u_below / v_below values of each sample in lower ranges.  out_host[3] = {integral of
      |F_u - F_v| over the local merged values, first merged value, last merged value}.  Workspace
      as uq_wasserstein_workspace_bytes(max(nu,1), max(nv,1)). */
int uq_wasserstein_1d_range(const float* u, int64_t nu, const float* v, int64_t nv,
                            int64_t u_below, int64_t v_below, int64_t nu_total, int64_t nv_total,
                            double* out_host, void* workspace, size_t workspace_bytes,
                            void* stream);


/*    uq_kde_density replaces the input-density score of KDEMLPModel.forward
      (nnueehcs/models.py:209-222): -exp(KernelDensity(bandwidth, kernel='gaussian')
      .fit(fit).score_samples(x)) -- the negated d-dimensional Gaussian KDE of the `m` fitted rows
      at each of the `n` query rows.  fit: [m][d], x: [n][d] float32 row-major on device;
      bandwidth: sklearn's bandwidth_ (for 'scott': m^(-1/(d+4)), uq_kde_scott_bandwidth);
      out: [n] float64 on device (the reference returns a float64 tensor).  Asynchronous. */
double uq_kde_scott_bandwidth(int64_t m, int32_t d);
/*    sklearn's other named rule, bandwidth='silverman' (the reference's KDE search space offers
      both, examples/bo_driven/config_kde.yaml:385-390): (m (d + 2) / 4)^(-1/(d+4)). */
double uq_kde_silverman_bandwidth(int64_t m, int32_t d);
size_t uq_kde_density_workspace_bytes(int64_t n, int64_t m);
int uq_kde_density(const float* fit, int64_t m, const float* x, int64_t n, int32_t d,
                   double bandwidth, double* out, void* workspace, size_t workspace_bytes,
                   void* stream);

/*    Per-rank steps of the sharded BINNED Wasserstein (no counterpart in the reference).
      uq_bin_moments ADDS one shard to the caller-zeroed tables cnt / ksum (uint64 [uq_key_bins()]
      each, device): values per key bin and the sum of their low 18 key bits.  The four tables
      [cnt_u | ksum_u | cnt_v | ksum_v] are all-reduced over the ranks (one collective), then
      uq_wasserstein_from_bins writes out_host[4] = {integral over the bins on which F_u - F_v
      keeps one sign, ambiguous u values, ambiguous v values, values in inf/NaN bins} and
      flags_out[bin] = 1 for ambiguous bins (uint8 [bins], device).  If values are ambiguous,
      uq_compact_flagged collects a shard's ambiguous values (out: n floats of room; *count_host =
      how many), the ranks all-gather them, and uq_wasserstein_ambiguous integrates those bins
      exactly; the distance is the sum of the two parts.  Workspaces:
      uq_wasserstein_workspace_bytes(1, 1) for from_bins / compact_flagged,
      uq_wasserstein_workspace_bytes(max(nu_amb,1), max(nv_amb,1)) for ambiguous. */
int uq_bin_moments(const float* x, int64_t n, uint64_t* cnt, uint64_t* ksum, void* stream);
int uq_wasserstein_from_bins(const uint64_t* tables, int64_t nu_total, int64_t nv_total,
                             uint8_t* flags_out, double* out_host, void* workspace,
                             size_t workspace_bytes, void* stream);
int uq_compact_flagged(const float* x, int64_t n, const uint8_t* flags, float* out,
                       int64_t* count_host, void* workspace, size_t workspace_bytes,
                       void* stream);
int uq_wasserstein_ambiguous(const float* u_amb, int64_t nu_amb, const float* v_amb,
                             int64_t nv_amb, const uint64_t* tables, int64_t nu_total,
                             int64_t nv_total, double* out_host, void* workspace,
                             size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NNUEEHCS_B200_H */
