/*
 * b2f.h -- C ABI of libb200forest.so, the B200-native scoring engine behind the
 * credit-default service's `model.predict()`.
 *
 * The reference has no native code and therefore no FFI of its own: its hot path is the
 * Python call `ml_models["credit_default"].predict(input_df)` (reference app/main.py:72), which
 * lands in `CustomModel.predict` (reference databricks/src/02-register-model.ipynb:330-353) and
 * from there in scikit-learn.  This header is the boundary a maintainer of the reference binds
 * with ctypes to replace that arithmetic (see INTEGRATION.md for the stub).  Each entry point
 * names the reference call it replaces.
 *
 * Conventions
 *   - plain C, no C++/torch types; all sizes explicit; little-endian host.
 *   - functions returning int: 0 = success, negative = error (B2F_E*); the message for the
 *     calling thread is available from b2f_last_error().
 *   - the caller owns every host buffer; the library owns device memory and CUDA streams.
 *   - one b2f_model per GPU; calls on one handle must be serialised by the caller
 *     (different handles may be driven from different threads concurrently).
 *   - there is NO CPU fallback: without a usable CUDA device every compute call fails.
 *
 * Row layout ("encoded row", what the host-side encoder produces from a LoanApplicant,
 * reference app/model.py:8-34): B2F_ROW_WORDS = 24 little-endian 32-bit words = 96 bytes,
 *   words 0 .. n_cat-1        int32   category code = index into the model's sorted vocabulary
 *                                     of that feature, -1 = unknown or missing
 *                                     (== OneHotEncoder(handle_unknown="ignore") all-zero block,
 *                                     reference 01-train-model.ipynb:200-206)
 *   words n_cat .. n_cat+n_num-1  float32 numeric feature (float64 -> float32 round-to-nearest,
 *                                     as sklearn's predict does); NaN = missing, imputed on the
 *                                     GPU with the training median (01-train-model.ipynb:212)
 *   remaining words           ignored (padding to 96 B so a row is six 16-byte vectors)
 * For the credit-default schema n_cat = 9, n_num = 14, in LoanApplicant field order.
 */
#ifndef B2F_H
#define B2F_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2F_ROW_WORDS 24
#define B2F_ROW_BYTES 96
#define B2F_PACKED_ROW_BYTES 64
#define B2F_MAX_TREES 1024
#define B2F_MOMENT_WORDS 3 /* per feature: count, mean, M2 */

/* row formats (the *_ex entry points take one; the plain entry points use B2F_ROWS_WORDS24) */
#define B2F_ROWS_WORDS24 0  /* 24 x 32-bit words, 96 B (layout above) */
#define B2F_ROWS_PACKED64 1 /* 16 x 32-bit words, 64 B: words 0..1 = nine 7-bit fields (category code + 1, 0 = unknown /
                               missing), little-endian bit order, field j at bit 7j; words 2..15 = the 14 float32 numerics.
                               One third fewer bytes over PCIe; needs exactly 9 categoricals of <= 126 categories and <= 14 numerics (the credit-default shape). */

#define B2F_ROWS_RANKED 2   /* per-model "ranked" rows (csrc/forest_rank.h): the categorical fields bit-packed in the first 4 or 8 bytes
                               (code + 1, 0 = unknown / missing), then one uint16 per numeric feature = the RANK of the value among the
                               forest's distinct split values of that feature (missing -> the rank of the imputation value), zero
                               padded to a multiple of 8 bytes: 32 bytes per row for the credit-default schema.  Exact by construction
                               (a forest only compares a value with its own split values) and scored by the integer-compare kernel
                               k_forest_predict_rank.  Available when b2f_rank_info.ok; rows come from b2f_encoder_encode (after
                               b2f_encoder_attach_ranker) or b2f_ranker_rank_rows. */

/* error codes */
#define B2F_OK 0
#define B2F_EINVAL (-1)  /* bad argument / malformed forest blob */
#define B2F_ECUDA (-2)   /* CUDA runtime error (message has the cudaError string) */
#define B2F_ENODEV (-3)  /* no usable CUDA device */
#define B2F_ENOMEM (-4)  /* host or device allocation failed */
#define B2F_ENCCL (-5)   /* NCCL error or NCCL library not loadable */
#define B2F_ESTATE (-6)  /* call not valid in this state (e.g. communicator not initialised) */
#define B2F_ERANGE (-7)  /* a numeric input is infinite or overflows float32 (sklearn raises ValueError there) */
#define B2F_EIRREGULAR (-8) /* b2f_json_parser_parse: the body is outside the fast path's grammar; use the general validator */

/* aggregation modes stored in the forest blob */
#define B2F_AGG_RF_MEAN 0       /* RandomForestClassifier.predict_proba: mean of leaf class fractions */
#define B2F_AGG_GBDT_LOGISTIC 1 /* binary GradientBoosting: expit(init + sum lr*leaf) */
#define B2F_AGG_IFOREST 2       /* IsolationForest: score = 2^(-sum path length / (n_trees * c(max_samples))) + offset_,
                                   flag = score > threshold (alibi-detect IForest: score = -decision_function) */

/* walk modes chosen at model creation */
#define B2F_WALK_SMEM 0   /* whole forest resident in shared memory (TMA bulk copy per CTA) */
#define B2F_WALK_GLOBAL 1 /* forest walked from global memory / L2 (too large for shared memory) */

typedef struct b2f_model b2f_model;
typedef uint64_t b2f_ticket;

/* one scored row, for b2f_predict_pairs: both results of a row side by side, so a chunk comes back in
 * ONE device-to-host copy instead of two */
typedef struct b2f_scored {
    float proba1;  /* P(class 1) */
    int32_t label; /* hard class label */
} b2f_scored;

/* one fully scored row, for b2f_predict_full: classifier and outlier detector evaluated on the same encoded row */
typedef struct b2f_scored_full {
    double proba1;       /* P(class 1), float64 as sklearn returns it */
    int32_t label;       /* hard class label */
    int32_t is_outlier;  /* outlier_score > threshold */
    float outlier_score; /* isolation-forest score (alibi-detect `instance_score`) */
    int32_t reserved;
} b2f_scored_full;

typedef struct b2f_info {
    int32_t device;
    int32_t sm_count;
    int32_t agg_mode;
    int32_t walk_mode;
    int32_t n_trees;
    int32_t n_groups;
    int32_t max_depth;
    int32_t n_cat;
    int32_t n_num;
    int32_t smem_bytes;     /* dynamic shared memory per CTA of the predict kernel */
    int32_t block_threads;  /* threads per CTA of the predict kernel */
    int32_t rows_per_warp;  /* rows walked concurrently by one warp */
    int64_t forest_bytes;   /* bytes of the node + leaf arrays on the device */
    int64_t launches;       /* kernels launched by this handle so far (predict + moments) */
    int64_t launches_tile;  /* ... of which the large-batch tile kernel */
    int64_t tile_min_rows;  /* launches of at least this many rows take the tile kernel (if tile_ok) */
    int32_t tile_ok;        /* the forest's trees fit the tile kernel's shared-memory ring */
    int32_t tile_resident;  /* ... and the whole forest stays resident in it (no streaming) */
    int32_t packed_ok;      /* B2F_ROWS_PACKED64 is accepted for this model */
    int32_t tile_warps;     /* consumer warps per CTA of the tile kernel (16..24) */
    int64_t launches_split; /* ... of which the small-batch (groups-across-warps) kernel */
    int64_t split_max_rows; /* launches of at most this many rows take it */
    int32_t outlier_trees;  /* trees of the attached outlier forest (0 = none attached) */
    int32_t rank_ok;        /* B2F_ROWS_RANKED is accepted (k_forest_predict_rank: forest resident in its rank layout) */
    int64_t launches_rank;  /* ... of which the rank kernel */
    int32_t rank_smem_bytes; /* dynamic shared memory per CTA of the rank kernel */
    int32_t rank_row_bytes;  /* bytes per ranked row */
    int32_t rank_stream;     /* the rank layout streams through shared memory piece by piece (too large to stay resident) */
    int32_t rank_last_pdl;   /* the last rank launch went out with programmatic dependent launch (0: its rows overlapped what a
                                rank launch of the current programmatic chain on its stream writes, or B2F_NO_PDL is set).  "Last" holds for one calling thread: the scorer's workers launch concurrently
                                on the model's slot streams, like the launch counters above this field is not synchronised */
} b2f_info;

/* ---- library / device ------------------------------------------------------------------ */
const char *b2f_version(void);
const char *b2f_last_error(void);
int b2f_device_count(void); /* number of CUDA devices, or B2F_ENODEV */

/* ---- model lifetime: replaces mlflow.pyfunc.load_model(...) in lifespan (app/main.py:20-31)
 *      for the classifier part (CustomModel.load_context, 02-register-model.ipynb:317-328) ---- */
/* structural check of a forest blob (header, group table, every node word keeps the walk in bounds);
 * needs no GPU.  b2f_model_create() runs the same check. */
int b2f_blob_validate(const void *forest_blob, size_t nbytes);
b2f_model *b2f_model_create(const void *forest_blob, size_t nbytes, int device); /* NULL on error */
void b2f_model_destroy(b2f_model *m);
int b2f_model_info(const b2f_model *m, b2f_info *out);

/* ---- ranked rows (no GPU involved): the forest's split-value tables and the row layout built from a forest blob -----------
 * Replaces nothing in the reference by itself; it is the exact re-encoding that lets `x <= threshold` (sklearn's float32-vs-float64
 * compare behind 02-register-model.ipynb:335-337) run as a 16-bit integer compare on the GPU. */
typedef struct b2f_rank_info {
    int32_t ok;            /* 1: the forest has a rank layout and B2F_ROWS_RANKED is accepted */
    int32_t row_bytes;     /* bytes per ranked row (multiple of 8) */
    int32_t cat_bytes;     /* 4 or 8: size of the categorical block at the start of a row */
    int32_t n_cat, n_num;
    int32_t depth;         /* depth every tree is padded to */
    int32_t n_trees;
    int32_t layout_bytes;  /* bytes of the rank layout of the forest (shared-memory resident in the kernel) */
    int32_t cat_shift[16]; /* bit position of categorical field j inside the block */
    int32_t cat_bits[16];  /* its width */
    int32_t n_thresholds[24]; /* per numeric feature: number of distinct split values */
    int32_t n_pairs;       /* (categorical feature, category) pairs some node tests: pseudo-features n_num .. n_num + n_pairs - 1 */
    uint32_t pairs[128];   /* feature << 16 | category code, ascending */
    char why[160];         /* when !ok: the reason */
} b2f_rank_info;
typedef struct b2f_ranker b2f_ranker;
b2f_ranker *b2f_ranker_create(const void *forest_blob, size_t nbytes); /* NULL on a malformed blob; check b2f_rank_info.ok */
void b2f_ranker_destroy(b2f_ranker *r);
int b2f_ranker_info(const b2f_ranker *r, b2f_rank_info *out);
const float *b2f_ranker_thresholds(const b2f_ranker *r, int k, int32_t *count); /* sorted distinct split values of numeric k */
const void *b2f_ranker_layout(const b2f_ranker *r, int64_t *nbytes);            /* the rank layout (what the kernel walks) */
/* encoded rows (B2F_ROWS_WORDS24 or B2F_ROWS_PACKED64) -> ranked rows, multi-threaded */
int b2f_ranker_rank_rows(const b2f_ranker *r, const void *rows, int64_t n, int row_format, void *ranked_out, int threads);
int b2f_model_rank_info(const b2f_model *m, b2f_rank_info *out);

/* ---- native host-side row encoder (no GPU involved): columnar request data -> encoded rows -----------------
 * Replaces the pandas / sklearn lookup work in front of the arithmetic (reference app/main.py:54,
 * databricks/src/01-train-model.ipynb:197-221).  Categorical columns come as Arrow string arrays, numeric columns as
 * float64 arrays; rows are written (multi-threaded) straight into the caller's, normally pinned, staging buffer. */
typedef struct b2f_str_column {
    const void *offsets;     /* Arrow offsets buffer: int32[n+1] or int64[n+1] */
    const uint8_t *data;     /* Arrow UTF-8 data buffer */
    const uint8_t *validity; /* Arrow validity bitmap (bit set = present), or NULL when there are no nulls */
    int64_t offset;          /* logical offset of the array inside its buffers (Arrow slice) */
    int64_t data_bytes;      /* size of the data buffer in bytes */
    int32_t offsets_are_64;  /* 1: large_string (int64 offsets), 0: string (int32 offsets) */
    int32_t reserved;
} b2f_str_column;
typedef struct b2f_encoder b2f_encoder;
/* vocabularies concatenated feature by feature: entry s spans vocab_bytes[vocab_offsets[s] .. vocab_offsets[s+1]);
 * null_codes[j] = code a null entry of feature j gets (the imputer's constant category if fit saw one), or -1 */
b2f_encoder *b2f_encoder_create(int n_cat, int n_num, const int32_t *vocab_counts, const char *vocab_bytes,
                                const int64_t *vocab_offsets, const int32_t *null_codes);
void b2f_encoder_destroy(b2f_encoder *e);
/* num_cols[k] + i * num_strides[k] addresses row i of numeric column k (strides in elements).
 * Returns B2F_ERANGE if a value is infinite / overflows float32 (rows_out is then unspecified). */
/* give the encoder the forest's split-value tables (copied): b2f_encoder_encode then accepts B2F_ROWS_RANKED */
int b2f_encoder_attach_ranker(b2f_encoder *e, const b2f_ranker *r);
/* category codes only, column-major (codes_out[j * n + i]): -1 = not in the vocabulary, nulls take the feature's null code.
 * The drift detector (b2f_drift_score) takes its categorical columns in this form. */
int b2f_encoder_codes(const b2f_encoder *e, int64_t n, const b2f_str_column *cat_cols, int32_t *codes_out, int threads);
int b2f_encoder_encode(const b2f_encoder *e, int64_t n, const b2f_str_column *cat_cols, const double *const *num_cols,
                       const int64_t *num_strides, int row_format, void *rows_out, int threads);

/* ---- native request-body parser (no GPU involved): request BYTES -> the 23 columns in one pass -----------------
 * Replaces json.loads + one LoanApplicant object per row + pd.DataFrame(rows) (reference app/main.py:42-54,
 * app/model.py:8-34) for requests of the regular shape: a JSON array of objects whose keys are feature names,
 * categorical values plain strings (printable ASCII, no escapes), numeric values plain JSON numbers.  Anything else
 * (unknown / repeated keys, escapes, null, true, numbers in strings, malformed JSON ...) returns B2F_EIRREGULAR and the
 * caller hands the same bytes to the general validator, which applies the reference's coercions and 422 rules.
 * names: n_cat categorical then n_num numeric feature names, concatenated (name f = names[name_offsets[f] ..
 * name_offsets[f+1])); defaults: what an absent key takes (app/model.py:12-34). */
typedef struct b2f_json_parser b2f_json_parser;
b2f_json_parser *b2f_json_parser_create(int n_cat, int n_num, const char *names, const int32_t *name_offsets,
                                        const char *default_strs, const int32_t *default_str_offsets,
                                        const double *default_nums); /* NULL on a bad argument */
void b2f_json_parser_destroy(b2f_json_parser *p);
/* number of rows (>= 0), B2F_EIRREGULAR, or B2F_EINVAL; the column buffers below stay valid until the next parse */
int64_t b2f_json_parser_parse(b2f_json_parser *p, const char *body, int64_t len);
const double *b2f_json_parser_numeric(const b2f_json_parser *p, int k);        /* n_rows float64 of numeric feature k */
const int32_t *b2f_json_parser_str_offsets(const b2f_json_parser *p, int j);   /* n_rows + 1 Arrow offsets of categorical j */
const uint8_t *b2f_json_parser_str_data(const b2f_json_parser *p, int j, int64_t *nbytes); /* its UTF-8 bytes */

/* ---- pinned host memory for request batches (the batching ring lives in these) ------------- */
void *b2f_pinned_alloc(size_t nbytes); /* NULL on error */
void b2f_pinned_free(void *p);

/* page-locked memory whose pages sit on the NUMA node of GPU `device` (allocated and first touched from a thread bound to that
 * node's CPUs; the node comes from /sys/bus/pci/devices/<bdf>/numa_node).  Host-to-device copies then leave from memory local to
 * the GPU's PCIe root instead of crossing the socket interconnect.  Falls back to b2f_pinned_alloc's placement when the topology
 * is not exposed.  Free with b2f_pinned_free. */
void *b2f_pinned_alloc_near(int device, size_t nbytes);

/* one page-locked buffer for a stream dealt round-robin over several GPUs (b2f_predict_stream): stripe s (bytes
 * [s * stripe_bytes, (s + 1) * stripe_bytes)) is placed on the NUMA node of models[s mod n_models]'s GPU.  Free with
 * b2f_pinned_free_striped. */
void *b2f_pinned_alloc_striped(b2f_model **models, int n_models, size_t stripe_bytes, size_t total_bytes);
void b2f_pinned_free_striped(void *p);

/* ---- columnar request pipeline: replaces everything between `pd.DataFrame(data)` and `.tolist()` around the classifier call
 *      (app/main.py:54-72, 02-register-model.ipynb:330-337) for one request: the columns of the DataFrame go in (same column
 *      description as b2f_encoder_encode), the request is cut into chunks, and each chunk is encoded by a pool of host threads
 *      (bound to the GPU's NUMA node) straight into pinned staging, copied, scored and copied back while the next chunk is being
 *      encoded; results are collected chunk by chunk so the caller can build its output list while the tail is in flight. */
typedef struct b2f_scorer b2f_scorer;
b2f_scorer *b2f_scorer_create(b2f_model *m, const b2f_encoder *e, int threads /* 0 = b2f_host_threads_default(the model's device) */);
/* the default size of a scorer's thread pool: three quarters of the CPUs of the GPU's NUMA node, at most 48, and at most the
 * cgroup's CPU bandwidth minus two (b2f_host_cpu_limit: cpu.max quota / period, 0.0 when unlimited) -- polling workers beyond
 * the quota get the whole container throttled */
/* timeline of the last job, for tuning: out[2c], out[2c+1] = microseconds from b2f_scorer_start to "chunk c encoded" and to
 * "chunk c's H2D / kernel / D2H enqueued"; returns the number of chunks written (<= max_chunks) */
int b2f_scorer_trace(const b2f_scorer *s, double *out, int max_chunks);
int b2f_host_threads_default(int device);
double b2f_host_cpu_limit(void);
/* bind the calling thread (and the threads it creates later) to the CPUs of the GPU's NUMA node; returns the CPU count, 0 = unchanged.
 * A one-GPU serving process calls it before it builds request data: column buffers, response objects and staging then share a socket */
int b2f_bind_caller_near(int device);
/* NUMA node of a GPU (-1: not exposed) and the number of logical CPUs of that node this process may use */
int b2f_device_numa_node(int device, int *n_cpus);
void b2f_scorer_destroy(b2f_scorer *s);
/* out_mode: 0 = float proba1, 1 = double proba1, 3 = b2f_scored_full records (attached outlier forest; float32 row formats only).
 * chunk_rows 0 = choose.  Returns the number of chunks (>= 0) or a negative error; one job at a time per scorer; the column
 * buffers must stay valid until the last chunk has been waited for. */
int b2f_scorer_start(b2f_scorer *s, int64_t n, const b2f_str_column *cat_cols, const double *const *num_cols, const int64_t *num_strides,
                     int row_format, int out_mode, int64_t chunk_rows);
int b2f_scorer_wait(b2f_scorer *s, int chunk);       /* chunk `chunk` (rows b2f_scorer_chunk_range) is in the result buffer */
const void *b2f_scorer_results(const b2f_scorer *s); /* pinned result buffer of the current job: n x {float | double | b2f_scored_full} */
int64_t b2f_scorer_chunk_rows(const b2f_scorer *s); /* nominal rows per chunk (every chunk, when chunk_rows was given to b2f_scorer_start) */
/* the rows of chunk c (chunks are equal except the last; B200_FIRST_CHUNK_ROWS=<r> gives a library-chunked request a first
 * chunk of r rows) */
int b2f_scorer_chunk_range(const b2f_scorer *s, int c, int64_t *lo, int64_t *cnt);
int b2f_scorer_threads(const b2f_scorer *s);

/* ---- scoring: replaces classifier.predict_proba(df[all_features])[:, 1]
 *      (02-register-model.ipynb:335-337) and pipeline.predict (01-train-model.ipynb:290) --------
 * rows:   n encoded rows in HOST memory (pinned memory makes the copies asynchronous).
 * proba1: P(class 1) per row;  label: hard class label per row (sklearn tie rule: 1 iff p1 > p0,
 *         GBDT: raw >= 0).  Either output pointer may be NULL.
 * Copies host->device, runs the fused impute -> one-hot-as-equality -> tree-walk -> aggregate kernel
 * and copies the results back, pipelined over internal streams; returns when outputs are written. */
int b2f_predict(b2f_model *m, const void *rows, int64_t n, float *proba1, int32_t *label);
int b2f_predict_f64(b2f_model *m, const void *rows, int64_t n, double *proba1, int32_t *label);

/* same, with an explicit row format and output type */
int b2f_predict_ex(b2f_model *m, const void *rows, int64_t n, int row_format, void *proba1,
                   int proba_is_f64, int32_t *label);

/* both outputs interleaved per row (one D2H copy per pipelined chunk) */
int b2f_predict_pairs(b2f_model *m, const void *rows, int64_t n, int row_format, b2f_scored *out);

/* ---- classifier + outlier detector in one pass: replaces, on top of the above,
 *      `self.outliers.predict(df[numeric_features].values)` (02-register-model.ipynb:339,344; detector built at
 *      :232-233 as alibi-detect IForest = sklearn IsolationForest, score = -decision_function, flag = score > threshold).
 * The outlier forest is a second forest blob (agg_mode B2F_AGG_IFOREST) over the SAME encoded rows (its splits
 * test the numeric row words); attach it once, then b2f_predict_full copies each chunk of rows to the GPU once,
 * runs the classifier kernel and the isolation-forest kernel back to back on it and returns one 24-byte record
 * per row in ONE device-to-host copy.  A forest blob with agg_mode B2F_AGG_IFOREST is also a valid model on its
 * own (b2f_model_create): every predict entry point then returns (score, flag) in place of (proba1, label). */
int b2f_model_attach_outlier_forest(b2f_model *m, const void *forest_blob, size_t nbytes);
int b2f_predict_full(b2f_model *m, const void *rows, int64_t n, int row_format, b2f_scored_full *out);

/* asynchronous form for the request-batching ring: buffers must be pinned and stay valid until
 * b2f_wait(ticket) returns.  proba_is_f64 selects double (1) or float (0) outputs. */
int b2f_predict_async(b2f_model *m, const void *rows_pinned, int64_t n, void *proba1_pinned,
                      int proba_is_f64, int32_t *label_pinned, b2f_ticket *ticket);
/* proba_is_f64: 0 = float, 1 = double, 2 = proba1_pinned points at b2f_scored records (label_pinned ignored),
 * 3 = proba1_pinned points at b2f_scored_full records (needs an attached outlier forest) */
int b2f_predict_async_ex(b2f_model *m, const void *rows_pinned, int64_t n, int row_format,
                         void *proba1_pinned, int proba_is_f64, int32_t *label_pinned,
                         b2f_ticket *ticket);
int b2f_wait(b2f_model *m, b2f_ticket ticket);

/* one call over several GPUs: contiguous slices of the batch go round-robin to the models
 * (one per device); no inter-GPU traffic (rows are independent). */
int b2f_predict_multi(b2f_model **models, int n_models, const void *rows, int64_t n, void *proba1,
                      int proba_is_f64, int32_t *label);

/* proba_is_f64 as for b2f_predict_async_ex (2 / 3: proba1 points at b2f_scored / b2f_scored_full records) */
int b2f_predict_multi_ex(b2f_model **models, int n_models, const void *rows, int64_t n, int row_format,
                         void *proba1, int proba_is_f64, int32_t *label);

/* a long stream of rows in `batch`-row batches dealt round-robin: batch b -> models[b % n_models]; one host thread
 * per GPU inside the call, at most `inflight` (1..8) batches in flight per GPU; buffers should be pinned */
int b2f_predict_stream(b2f_model **models, int n_models, const void *rows, int64_t n, int64_t batch, int row_format,
                       void *proba1, int proba_is_f64, int32_t *label, int inflight);

/* ---- batch drift scores: replaces `self.drift.predict(df[self.all_features].values)` ---------------------------
 *      (02-register-model.ipynb:338; detector built at :224-229 as alibi-detect TabularDrift(x_ref, p_val=0.05,
 *      categories_per_feature={0..8: None}); the response carries 1 - p_val, :345-349).
 * Per feature of the request batch against the reference table: categorical -> chi-squared test on the 2 x K table of
 * category counts (scipy.stats.chi2_contingency), numeric -> two-sided two-sample Kolmogorov-Smirnov test with the
 * EXACT p-value (scipy.stats.ks_2samp(method="exact")).  The reference table stays in HBM (numeric columns sorted,
 * category counts); both the statistics and the exact lattice-path p-value recursion run on the GPU. */
typedef struct b2f_drift b2f_drift;
/* ref_sorted: n_num columns of n_ref float64 each, every column ascending (column-major);
 * cat_sizes[c]: number of distinct reference categories of categorical feature c; ref_counts: their counts, concatenated */
b2f_drift *b2f_drift_create(int device, int64_t n_ref, int n_num, const double *ref_sorted, int n_cat,
                            const int32_t *cat_sizes, const int64_t *ref_counts); /* NULL on error */
void b2f_drift_destroy(b2f_drift *d);
/* num_cols: n_num x n float64, column-major (column k at num_cols + k*n); cat_codes: n_cat x n int32, column-major,
 * code = index of the value among the feature's reference categories or -1 if it is not one of them.
 * Values that are not reference categories form extra columns of the contingency table (alibi-detect counts over the
 * union of reference and batch categories): new_offsets[n_cat + 1] / new_counts list their counts per feature
 * (both NULL when every batch value is a reference category).
 * Outputs, categorical features first then numeric ones: p_val (required), stat (chi-squared statistic / K-S D) and
 * flags (0 = ok; 1 = scipy itself switches to the asymptotic K-S formula there (lcm of the sample sizes >= 2^31): p_val is
 * kstwo.sf(D, round(m*n/(m+n))), computed by the library (b2f_kstwo_sf); 2 = NaN in the batch column: p_val is NaN) may be NULL.
 * device_ms (may be NULL): device time of the call (copies + kernels), from CUDA events. */
int b2f_drift_score(b2f_drift *d, int64_t n, const double *num_cols, const int32_t *cat_codes,
                    const int32_t *new_offsets, const int64_t *new_counts, double *p_val, double *stat,
                    int32_t *flags, float *device_ms);
int64_t b2f_drift_launches(const b2f_drift *d); /* kernels launched by this handle so far */
/* scipy.stats.kstwo.sf(x, n) for the sample sizes where ks_2samp leaves the exact method (host, scalar; b2f_drift_score applies
 * it itself to features it flags 1, so the p-values it returns are final) */
double b2f_kstwo_sf(double x, double n);

/* ---- device-resident interface (measurement and callers that already hold rows in HBM) ----- */
void *b2f_device_alloc(b2f_model *m, size_t nbytes);
void b2f_device_free(b2f_model *m, void *dptr);
int b2f_copy_h2d(b2f_model *m, void *dst_dev, const void *src_host, size_t nbytes);
int b2f_copy_d2h(b2f_model *m, void *dst_host, const void *src_dev, size_t nbytes);
/* enqueue one predict launch on the model's compute stream (asynchronous) */
int b2f_predict_device(b2f_model *m, const void *rows_dev, int64_t n, void *proba1_dev,
                       int proba_is_f64, int32_t *label_dev);
int b2f_predict_device_ex(b2f_model *m, const void *rows_dev, int64_t n, int row_format,
                          void *proba1_dev, int proba_is_f64, int32_t *label_dev);
int b2f_sync(b2f_model *m);
/* run `iters` launches back to back, each bracketed by CUDA events on the launching stream;
 * ms_each[iters] receives each launch's device time.  flush_l2 != 0 writes a >L2-sized scratch
 * buffer before every launch (outside the event bracket). */
int b2f_predict_device_timed(b2f_model *m, const void *rows_dev, int64_t n, void *proba1_dev,
                             int proba_is_f64, int32_t *label_dev, int iters, int flush_l2,
                             float *ms_each);

/* streaming form: `steps` launches cycling over `pool` distinct device-resident batches of n rows
 * laid out back to back (rows, proba and label alike), so that successive launches read different
 * HBM lines; ms_each[steps] (may be NULL) per launch, *ms_total for the whole region. */
int b2f_predict_stream_timed(b2f_model *m, const void *rows_dev, int64_t n, int pool, void *proba1_dev,
                             int proba_is_f64, int32_t *label_dev, int steps, float *ms_each,
                             float *ms_total);

int b2f_predict_stream_timed_ex(b2f_model *m, const void *rows_dev, int64_t n, int row_format, int pool,
                                void *proba1_dev, int proba_is_f64, int32_t *label_dev, int steps,
                                float *ms_each, float *ms_total);

/* ---- drift-monitor moments (BASELINE config 5; nearest reference call is
 *      self.drift.predict(...), 02-register-model.ipynb:338 -- no mean/var exists there) --------
 * For each of the 24 row words f: out[3f+0] = count of non-NaN values, out[3f+1] = mean,
 * out[3f+2] = M2 = sum (x-mean)^2, all float64.  Category words are read as integers. */
int b2f_moments(b2f_model *m, const void *rows, int64_t n, double *out /* 24*3 */);
int b2f_moments_device(b2f_model *m, const void *rows_dev, int64_t n, double *out /* host, 24*3 */);
int b2f_moments_device_timed(b2f_model *m, const void *rows_dev, int64_t n, int iters, int flush_l2,
                             float *ms_each, double *out);
/* Chan merge of k partial (count, mean, M2) triples per word, on the host (used after an all-gather) */
void b2f_moments_merge(const double *parts /* k*24*3 */, int k, double *out /* 24*3 */);

/* ---- NCCL plumbing for the cross-GPU moments merge (552-byte all-gather per rank) ----------- */
int b2f_comm_unique_id(void *id_out128);                                  /* rank 0 creates */
int b2f_comm_init_rank(b2f_model *m, int nranks, int rank, const void *id128); /* one process per GPU */
int b2f_comm_init_all(b2f_model **models, int n_models);                  /* one process, many GPUs */
/* all-gather this rank's (count, mean, M2) triples over NVLink and Chan-merge them */
int b2f_moments_allgather(b2f_model *m, const double *local /* 24*3 */, double *merged /* 24*3 */);
/* single-process form: per-device moments of per-device row slices, merged across all models */
int b2f_moments_multi(b2f_model **models, int n_models, const void *rows, int64_t n, double *out);

#ifdef __cplusplus
}
#endif
#endif /* B2F_H */
