/*
 * mdf_b200.h — C ABI of the B200-native structure-branch hot path of Metagenomic-DeepFRI.
 *
 * Every entry point is what a reference-side FFI binding for this path would bind
 * (INTEGRATION.md shows the ctypes stubs).  Plain pointers and sizes only; no torch / CUDA
 * types in the signatures (streams and device buffers travel as void*).  All functions return
 * 0 on success or a negative MDF_E* code; `mdf_last_error()` returns a thread-local message.
 * No exceptions cross the ABI.  The caller owns every buffer it passes in.
 *
 * Conventions
 *   - "host" pointers may be pageable or pinned; copies are asynchronous when pinned.
 *   - ragged batches use CSR-style int64 offset arrays of n+1 entries.
 *   - bit-packed contact maps: row i of an L x L map is `mdf_packed_row_words(L)` uint32
 *     words (rows padded to 128 bits), bit (j & 31) of word (j >> 5) = map[i][j].
 */
#ifndef MDF_B200_H
#define MDF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDF_OK            0
#define MDF_EINVAL       -1   /* bad argument (shape mismatch, invalid residue, ...) */
#define MDF_ECUDA        -2   /* CUDA runtime error (see mdf_last_error) */
#define MDF_ENOMEM       -3   /* workspace arena exhausted */
#define MDF_EUNSUPPORTED -4   /* model graph not supported by the fused pipeline */
#define MDF_ENOENT       -5   /* model / structure file cannot be opened */
#define MDF_EPARSE       -6   /* file is not what it should be (ONNX protobuf, coordinate cache ...) */

typedef struct mdf_ctx   mdf_ctx;    /* one per device: stream + workspace arena */
typedef struct mdf_model mdf_model;  /* one per loaded GCN head: weights resident in HBM */
typedef struct mdf_batch mdf_batch;  /* one uploaded batch of path inputs, resident in HBM */

const char *mdf_last_error(void);
int mdf_version(void);

/* ---- context --------------------------------------------------------------------------------
 * `arena`/`arena_bytes`: optional caller-provided device workspace (e.g. a torch uint8 tensor);
 * NULL lets the library cudaMalloc (and grow) its own.  `stream`: cudaStream_t as void*, NULL =
 * a private non-blocking stream. */
int mdf_ctx_create(int device, void *arena, size_t arena_bytes, void *stream, mdf_ctx **out);
int mdf_ctx_destroy(mdf_ctx *ctx);
int mdf_ctx_synchronize(mdf_ctx *ctx);
/* kernels launched by this context since creation (bench.py `gpu_launches`) */
int64_t mdf_ctx_launch_count(const mdf_ctx *ctx);

/* per-stage CUDA-event profiling: enable (clears old records), run, then fetch a text report with
 * one "name\tmilliseconds\tunits" line per recorded stage (units = algorithmic flops or bytes). */
int mdf_ctx_profile(mdf_ctx *ctx, int enable);
int mdf_ctx_profile_report(mdf_ctx *ctx, char *buf, size_t capacity);
/* also keep fp32 copies of the tensor-core engine's intermediates for mdf_batch_fetch (parity tests) */
int mdf_ctx_set_debug_taps(mdf_ctx *ctx, int enable);

static inline int mdf_packed_row_words(int L) { return ((L + 127) / 128) * 4; }

/* ---- contact_map_utils.pyx:17-37  pairwise_sqeuclidean(X, threads) ---------------------------
 * X host float32 [n, m] C-contiguous -> D host float32 [n, n].  Bit-exact (unfused fp32). */
int mdf_pairwise_sqeuclidean(mdf_ctx *ctx, const float *X, int n, int m, float *D);

/* ---- bio_utils.py:196-227  calculate_contact_map(coords, threshold, mode) --------------------
 * thr2 = float32(threshold**2) computed by the caller (NumPy weak-scalar rule); strict '<'.
 * matrix mode -> int32 [n, n]. */
int mdf_contact_map_dense(mdf_ctx *ctx, const float *coords, int n, float thr2, int32_t *cmap);
/* sparse mode (np.argwhere order).  Call with pairs == NULL to get *nnz, then with a buffer of
 * capacity >= *nnz pairs. */
int mdf_contact_map_sparse(mdf_ctx *ctx, const float *coords, int n, float thr2,
                           int32_t *pairs, int64_t capacity, int64_t *nnz);

/* ---- contact_map_utils.pyx:44-117  align_contact_map(q_aln, t_aln, sparse, gen, threads) -----
 * `sparse` host int32 [nnz, 2]; `out` host int32 [Lq, Lq] where Lq = non-gap query columns
 * (returned through *Lq_out; pass out == NULL to only query it). */
int mdf_align_contact_map(mdf_ctx *ctx, const char *q_aln, const char *t_aln, int aln_len,
                          const int32_t *sparse, int64_t nnz, int generated_contacts,
                          int32_t *out, int *Lq_out);

/* ---- bio_utils.py:348-385  build_align_contact_map x n (fused, batched) ----------------------
 * For protein p: coords rows [coord_off[p], coord_off[p+1]) of `coords` (float32 [*,3]);
 * alignment columns [aln_off[p], aln_off[p+1]) of q_aln / t_aln; output rows of Lq[p] =
 * seq_off[p+1]-seq_off[p] residues.  Exactly one of packed_out / dense_out may be non-NULL per
 * call: packed_out uint32 at word offset packed_off[p]; dense_out int32 [Lq,Lq] at element
 * offset dense_off[p].  Synchronous: runs as a job in the context's synchronous slot and waits for
 * it, so it works while two asynchronous jobs are in flight and leaves them undisturbed. */
int mdf_cmap_build_transfer(mdf_ctx *ctx, int n,
                            const float *coords, const int64_t *coord_off,
                            const char *q_aln, const char *t_aln, const int64_t *aln_off,
                            const int64_t *seq_off, float thr2, int generated_contacts,
                            uint32_t *packed_out, const int64_t *packed_off,
                            int32_t *dense_out, const int64_t *dense_off);

/* The same for n alignments given as arrays of per-alignment pointers (what `pipeline.py:476-481` holds: one gapped query, one
 * gapped target and one [Lt,3] float32 array per hit).  The library counts the query lengths (characters of q_aln[p] other than
 * '-'), writes the canonical offsets seq_off_out[n+1] (residues) and packed_off_out[n+1] (uint32 words, row p: Lq *
 * mdf_packed_row_words(Lq)), packs the inputs into pinned staging memory on MDF_HOST_THREADS host threads and runs the fused
 * kernels.  packed_out == NULL: sizes only (host work, no GPU, ctx may be NULL) - call once to size the output, once to fill it;
 * packed_capacity_words < packed_off_out[n] is MDF_EINVAL.  packed_out may be pageable or pinned.  Synchronous, like
 * mdf_cmap_build_transfer. */
int mdf_cmap_build_transfer_ragged(mdf_ctx *ctx, int n,
                                   const float *const *coords, const int *coord_rows,
                                   const char *const *q_aln, const char *const *t_aln, const int *aln_len,
                                   float thr2, int generated_contacts,
                                   uint32_t *packed_out, size_t packed_capacity_words,
                                   int64_t *packed_off_out, int64_t *seq_off_out);

/* ---- predict.pyx:50-73  Predictor.__init__ / _load_model --------------------------------------
 * The host side parses the .onnx file and hands the initialisers over as fp32 host arrays in
 * ONNX layout. */
typedef struct mdf_model_desc {
    int n_channels;          /* 26 */
    int lstm_hidden;         /* H */
    int n_lstm;              /* stacked LSTM layers (2) */
    const float *lstm_W[4];  /* ONNX [1,4H,in]  gate order i,o,f,c */
    const float *lstm_R[4];  /* ONNX [1,4H,H] */
    const float *lstm_B[4];  /* ONNX [1,8H] or NULL */
    int lm_dim;              /* E */
    const float *aa_W;       /* [26,E] */
    const float *lm_W;       /* [H,E] */
    const float *lm_b;       /* [E] or NULL */
    int n_gc;                /* GraphConv layers (<= 8) */
    int gc_dims[8];
    const float *gc_W[8];    /* [in,out] */
    const float *gc_b[8];    /* [out] or NULL */
    int gc_activation;       /* 0 = linear, 1 = relu, 2 = elu */
    float gc_alpha;          /* elu alpha */
    float eps;               /* degree normalisation epsilon */
    int fc_dim;              /* F */
    const float *fc_W;       /* [sum(gc_dims),F] */
    const float *fc_b;       /* [F] or NULL */
    int n_terms;             /* C */
    const float *out_W;      /* [F,2C] */
    const float *out_b;      /* [2C] or NULL */
} mdf_model_desc;

int mdf_model_create(mdf_ctx *ctx, const mdf_model_desc *desc, mdf_model **out);
int mdf_model_destroy(mdf_model *model);

/* ---- predict.pyx:62-73  Predictor._load_model: straight from the `.onnx` file the reference hands to onnxruntime -----
 * The file is decoded (protobuf wire format, no library) and the graph RECOGNISED as a DeepFRI GCN head: weights are found by
 * dataflow role, hyper-parameters read from shapes / op types, and the adjacency-normalisation sub-graph is verified by
 * evaluating it on two small probe maps at load time (it must equal D (A - diag A + I) D, d = 1 / (eps + sqrt(rowsum))).
 * MDF_ENOENT: cannot open; MDF_EPARSE: not an ONNX protobuf; MDF_EUNSUPPORTED: not a graph the fused pipeline computes
 * (mdf_last_error says why).  There is no fallback executor. */
int mdf_model_load(mdf_ctx *ctx, const char *onnx_path, mdf_model **out);
/* head sizes of a loaded model; any out pointer may be NULL.  gc_dims: room for 8 ints */
int mdf_model_info(const mdf_model *model, int *n_terms, int *lstm_hidden, int *lm_dim, int *n_gc, int *gc_dims, int *fc_dim);
/* Host-only (no GPU needed): parse + recognise `onnx_path` and describe it as one JSON object in `buf`:
 * {"kind": "gcn" | "cnn", "input_names": [...], "n_terms": C, hyper-parameters ..., "roles": {role: initialiser name}}. */
int mdf_onnx_inspect(const char *onnx_path, char *buf, size_t capacity);
/* Host-only: the recognised weight playing `role` ("lstm1_W", "lm_W", "gc2_W", "fc_b", "out_W", "conv3_W", "scale", "shift" ...)
 * exactly as the pipeline will use it (Gemm transposes undone, conv bias + BatchNormalization folded).  buf == NULL only
 * reports *count (0 for an absent optional bias). */
int mdf_onnx_tensor(const char *onnx_path, const char *role, float *buf, int64_t capacity, int64_t *count);
/* 0 = fp32 SIMT reference engine, 1 = tcgen05 tensor-core engine */
int mdf_model_set_engine(mdf_model *model, int engine);
int mdf_model_get_engine(const mdf_model *model);

/* ---- predict.pyx:75-102  Predictor.forward_pass(seqres, cmap) ---------------------------------
 * seq: ASCII residues (alphabet "-DGULNTKHYWCPVSOIEFXQABZRM", anything else -> MDF_EINVAL);
 * cmap: host int32 [L, L] holding 0/1 (other values -> MDF_EINVAL); scores: host float32 [C].
 * A bad residue is reported before a bad map.  This and mdf_gcn_forward_packed are synchronous: each runs as a job in the
 * context's synchronous slot and waits for it, so they work while two asynchronous jobs are in flight and leave them undisturbed. */
int mdf_gcn_forward_dense(mdf_model *model, const char *seq, int L, const int32_t *cmap, float *scores);

/* batched GCN forward on bit-packed maps (host buffers): scores host float32 [n, C] */
int mdf_gcn_forward_packed(mdf_model *model, int n, const char *seq, const int64_t *seq_off,
                           const uint32_t *packed, const int64_t *packed_off, float *scores);

/* ---- the whole path: pipeline.py:476-481 + :301-319 for n proteins ----------------------------
 * coords + alignment + query sequence -> GO-term scores, everything in between stays in HBM.
 * `seq` must equal the gap-stripped query alignment.  Host buffers in, host scores out. */
int mdf_path_forward(mdf_model *model, int n,
                     const char *seq, const int64_t *seq_off,
                     const float *coords, const int64_t *coord_off,
                     const char *q_aln, const char *t_aln, const int64_t *aln_off,
                     float thr2, int generated_contacts, float *scores);

/* Asynchronous form: mdf_path_submit enqueues the host->device copies, every kernel and the device->host copy of the scores
 * and returns; mdf_path_wait blocks until `scores` is complete and reports device-side input errors.  Up to TWO jobs may be in
 * flight per context (each owns one of the context's two job slots): while job k computes, the inputs of job k + 1 are copied
 * into the other slot, so H2D / D2H and host-side packing overlap the kernels.  Flat input buffers and `scores` must stay valid
 * until mdf_path_wait returns (pinned memory makes the copies truly asynchronous).  mdf_path_forward == submit + wait. */
typedef struct mdf_job mdf_job;
int mdf_path_submit(mdf_model *model, int n,
                    const char *seq, const int64_t *seq_off,
                    const float *coords, const int64_t *coord_off,
                    const char *q_aln, const char *t_aln, const int64_t *aln_off,
                    float thr2, int generated_contacts, float *scores, mdf_job **job);
/* Ragged form: protein p is given by its own pointers - seq[p] (seq_len[p] residues, no gaps), coords[p] (float32
 * [coord_rows[p], 3]), q_aln[p] / t_aln[p] (aln_len[p] alignment columns each) - exactly what pipeline.py:476-481 holds per
 * alignment.  The library packs them into pinned staging memory on `MDF_HOST_THREADS` (default 4) host threads; the
 * caller's input buffers may be released as soon as the call returns. */
int mdf_path_submit_ragged(mdf_model *model, int n,
                           const char *const *seq, const int *seq_len,
                           const float *const *coords, const int *coord_rows,
                           const char *const *q_aln, const char *const *t_aln, const int *aln_len,
                           float thr2, int generated_contacts, float *scores, mdf_job **job);
/* Waits for a job of either kind - mdf_path_submit* or mdf_cnn_submit_ragged - until its outputs are on the host, and reports
 * device-side input errors (a residue outside the alphabet: "Invalid character in sequence"). */
int mdf_path_wait(mdf_job *job);
/* Alignment and prediction in one job: pair p is (query[p], target[p], coords[p]) - the GCN's query sequence (q_len[p] residues),
 * its best-hit target sequence (t_len[p]) and the target's C-alpha coordinates (float32 [coord_rows[p], 3]).  The pairs are
 * aligned on the device (global Needleman-Wunsch with affine gaps, exactly as mdf_nw_align: same matrix / alphabet / A <= 32 /
 * gap rules, same scores and alignment strings) and the traceback writes the query-frame coordinate table of the contact-map
 * stage directly - the result equals mdf_path_submit_ragged over the gapped strings insert_gaps (alignment.py:38-62) makes from
 * that alignment.  Per pair the job also returns the NW score, the alignment length and the number of M columns (identity =
 * n_match / aln_len); with `ops`, the alignment string of pair p at byte ops_off[p] (room for q_len[p] + t_len[p] columns),
 * ops_len[p] columns.  A residue outside the matrix alphabet fails here, naming the pair; a query residue outside the GCN
 * alphabet is reported by mdf_path_wait.  Job slots, asynchrony and mdf_path_wait as mdf_path_submit_ragged; the per-pair
 * outputs are complete when mdf_path_wait returns. */
int mdf_path_submit_pairs(mdf_model *model, int n,
                          const char *const *query, const int *q_len, const char *const *target, const int *t_len,
                          const float *const *coords, const int *coord_rows,
                          const int8_t *matrix, const char *alphabet, int A, int gap_open, int gap_extend,
                          float thr2, int generated_contacts, float *scores,
                          int32_t *nw_score, int32_t *aln_len, int32_t *n_match,
                          char *ops, const int64_t *ops_off, int *ops_len, mdf_job **job);

/* Same path split into upload / run / fetch so that the compute can be timed with inputs
 * already resident in HBM (bench.py `value`). */
int mdf_batch_upload(mdf_ctx *ctx, int n,
                     const char *seq, const int64_t *seq_off,
                     const float *coords, const int64_t *coord_off,
                     const char *q_aln, const char *t_aln, const int64_t *aln_off,
                     mdf_batch **out);
/* Resident form of mdf_path_submit_pairs: query p = seq[seq_off[p] .. seq_off[p+1]), target p = target[target_off[p] ..
 * target_off[p+1]), coordinates p = rows coord_off[p] .. coord_off[p+1] of coords (float32 [*, 3]).  The pairs are aligned once,
 * here; mdf_path_run / mdf_path_run_shared / mdf_batch_fetch / mdf_batch_unpack_dense then work on the batch as on any other.
 * mdf_batch_fetch_alignment returns the per-pair outputs of the alignment (as mdf_path_submit_pairs; ops == NULL: none). */
int mdf_batch_upload_pairs(mdf_ctx *ctx, int n,
                           const char *seq, const int64_t *seq_off,
                           const char *target, const int64_t *target_off,
                           const float *coords, const int64_t *coord_off,
                           const int8_t *matrix, const char *alphabet, int A, int gap_open, int gap_extend,
                           mdf_batch **out);
int mdf_batch_fetch_alignment(mdf_batch *batch, int32_t *nw_score, int32_t *aln_len, int32_t *n_match,
                              char *ops, const int64_t *ops_off, int *ops_len);
int mdf_batch_destroy(mdf_batch *batch);
int mdf_path_run(mdf_model *model, mdf_batch *batch, float thr2, int generated_contacts);
/* mdf_path_run that keeps what an earlier run on this batch computed and this head shares: the contact maps and degrees
 * (same thr2 / generated_contacts / eps) and the LSTM-LM output (same LM weights).  pipeline.py:546-655 runs the MF / BP /
 * CC / EC heads one after the other over the same proteins; mdf_path_run itself always recomputes everything. */
int mdf_path_run_shared(mdf_model *model, mdf_batch *batch, float thr2, int generated_contacts);
/* forget what earlier runs left on this batch for mdf_path_run_shared (the next shared run recomputes maps and LM output) */
int mdf_batch_invalidate(mdf_batch *batch);
/* stage selector for profiling / unit parity: 1 = cmap only, 2 = + LSTM-LM, 3 = + GraphConv, 4 = all */
int mdf_path_run_stages(mdf_model *model, mdf_batch *batch, float thr2, int generated_contacts, int upto);
int mdf_batch_fetch_scores(mdf_model *model, mdf_batch *batch, float *scores /* host [n,C] */);
/* debugging / parity taps: copy an intermediate of the last run to the host.
 * what: 0 = packed cmaps (uint32 words, offsets as mdf_packed_row_words), 1 = degree vector d,
 * 2 = LSTM layer-1 output [T,H], 3 = LSTM layer-2 output [T,H], 4 = X0 [T,E],
 * 5 = pooled [n, sum(gc)], 6 = last GraphConv output [T, g].  fp32 unless noted. */
int mdf_batch_fetch(mdf_model *model, mdf_batch *batch, int what, void *dst, size_t dst_bytes);

/* Reference-layout output of the contact-map stage of the last run: dense int32 [Lq, Lq] per protein (bio_utils.py:348-385),
 * protein p at element offset sum_{q<p} Lq^2 of `dense_device` (DEVICE memory; NULL = workspace scratch, for timing the
 * HBM-bound variant of K1/K2).  *cells_out = total cells. */
int mdf_batch_unpack_dense(mdf_batch *batch, int32_t *dense_device, int64_t *cells_out);

/* device pointer of the scores of the last mdf_path_run ([n, C] float32) */
const float *mdf_batch_scores_device(const mdf_batch *batch);

/* ---- predict.pyx:91-95  Predictor.forward_pass(seqres, cmap=None): the sequence-only DeepCNN branch ----
 * (models `DeepCNN-MERGED_*.onnx`, mDeepFRI/__init__.py:68; used for every query without a structure hit,
 * pipeline.py:600-620 / :638-648).  Graph: parallel Conv1D layers over the one-hot sequence ('same' padding) ->
 * concat -> BatchNormalization -> ReLU -> global max-pool over residues -> FuncPredictor dense -> softmax.
 * The host side folds conv bias + BatchNormalization into one scale / shift per channel. */
#define MDF_MAX_CONV 32
typedef struct mdf_cnn_desc {
    int n_channels;                     /* 26 */
    int n_conv;                         /* parallel Conv1D layers (<= MDF_MAX_CONV) */
    int conv_width[MDF_MAX_CONV];       /* kernel sizes (<= 128) */
    int conv_filters[MDF_MAX_CONV];     /* filters per layer (multiples of 128) */
    int conv_pad_left[MDF_MAX_CONV];    /* zero residues before position 0 (TF 'same': (w - 1) / 2) */
    const float *conv_W[MDF_MAX_CONV];  /* ONNX Conv layout [filters, 26, width] */
    const float *scale;                 /* [sum filters] y = conv * scale + shift, then ReLU */
    const float *shift;                 /* [sum filters] */
    int n_terms;                        /* C */
    const float *out_W;                 /* [sum filters, 2C] */
    const float *out_b;                 /* [2C] or NULL */
} mdf_cnn_desc;
typedef struct mdf_cnn_model mdf_cnn_model;

int mdf_cnn_model_create(mdf_ctx *ctx, const mdf_cnn_desc *desc, mdf_cnn_model **out);
int mdf_cnn_model_destroy(mdf_cnn_model *model);
/* same from a single-input `DeepCNN-*.onnx` file (conv bias + BatchNormalization folded into scale / shift while loading) */
int mdf_cnn_model_load(mdf_ctx *ctx, const char *onnx_path, mdf_cnn_model **out);
/* n sequences (ASCII residues, CSR offsets; every sequence needs >= 1 residue) -> scores host float32 [n, C].  Synchronous:
 * runs as a job in the context's synchronous slot and waits for it, so it works while two asynchronous jobs are in flight and
 * leaves them undisturbed.  It does not touch the resident batch of mdf_cnn_upload: mdf_cnn_fetch after it returns the last
 * mdf_cnn_run's results, not this call's. */
int mdf_cnn_forward(mdf_cnn_model *model, int n, const char *seq, const int64_t *seq_off, float *scores);
/* same with the sequences already resident: upload once, run many times (bench `value`), fetch */
int mdf_cnn_upload(mdf_cnn_model *model, int n, const char *seq, const int64_t *seq_off);
int mdf_cnn_run(mdf_cnn_model *model);
int mdf_cnn_fetch(mdf_cnn_model *model, float *scores /* host [n, C] */, float *pooled /* host [n, sum filters] or NULL */);
/* Asynchronous mdf_cnn_forward from per-sequence pointers (pipeline.py:607-613 holds one str per unaligned query).  Takes one of
 * the context's two asynchronous job slots - the same slots mdf_path_submit* use, so CNN and GCN jobs may be in flight
 * together - packs the sequences into the slot's pinned block on MDF_HOST_THREADS threads, enqueues H2D, encode, conv, head
 * and the D2H of the scores, and returns; mdf_path_wait completes the job.  Every sequence needs >= 1 residue (MDF_EINVAL here, naming the index);
 * a residue outside the alphabet is reported by mdf_path_wait ("Invalid character in sequence").  The caller's strings may be
 * released when the call returns; `scores` (host float32 [n, C]) must stay valid until mdf_path_wait returns. */
int mdf_cnn_submit_ragged(mdf_cnn_model *model, int n, const char *const *seq, const int *seq_len, float *scores, mdf_job **job);

/* ---- pdb.py:130-162 extract_calpha_coords / bio_utils.py:230-302 extract_residues_coordinates: coordinate ingest (host only) ----
 * C-alpha coordinates of one PDB text with biotite's selection as the reference applies it: first model, ATOM records (HETATM =
 * hetero, excluded), chain `chain`, atom name "CA", first alternate location per residue.  coords float32 [capacity, 3];
 * residues (one-letter, ProteinSequence alphabet; a name outside it -> MDF_EINVAL "non-standard residue XXX") and resnames3
 * (3 chars per atom, not terminated) may be NULL.  All three NULL: only count (*n_out).  A structure without the chain ->
 * MDF_EINVAL "Chain A not found in structure." (bio_utils.py:243-244). */
int mdf_pdb_calpha(const char *text, size_t len, char chain, float *coords, char *residues, char *resnames3, int capacity, int *n_out);
/* n texts on `threads` host threads.  rows[p] = C-alpha count (-1: chain not found, no rows); coords = flat float32
 * [sum rows, 3] (NULL: only count into rows / *total_rows). */
int mdf_pdb_calpha_batch(int n, const char *const *texts, const int64_t *lens, char chain, int threads, int *rows, float *coords,
                         int64_t capacity_rows, int64_t *total_rows);

/* C-alpha cache: one mmap-able file per structure database (ids, float32 [L, 3] blocks, id hash table), written once.
 * Lookups return pointers INTO the mapping (valid until close) - the (pointer, rows) arrays mdf_path_submit_ragged takes. */
typedef struct mdf_coords_cache mdf_coords_cache;
int mdf_coords_cache_create(const char *path, int64_t n, const char *const *ids, const int *rows, const float *const *coords);
int mdf_coords_cache_open(const char *path, mdf_coords_cache **out);
int mdf_coords_cache_close(mdf_coords_cache *cache);
int64_t mdf_coords_cache_size(const mdf_coords_cache *cache);
/* unknown id -> coords_out[p] = NULL, rows_out[p] = -1; *missing (may be NULL) = how many */
int mdf_coords_cache_lookup(const mdf_coords_cache *cache, int64_t n, const char *const *ids, const float **coords_out, int *rows_out,
                            int64_t *missing);
int mdf_coords_cache_entry(const mdf_coords_cache *cache, int64_t index, char *id_buf, size_t capacity, int *rows);

/* ---- alignment.py:163-221  best_hit_database / align_pairwise: batched global alignment (NW, affine gaps) on the GPU --------
 * What the reference asks of PyOpal: pyopal.Aligner(scoring_matrix, gap_open, gap_extend).align(query, db, algorithm="nw",
 * mode="full" | "score").  query[p] / target[p]: q_len[p] / t_len[p] letters of `alphabet` (anything else -> MDF_EINVAL);
 * matrix: A x A int8 row-major in the order of `alphabet`, A <= 32 (VTML80 by default in the reference: the caller passes the
 * values of scoring_matrices.ScoringMatrix.from_name(...)); a gap of length k costs gap_open + (k - 1) * gap_extend, end gaps
 * included.  scores[p] = optimal score.  ops != NULL: the alignment string of pair p over M (equal residues) / X (mismatch) /
 * I ('-' in the query) / D ('-' in the target) - the dialect mDeepFRI.alignment.insert_gaps reads - at ops + ops_off[p] (room
 * for q_len[p] + t_len[p] columns), ops_len[p] columns long, not terminated.  ops == NULL: scores only. */
int mdf_nw_align(mdf_ctx *ctx, int n, const char *const *query, const int *q_len, const char *const *target, const int *t_len,
                 const int8_t *matrix, const char *alphabet, int A, int gap_open, int gap_extend,
                 int32_t *scores, char *ops, const int64_t *ops_off, int *ops_len);

#ifdef __cplusplus
}
#endif
#endif /* MDF_B200_H */
