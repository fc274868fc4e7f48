/*
 * rsb.h -- C-ABI of librsb (retrieval-scaling on B200): the drop-in boundary for the reference's
 * query -> top-k retrieval path.  Plain C types only: device pointers, sizes and a cudaStream_t passed
 * as void*.  No torch / C++ types cross this boundary.
 *
 * The reference (RulinShao/retrieval-scaling @ 9da3070) has no FFI of its own: its seam is the SWIG'd
 * `faiss` object protocol used by src/indicies/*.py.  Each entry point below names the reference call
 * site it replaces (paths relative to the reference root).  INTEGRATION.md shows the ctypes stub a
 * reference maintainer would add.
 *
 * Conventions
 *   - every function returns an int status: RSB_OK (0) or a negative RSB_ERR_* class; the message of the
 *     last error on the calling thread is available from rsb_last_error().  Nothing aborts the process and
 *     nothing falls back to the CPU.
 *   - all `*_dev` pointers are CUDA device pointers on the current device; they are owned by the caller.
 *     The library owns index storage behind the opaque handle (create/.../free).
 *   - work is enqueued on `stream`; results are valid after the stream is synchronised.  Functions that
 *     must read a size back (rsb_finalize) synchronise the stream themselves and say so.
 *   - search semantics are those of faiss 1.8.0 METRIC_INNER_PRODUCT indexes: scores float32, rows sorted
 *     by score descending, missing results padded with id -1 / score -FLT_MAX.
 */
#ifndef RSB_H_
#define RSB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSB_VERSION 100 /* 0.1.0 */

enum {
    RSB_OK = 0,
    RSB_ERR_INVALID = -1,     /* bad argument                         -> ValueError          */
    RSB_ERR_CUDA = -2,        /* CUDA runtime / launch failure        -> RuntimeError        */
    RSB_ERR_STATE = -3,       /* e.g. search before train             -> RuntimeError        */
    RSB_ERR_UNSUPPORTED = -4, /* e.g. nbits != 8                      -> NotImplementedError */
    RSB_ERR_OOM = -5          /* cudaMalloc failed / workspace small  -> MemoryError         */
};

enum { RSB_FLAT = 0, RSB_IVFFLAT = 1, RSB_IVFPQ = 2 };

typedef struct rsb_index rsb_index_t;
typedef void* rsb_stream_t; /* cudaStream_t */

int rsb_version(void);
const char* rsb_last_error(void);

/* ---- construction -------------------------------------------------------------------------------- */
/* faiss.IndexFlatIP(d)                                               <- src/indicies/flat.py:42        */
int rsb_flat_create(int d, rsb_index_t** out);
/* faiss.IndexIVFFlat(IndexFlatIP(d), d, nlist, METRIC_INNER_PRODUCT) <- src/indicies/ivf_flat.py:143-149 */
int rsb_ivfflat_create(int d, int nlist, rsb_index_t** out);
/* faiss.IndexIVFPQ(IndexFlatIP(d), d, nlist, M, nbits, METRIC_INNER_PRODUCT)
 *                                                                    <- src/indicies/ivf_pq.py:146-152
 * Sub-quantizer counts: M = 16, 32 or 64 run the tuned ADC scan (K = M/16 lanes of a warp cooperate on one vector with
 * a bank-conflict-free look-up layout that exists for K in {1, 2, 4}: csrc/rsb_layout.h); any other multiple of 4 up to
 * 128 dividing d (e.g. 24 / 48 / 96 on d = 768, which faiss and the reference's n_subquantizers key accept) runs a
 * functionally complete generic path (natural code order, [m][256] tables, one thread per vector) -- correct, not tuned.
 * RESTRICTION (narrower than faiss): nbits must be 8 (tables of 256 entries, one byte per code); nbits = 4 / 10 / 12 /
 * 16 and other M return RSB_ERR_UNSUPPORTED (-> NotImplementedError in Python). */
int rsb_ivfpq_create(int d, int nlist, int M, int nbits, rsb_index_t** out);
int rsb_free(rsb_index_t* h);

/* ---- trained state (what index.train() produces; ivf_flat.py:166, ivf_pq.py:170) ------------------ */
/* coarse centroids [nlist, d] float32, copied */
int rsb_set_centroids(rsb_index_t* h, const float* centroids_dev, rsb_stream_t stream);
/* PQ codebook [M, 256, d/M] float32, copied */
int rsb_set_pq_codebook(rsb_index_t* h, const float* codebook_dev, rsb_stream_t stream);
int rsb_get_centroids(rsb_index_t* h, float* out_dev, rsb_stream_t stream);
int rsb_get_pq_codebook(rsb_index_t* h, float* out_dev, rsb_stream_t stream);

/* ---- population (index.add(x): flat.py:58, ivf_flat.py:180, ivf_pq.py:185) ------------------------- */
/* ids_dev may be NULL: ids are then sequential from ntotal (faiss behaviour).  IVF: list = argmax_c <x,c>
 * computed here in fp32; IVFPQ additionally encodes the residual.  ws_dev/ws_bytes: see rsb_add_workspace_bytes. */
size_t rsb_add_workspace_bytes(rsb_index_t* h, int64_t n);
int rsb_add(rsb_index_t* h, const float* x_dev, int64_t n, const int64_t* ids_dev,
            void* ws_dev, size_t ws_bytes, rsb_stream_t stream);
/* as rsb_add but the coarse assignment is supplied by the caller (int32 list id per row) */
int rsb_add_preassigned(rsb_index_t* h, const float* x_dev, int64_t n, const int64_t* ids_dev,
                        const int32_t* list_dev, rsb_stream_t stream);
/* IVFPQ only: rows are already PQ codes [n, M] uint8 (e.g. read from an existing index file) */
int rsb_add_codes(rsb_index_t* h, const uint8_t* codes_dev, int64_t n, const int64_t* ids_dev,
                  const int32_t* list_dev, rsb_stream_t stream);
/* Build the searchable layout (CSR inverted lists; PQ codes interleaved per 32 vectors).  Synchronises
 * `stream`.  rsb_search calls it implicitly when adds are pending. */
int rsb_finalize(rsb_index_t* h, rsb_stream_t stream);

/* ---- introspection --------------------------------------------------------------------------------- */
enum {
    RSB_INFO_KIND = 0, RSB_INFO_D = 1, RSB_INFO_NLIST = 2, RSB_INFO_M = 3, RSB_INFO_NBITS = 4,
    RSB_INFO_NTOTAL = 5,       /* index.ntotal     */
    RSB_INFO_IS_TRAINED = 6,   /* index.is_trained */
    RSB_INFO_MAX_LIST_LEN = 7,
    RSB_INFO_INDEX_BYTES = 8   /* device bytes held by the searchable layout */
};
int rsb_info(rsb_index_t* h, int what, int64_t* out);
/* list sizes [nlist] int64 to a device buffer */
int rsb_list_sizes(rsb_index_t* h, int64_t* sizes_dev, rsb_stream_t stream);
/* Export the inverted lists in natural CSR order (insertion order inside each list), as the oracle and a
 * faiss file writer want them: offsets_dev [nlist+1] int64, payload_dev = uint8 codes [ntotal, M] (IVFPQ)
 * or float32 vectors [ntotal, d] (IVFFLAT / FLAT), ids_dev [ntotal] int64.  Any pointer may be NULL. */
int rsb_export_lists(rsb_index_t* h, int64_t* offsets_dev, void* payload_dev, int64_t* ids_dev,
                     rsb_stream_t stream);

/* ---- search (index.search(x, k) + index.nprobe: flat.py:139, ivf_flat.py:73,225, ivf_pq.py:76,230) --- */
size_t rsb_workspace_bytes(rsb_index_t* h, int nq, int k, int nprobe);
/* q_dev [nq, d] float32; D_dev [nq, k] float32; I_dev [nq, k] int64.  nprobe ignored for FLAT. */
int rsb_search(rsb_index_t* h, const float* q_dev, int nq, int k, int nprobe,
               float* D_dev, int64_t* I_dev, void* ws_dev, size_t ws_bytes, rsb_stream_t stream);
/* faiss IndexIVF::search_preassigned: as rsb_search, but the probed lists list_dev [nq, nprobe] int64 (-1 =
 * skip) and their coarse scores coarse_dis_dev [nq, nprobe] float32 (<q, c_list>, added to every PQ score of
 * that list; ignored by IVFFLAT) come from the caller instead of the coarse quantizer. */
int rsb_search_preassigned(rsb_index_t* h, const float* q_dev, int nq, int k, int nprobe,
                           const int64_t* list_dev, const float* coarse_dis_dev, float* D_dev, int64_t* I_dev,
                           void* ws_dev, size_t ws_bytes, rsb_stream_t stream);
/* Multi-GPU form of rsb_search_preassigned (one process per GPU, datastore partitioned across the GPUs; replaces the
 * reference's one-process-per-shard search, src/search.py:282-296): the per-query running top-k thresholds live in
 * caller-owned peer-mapped arrays.  tau_local_dev [nq] uint32 is THIS GPU's array; tau_peers_dev is a DEVICE array of
 * `npeers` base pointers, one per GPU of the job (the own entry is recognised and skipped).  Whenever the scan raises a
 * threshold it also raises it on every peer (relaxed system-scope max reduction over NVLink), so every GPU filters
 * with the best bound found anywhere; results are unchanged (a bound is always the k-th best score of real
 * candidates of that query).  The caller zeroes the arrays before the first search of a batch on ANY GPU and keeps
 * the GPUs within one batch of each other (a cross-GPU barrier per batch, which the top-k combine provides). */
int rsb_search_preassigned_shared(rsb_index_t* h, const float* q_dev, int nq, int k, int nprobe,
                                  const int64_t* list_dev, const float* coarse_dis_dev, float* D_dev, int64_t* I_dev,
                                  void* ws_dev, size_t ws_bytes, uint32_t* tau_local_dev,
                                  uint32_t* const* tau_peers_dev, int npeers, rsb_stream_t stream);
/* Copy `bytes` from src_dev to dst_ptrs_dev[p] + dst_offset_bytes for every p < npeers (peer-mapped destinations; P2P
 * stores over NVLink).  Used to publish a rank's slice of the coarse-quantizer tables to every GPU without NCCL.
 * 16-byte aligned pointers / sizes. */
int rsb_peer_broadcast(const void* src_dev, size_t bytes, void* const* dst_ptrs_dev, int npeers, size_t dst_offset_bytes,
                       rsb_stream_t stream);
/* coarse quantizer only: top-`nprobe` lists per query (the IndexFlatIP quantizer's search).
 * list_dev [nq, nprobe] int64, score_dev [nq, nprobe] float32 (may be NULL). */
int rsb_coarse(rsb_index_t* h, const float* q_dev, int nq, int nprobe, int64_t* list_dev, float* score_dev,
               void* ws_dev, size_t ws_bytes, rsb_stream_t stream);

/* ---- shard merge (src/search.py:357-367; api/serve_main_node.py:130-163) ---------------------------- */
/* D_all_dev/I_all_dev [nshards, nq, k]: concat per query, sort by score desc (ties: lower shard, then lower
 * rank, i.e. Python's stable sort over shard order), keep k_out.  Entries with id < 0 are ignored. */
int rsb_merge_topk(const float* D_all_dev, const int64_t* I_all_dev, int nshards, int nq, int k, int k_out,
                   float* D_dev, int64_t* I_dev, rsb_stream_t stream);

/* Fused gather + merge for one box: D_ptrs_dev / I_ptrs_dev are DEVICE arrays of nshards pointers; entry s points
 * at shard s's [nq, k] scores / ids, which may live on another GPU (peer-mapped / symmetric memory).  The kernel
 * reads them in place with P2P loads over NVLink, so no all-gather buffer is materialised.  The caller orders the
 * producers before this call (cross-GPU barrier). */
int rsb_merge_topk_peers(const float* const* D_ptrs_dev, const int64_t* const* I_ptrs_dev, int nshards, int nq, int k,
                         int k_out, float* D_dev, int64_t* I_dev, rsb_stream_t stream);
/* Query-sliced form of the same merge (same reference semantics, src/search.py:357-367): this GPU merges only
 * queries [q0, q0 + nq_slice) from all shards and stores each merged row into every one of the `nout` result
 * buffers D_outs_dev[o] / I_outs_dev[o] (each [nq, k_out], peer-mapped), i.e. the gather of the inputs and the
 * broadcast of the outputs are both P2P traffic of this one kernel.  The caller provides a cross-GPU barrier before
 * (inputs complete) and after (outputs complete). */
int rsb_merge_topk_peers_scatter(const float* const* D_ptrs_dev, const int64_t* const* I_ptrs_dev, int nshards, int q0,
                                 int nq_slice, int k, int k_out, float* const* D_outs_dev, int64_t* const* I_outs_dev,
                                 int nout, rsb_stream_t stream);

/* ---- dense exact search without an index object (used for ground truth / k-means assignment) -------- */
size_t rsb_knn_workspace_bytes(int nq, int64_t n, int k);
int rsb_knn_ip(const float* q_dev, int nq, const float* x_dev, int64_t n, int d, int k, int64_t id_offset,
               float* D_dev, int64_t* I_dev, void* ws_dev, size_t ws_bytes, rsb_stream_t stream);

/* ---- training steps (index.train(x): src/indicies/ivf_flat.py:166, ivf_pq.py:170 -> faiss Clustering /
 *      ProductQuantizer::train).  Lloyd iterations are driven by the host (retrieval_scaling_b200/train.py); the
 *      arithmetic runs here.  Coarse assignment step = rsb_coarse(..., nprobe = 1) on a scratch handle holding the
 *      current centroids. ------------------------------------------------------------------------------------ */
/* sums_dev [k, d] += x[i], counts_dev [k] (float) += 1 for assign_dev[i] (int32, out-of-range ids are skipped) */
int rsb_kmeans_accumulate(const float* x_dev, int64_t n, int d, const int32_t* assign_dev, int k, float* sums_dev,
                          float* counts_dev, rsb_stream_t stream);
/* PQ k-means assignment step: codes_dev [n, M] = argmin_j || r[i, m-th slice] - codebook[m][j] ||^2 (ksub = 256) */
int rsb_pq_assign(const float* r_dev, int64_t n, int d, int M, const float* codebook_dev, uint8_t* codes_dev,
                  rsb_stream_t stream);
/* PQ k-means update step: sums_dev [M, 256, d/M] += slices, counts_dev [M, 256] (float) += 1 */
int rsb_pq_accumulate(const float* r_dev, int64_t n, int d, int M, const uint8_t* codes_dev, float* sums_dev,
                      float* counts_dev, rsb_stream_t stream);

/* ---- options -------------------------------------------------------------------------------------------- */
enum {
    RSB_OPT_COARSE_TENSOR = 0 /* 1 (default): coarse quantizer scores by 3xTF32 on tcgen05 tensor cores (fp32-equivalent
                                 accuracy); 0: CUDA-core fp32 FMA tiles */
};
int rsb_set_option(rsb_index_t* h, int option, int64_t value);

/* ---- profiling: per-stage CUDA-event timings of the last rsb_search on this handle ------------------- */
enum {
    RSB_PROF_COARSE_MS = 0, /* centroid scan (sgemm + select)          */
    RSB_PROF_SETUP_MS = 1,  /* (query,list) work-list construction      */
    RSB_PROF_LUT_MS = 2,    /* PQ look-up-table build                   */
    RSB_PROF_SCAN_MS = 3,   /* inverted-list scan kernel (the hot one)  */
    RSB_PROF_MERGE_MS = 4,  /* per-query top-k merge                    */
    RSB_PROF_SCAN_BYTES = 5,/* algorithmic bytes of the scan: sum over probed (q,list) pairs of len*row_bytes */
    RSB_PROF_PAIRS = 6,     /* number of valid (q,list) pairs            */
    RSB_PROF_LAUNCHES = 7,  /* kernels launched by the last search       */
    RSB_PROF_SCAN_PATH = 8, /* IVFPQ scan: 1 = literal-offset shared-memory look-ups, 2 = generic addressing */
    RSB_PROF_COUNT = 9
};
int rsb_set_profiling(rsb_index_t* h, int enable);
/* synchronises the events of the last search; out[RSB_PROF_COUNT] doubles */
int rsb_get_profile(rsb_index_t* h, double* out, int n);

/* ---- query encoder: BERT-base forward in fp16 on tcgen05 tensor cores ------------------------------------
 * Replaces `model(**encoded_batch)` (src/search.py:92) for `Contriever(BertModel)` (contriever/src/contriever.py:
 * 11-55) and plain HF BERT checkpoints with CLS pooling (src/search.py:93-94).  Token streams are un-padded:
 * input_ids / token_type_ids are [T] int32 (padding removed), cu_seqlens [B+1] int32 prefix sums. */
typedef struct rsb_bert rsb_bert_t;
const char* rsb_bert_last_error(void);
int rsb_bert_create(int hidden, int layers, int heads, int intermediate, int vocab, int max_pos, int type_vocab,
                    float ln_eps, rsb_bert_t** out);
int rsb_bert_free(rsb_bert_t* h);
/* name = HF BertModel state_dict key (e.g. "encoder.layer.3.attention.self.query.weight"); data fp16, copied */
int rsb_bert_load(rsb_bert_t* h, const char* name, const void* f16_dev, int64_t n_elements, rsb_stream_t stream);
size_t rsb_bert_workspace_bytes(rsb_bert_t* h, int total_tokens);
/* pooling: 0 = mean over tokens (Contriever), 1 = CLS row.  out_f16_dev [B, 768] fp16 */
int rsb_bert_forward(rsb_bert_t* h, const int32_t* input_ids_dev, const int32_t* token_type_ids_dev,
                     const int32_t* cu_seqlens_dev, int B, int T, int max_seqlen, int pooling, void* out_f16_dev,
                     void* ws_dev, size_t ws_bytes, rsb_stream_t stream);
int64_t rsb_bert_launches(rsb_bert_t* h);
/* the forward's attention on its own: softmax(Q K^T / 8) V per (sequence, head) of the un-padded qkv_f16_dev
 * [T, 3 x 768] (Q | K | V of each token, heads of 64 contiguous) into ctx_f16_dev [T, 768]; cu_seqlens_dev [B+1] int32,
 * max_seqlen >= the longest sequence (<= 512) */
int rsb_bert_attention(rsb_bert_t* h, const void* qkv_f16_dev, const int32_t* cu_seqlens_dev, int B, int T, int max_seqlen,
                       void* ctx_f16_dev, rsb_stream_t stream);
/* the forward's LayerNorm on its own (eps of the handle): in / out [T, 768], gamma / beta [768], all fp16 */
int rsb_bert_layernorm(rsb_bert_t* h, const void* in_f16_dev, int T, const void* gamma_f16_dev, const void* beta_f16_dev,
                       void* out_f16_dev, rsb_stream_t stream);
/* the encoder's tensor-core GEMM on its own: C[M,N] = A[M,K] . W[N,K]^T + bias (epilogue 0), GELU (1) or
 * + residual (2); all fp16 row-major device pointers, N % 128 == 0, K % 64 == 0.  N % 256 == 0 up to 4096 runs the
 * CTA-pair kernel the forward uses, other N a one-tile-per-CTA kernel.  `epilogue | RSB_GEMM_ROWS_REVERSED` makes the
 * CTA-pair kernel visit the row tiles last-to-first (the order of the forward's FFN2); the one-tile-per-CTA kernel has
 * no tile order and ignores it, and so does every call when the environment sets RSB_NO_SNAKE.  The result is the same
 * either way. */
#define RSB_GEMM_ROWS_REVERSED 0x100
int rsb_gemm_f16(const void* A_dev, const void* W_dev, const void* bias_dev, const void* residual_dev, void* C_dev,
                 int M, int N, int K, int epilogue, rsb_stream_t stream);

/* diagnostic: shared-window address at which dynamic shared memory starts (the scan kernel folds it into LDS) */
int rsb_debug_smem_base(void);

/* ---- layout self-description (lets host-side tests pin the interleaved PQ layout without a GPU) ------- */
/* byte offset, inside a 32-vector block of M*32 bytes, of sub-quantizer m of block-local vector v */
int rsb_pq_layout_offset(int M, int v, int m);
/* float index, inside one 256x64 look-up-table row block, where entry (j, m) lives (first replica) */
int rsb_pq_lut_index(int M, int j, int m);

#ifdef __cplusplus
}
#endif
#endif /* RSB_H_ */
