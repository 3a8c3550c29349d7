/*
 * hgr_b200.h -- C ABI of libhgr_b200.so: the B200 (sm_100a) scoring head of HGR-Net.
 *
 * The reference (WilliamYi96/HGR-Net) is pure Python/PyTorch and has no FFI; the seam this
 * library sits behind is the `tree_model` nn.Module API used by the reference's main.py
 * (SURVEY.md section 8b).  Each entry point below names the reference code it replaces
 * (paths relative to the reference checkout).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *  - plain pointers and sizes; every pointer is a DEVICE pointer unless stated otherwise;
 *  - the caller owns all memory; the library never allocates device memory and keeps no
 *    state between calls (TMA descriptors are rebuilt per call on the host);
 *  - work is enqueued on `stream` (a cudaStream_t passed as void*); calls are asynchronous;
 *  - every function returns 0 (HGR_OK) or a negative HGR_ERR_* code; hgr_last_error()
 *    returns a thread-local message for the last failure;
 *  - matrices are row-major and dense (leading dimension == number of columns) unless a
 *    leading dimension is passed explicitly;
 *  - no CPU fallback exists: without a CUDA device every compute entry returns HGR_ERR_CUDA.
 */
#ifndef HGR_B200_H
#define HGR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HGR_ABI_VERSION 1

#define HGR_OK 0
#define HGR_ERR_BAD_ARG (-1)      /* null pointer, negative size, misaligned pointer        */
#define HGR_ERR_UNSUPPORTED (-2)  /* shape / dtype / K outside what the kernels implement   */
#define HGR_ERR_CUDA (-3)         /* CUDA runtime / driver error, message has the code      */
#define HGR_ERR_WORKSPACE (-4)    /* workspace smaller than hgr_*_workspace_bytes()         */

/* element types of feature matrices */
#define HGR_F32 0
#define HGR_BF16 1
#define HGR_F16 2

/* Hit@k cut-offs of the reference's eval loop (main.py:120) */
#define HGR_NUM_HITS 5
#define HGR_TOPK_MAX 32 /* K <= 32; the reference uses maxk = 20 (main.py:137)              */

/* implementation selector of hgr_score_topk (all compute the same result) */
#define HGR_IMPL_AUTO 0
#define HGR_IMPL_SIMT 1     /* CUDA-core kernel: any shape, exactness fallback and debug aid */
#define HGR_IMPL_TCGEN05 2  /* production: TMA + tcgen05/TMEM CTA-pair kernel (cta_group::2), fused top-k epilogue with
                             * deferred-insert lists; narrow (speculative) lists where provably cheap, certified and
                             * repaired exactly by the merge kernel */
#define HGR_IMPL_TCGEN05_EXACT 4  /* the same kernel with speculation off: every list holds K entries */
#define HGR_IMPL_TCGEN05_NULL 5   /* diagnostics: production main loop, trivial epilogue; outputs untouched */
#define HGR_IMPL_TCGEN05_SKETCH 12 /* the same main loop with the floor-sketch epilogue (K <= 20): unsorted candidate lists
                                    * filtered against a per-row floor shared by all workers through global memory --
                                    * exact by construction, cost independent of the bank order (no repair pass) */
/* OR-ed into `impl`: run only the GEMM + fused top-k kernel and leave the per-CTA partial lists in
 * the workspace (outputs untouched).  Lets bench.py time the dominant kernel alone for the roofline. */
#define HGR_IMPL_FLAG_NO_MERGE 0x100
/* OR-ed into `impl`: HGR_IMPL_GRID_SHARE(c) plans the tcgen05 scoring kernel for one of c batches meant to run at the
 * same time on round-robin streams: floor(CTA pairs / c) pairs, rounded down to a multiple of the row tiles, instead of
 * all of them (fewer, longer worker streams and lists; same results).  c in [1, HGR_GRID_SHARE_MAX]; 0 and 1 mean the
 * whole grid.  The floor-sketch variant and the SIMT kernel always use the whole grid.  hgr_score_topk_grid_share gives
 * the share the library recommends for a shape. */
#define HGR_IMPL_GRID_SHARE_SHIFT 12
#define HGR_IMPL_GRID_SHARE_MASK (0xF << HGR_IMPL_GRID_SHARE_SHIFT)
#define HGR_IMPL_GRID_SHARE(c) ((c) << HGR_IMPL_GRID_SHARE_SHIFT)
#define HGR_GRID_SHARE_MAX 8

int hgr_version(void);
const char* hgr_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t hgr_launch_count(void);

/*
 * Class-bank builder: out[r] = normalize( sum_{j in row(r)} w[j] * E[col[j]] ), fp32 math.
 *
 * Replaces `text_feats / text_feats.norm(dim=-1, keepdim=True)` of update_classifier
 * (model/clip_tree.py:318-325), the image-feature normalisation of forward
 * (model/clip_tree.py:330) and of train_batch (:225,:262), and -- with row_map -- the
 * `logits[:, test_index]` column gather of main.py:136 (gather bank rows once instead of
 * logit columns per batch).  The multi-node CSR form is the hierarchy aggregation named by
 * north_star; its operator shape follows baseline/DGP/models/gcn_dense_att.py:31-46,:116.
 *
 *  E        [n_src, D] of e_dtype (HGR_F32 | HGR_BF16 | HGR_F16), D % 8 == 0
 *  rowptr   [n_rows+1] int32 CSR offsets, or NULL for the identity CSR (row i = {i}, w = 1)
 *  col, w   [nnz] int32 / fp32; w may be NULL (all ones)
 *  row_map  [n_out] int32: output row r is CSR row row_map[r]; NULL -> r
 *  out      [n_out, D] of out_dtype (HGR_BF16 | HGR_F32)
 *  out_norm [n_out] fp32 pre-normalisation L2 norms, or NULL
 * A zero-norm row yields NaNs exactly like the reference's division.
 */
int hgr_aggregate_normalize(const void* E, int e_dtype, int64_t n_src, int64_t D,
                            const int32_t* rowptr, const int32_t* col, const float* w,
                            int64_t n_rows, const int32_t* row_map, int64_t n_out,
                            void* out, int out_dtype, float* out_norm, void* stream);

/*
 * Bank refresh in ONE pass (model/clip_tree.py:318-325 + the `logits[:, test_index]` gather of main.py:136): a chunk
 * of text features is row-normalised straight into its rows of the all-node bank `out` (bf16 [n_rows, D] -- pass the
 * chunk's slice of `zsl_weights`), and every row r with dst_map[r] >= 0 is ALSO written to row dst_map[r] of `out2`,
 * the test-class bank in its own (e.g. permuted) row order.  Replaces the reference's two halves + `torch.cat` +
 * normalise and a second pass for the gathered bank.  dst_map / out2 may both be NULL.
 */
int hgr_normalize_rows_dual(const void* E, int e_dtype, int64_t n_rows, int64_t D, void* out, const int32_t* dst_map,
                            void* out2, void* stream);

/*
 * Fused eval head: logits = scale * X @ bank^T are produced tile by tile on the tensor
 * cores and reduced on the fly to the per-row sorted top-K and the Hit@{1,2,5,10,20}
 * counters; the B x C logit matrix is never written to memory.
 *
 * Replaces `feats @ self.zsl_weights.T` (model/clip_tree.py:331) + `logits[:, test_index]`,
 * `.topk(maxk, 1, True, True)`, `model.test_index[pred]`, `pred.eq(targets)` and the
 * per-k `correct[:k].sum()` of main.py:136-147.
 *
 *  X         [B, D] bf16, already row-normalised (hgr_aggregate_normalize)
 *  bank      [C, D] bf16 class bank (rows of the test classes), 16-byte aligned, D % 8 == 0
 *  col_id    [C] int32 node id of bank row c (== test_index), or NULL -> id_base + c
 *  targets   [B] int32 node id of the label of each image, or NULL (no hit counting)
 *  topk_val  [B, K] fp32 logits, sorted descending; ties broken by ascending bank row
 *  topk_idx  [B, K] int32 node ids (col_id applied)
 *  hits      [HGR_NUM_HITS] int64, INCREMENTED by the number of rows whose label is within
 *            the top-{1,2,5,10,20}; NULL to skip.  (k beyond K counts within K.)
 *  workspace at least hgr_score_topk_workspace_bytes(B, C, D, K) bytes, 16-byte aligned, ZERO on first use and
 *            reserved for the scoring family (hgr_score_topk, _scatter, _scatter_bounded, hgr_score_topk_splits,
 *            _splits_scatter_bounded) between calls: its header carries state from one call to the next (the rows the
 *            last call re-scanned exactly, in its first word, and the launch epoch of the floor-sketch variant), so it
 *            is never cleared per batch and no other call may write it
 * If C < K the missing entries are (-inf, -1).
 */
size_t hgr_score_topk_workspace_bytes(int64_t B, int64_t C, int64_t D, int K);
/* The decisions hgr_score_topk takes for a shape on the tcgen05 path, without launching anything (host only; on a
 * box without a GPU the SM count of a B200 is assumed): plan[0..7] = {workers (CTA pairs), row tiles, 16-row units
 * per row tile, partial lists per row, entries per list (< K: speculative), epilogue warps per TMEM quarter, operand
 * ring depth, bank rows streamed per worker}. */
int hgr_score_topk_plan(int64_t B, int64_t C, int64_t D, int K, int32_t* plan /* [8] */);
/* hgr_score_topk_plan for a call with impl | HGR_IMPL_GRID_SHARE(grid_share). */
int hgr_score_topk_plan_shared(int64_t B, int64_t C, int64_t D, int K, int grid_share, int32_t* plan /* [8] */);
/* The grid share the library recommends for a batch of this shape that runs beside others (host only): > 1 on short
 * streams (few bank columns per worker on the whole grid), 1 otherwise and for shapes the tcgen05 kernel does not take. */
int hgr_score_topk_grid_share(int64_t B, int64_t C, int64_t D, int K);
/* What one batch of hgr_score_topk asks of an SM, for checking which of its kernels can share one: {threads, registers
 * per thread, static shared memory, dynamic shared memory} of (0) the row normalise of x_dtype [B, D] features into
 * bf16, (1) the tcgen05 scoring kernel, (2) the merge of its partial lists.  Needs a device. */
int hgr_score_topk_footprint(int64_t B, int64_t C, int64_t D, int K, int x_dtype, int32_t* out /* [12] */);
/* hgr_score_topk_footprint for a call with impl | HGR_IMPL_GRID_SHARE(grid_share). */
int hgr_score_topk_footprint_shared(int64_t B, int64_t C, int64_t D, int K, int grid_share, int x_dtype,
                                    int32_t* out /* [12] */);
int hgr_score_topk(const void* X, const void* bank, const int32_t* col_id, int32_t id_base,
                   const int32_t* targets, int64_t B, int64_t C, int64_t D, float scale, int K,
                   void* workspace, size_t workspace_bytes, float* topk_val, int32_t* topk_idx,
                   int64_t* hits, int impl, void* stream);

/*
 * Merge P partial top-K lists per row into the final sorted top-K and the hit counters.
 * Used for the class-sharded multi-GPU head (one list per rank after the NCCL all-gather)
 * and internally for the per-CTA partial lists of hgr_score_topk.
 *
 *  part_val / part_idx  [P, B, K] fp32 / int32 (idx already global node ids; -1 = empty);
 *                       consecutive parts are part_stride ELEMENTS apart (0 -> B*K, dense), so a
 *                       gathered buffer of per-rank {val[B,K], idx[B,K]} records can be merged in place
 *  outputs as hgr_score_topk.  Order: value descending, then part index, then position.
 */
int hgr_topk_merge(const float* part_val, const int32_t* part_idx, int64_t P, int64_t B, int K,
                   int64_t part_stride, const int32_t* targets, float* topk_val, int32_t* topk_idx,
                   int64_t* hits, void* stream);

/*
 * ---- class-sharded head over PEER MEMORY (one process per GPU, NVLink / NVSwitch) ----------------------------
 * The reference is single-GPU (main.py:226); SURVEY.md section 8e shards the class bank row-wise over G ranks.
 * Every rank scores the whole image batch against its shard; image rows are owned block-wise
 * (rank g owns rows [g * block_rows, (g + 1) * block_rows)), and a rank's local top-K of a row is written by the
 * producing kernel straight into the OWNER's exchange buffer over NVLink -- no collective call and no staging
 * copy on the data path.  The owner merges its G lists per row (hgr_topk_merge) and counts Hit@k for its rows.
 *
 * hgr_peer_alloc / hgr_peer_open   cudaMalloc'd (zeroed) exchange buffer + its 64-byte CUDA IPC handle; a peer
 *                                  process maps it with hgr_peer_open (peer access is enabled on first use).
 * hgr_score_topk_scatter           hgr_score_topk whose final [B, K] lists go, block of rows by block of rows, to
 *                                  val_blocks[g] / idx_blocks[g] (HOST arrays of n_blocks device pointers, local
 *                                  or peer); no hit counting (a hit needs the merged, global rank).  workspace as
 *                                  hgr_score_topk's (zero on first use, reserved for the scoring family).
 * hgr_peer_signal                  after the scatter: publish this rank's next sequence number (device counter
 *                                  *seq, incremented by the kernel) to flags[g] (one word on every rank g).
 * hgr_peer_wait                    before the merge: increment the consumer's own device counter *seq and spin
 *                                  until all n local flag words have reached it.  Traps (never hangs) after 10 s
 *                                  (HGR_PEER_TIMEOUT_MS overrides).
 * Both counters advance once per launch, so a signal/wait pair can live in a replayed CUDA graph.
 */
#define HGR_IPC_HANDLE_BYTES 64
#define HGR_MAX_PEERS 16
int hgr_peer_alloc(size_t bytes, void** ptr, unsigned char* handle /* [HGR_IPC_HANDLE_BYTES] */);
int hgr_peer_open(const unsigned char* handle, void** ptr);
int hgr_peer_close(void* ptr);
int hgr_peer_free(void* ptr);
int hgr_score_topk_scatter(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, int64_t B,
                           int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                           int64_t block_rows, int n_blocks, float* const* val_blocks,
                           int32_t* const* idx_blocks, int impl, void* stream);
/*
 * GLOBAL CERTIFICATE of the class-sharded head.  A shard's share of a row's stream is short (N = 8: 2,731 of 21,841
 * classes, cut into 4 lists per row), and short streams with exact K-entry lists are all list warm-up (measured:
 * 39.4 us per call at the N = 8 shard against 26.7 us with 10-entry lists).  Narrow lists cannot be certified against
 * the shard's OWN K-th value (a quarter of the shard's top-20 sits in every list), but they can against the GLOBAL
 * K-th value, which only the owner of the row knows.  So:
 *
 * hgr_score_topk_scatter_bounded   hgr_score_topk_scatter with lists sized for the row's global stream of C_total
 *                                  classes; no local certificate, no local repair.  Next to the final list of a row
 *                                  the producer stores bound_blocks[g][row - g * block_rows] = scale * (the largest
 *                                  last entry of its FULL narrow lists; -inf when no list dropped anything): every
 *                                  candidate the shard did not report is <= that bound.  workspace as
 *                                  hgr_score_topk's (zero on first use, reserved for the scoring family).
 * hgr_topk_merge_certified         hgr_topk_merge of the P = n_shards lists of the owner's rows; a row is certified
 *                                  when its merged K-th value beats every shard's bound STRICTLY.  Otherwise the
 *                                  doubtful shards are re-scanned exactly on the CUDA cores with the row's features
 *                                  X[row] against shards[p].bank (device pointers in DEVICE memory; a peer's bank is
 *                                  read over NVLink), bank rows mapped to node ids by shards[p].col_id / id_base and
 *                                  values multiplied by `scale` like the producers did.  With bank rows in random
 *                                  order this is a < 1e-4-per-batch event by construction of the list length
 *                                  (hgr_score_topk_global_list_len); *repair_count (optional, device) counts the rows.
 * The result is exact either way -- same contract as hgr_score_topk.
 */
typedef struct hgr_shard {
  const void* bank;       /* [C, D] bf16, 16-byte aligned */
  const int32_t* col_id;  /* [C] node ids or NULL -> id_base + bank row */
  int64_t C;
  int32_t id_base;
  int32_t reserved;
} hgr_shard_t;
int hgr_score_topk_global_list_len(int64_t B, int64_t C, int64_t D, int K, int64_t C_total);
int hgr_score_topk_scatter_bounded(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, int64_t B,
                                   int64_t C, int64_t D, float scale, int K, void* workspace, size_t workspace_bytes,
                                   int64_t block_rows, int n_blocks, float* const* val_blocks,
                                   int32_t* const* idx_blocks, float* const* bound_blocks, int64_t C_total, int impl,
                                   void* stream);
int hgr_topk_merge_certified(const float* part_val, const int32_t* part_idx, const float* part_bound, int64_t P,
                             int64_t B, int K, int64_t part_stride, int64_t bound_stride, const int32_t* targets,
                             float* topk_val, int32_t* topk_idx, int64_t* hits, const void* X, int64_t D,
                             const hgr_shard_t* shards, float scale, unsigned int* repair_count, void* stream);
 /* hgr_normalize_rows_bcast: feature ingest of the sharded head.  A rank copies only ITS block of image rows from the
  * host; this kernel normalises them (clip_tree.py:330) and stores row r at row (row0 + r) of every destination
  * dst[g] (HOST array of n_dst device pointers to bf16 [*, D] arrays, local or peer), so the A operand of
  * hgr_score_topk is replicated over NVLink by the producer instead of n_dst times over PCIe. */
int hgr_normalize_rows_bcast(const void* E, int e_dtype, int64_t n_rows, int64_t D, int64_t row0, int n_dst,
                             void* const* dst, void* stream);
int hgr_peer_signal(uint32_t* const* flags, int n, uint32_t* seq, void* stream);
int hgr_peer_wait(const uint32_t* flags, int n, uint32_t* seq, void* stream);

/*
 * HOST helper of row a7 (no device work): draw-identical replay of the index selection of CPython's
 * `random.sample(population, k)` -- the call the reference draws its negatives with (model/clip_tree.py:134; 17 calls
 * per OM step at cfg 3) -- on a window of Mersenne-Twister outputs.  words[i] is the i-th 32-bit output the generator
 * would produce next (a k-bit getrandbits, k <= 32, is `word >> (32 - k)`); n = len(population); setsize is CPython's
 * threshold between its two algorithms (21, + 4 ** ceil(log4(3 k)) when k > 5): n <= setsize runs the pool algorithm
 * (j = randbelow(n - i); result[i] = pool[j]; pool[j] = pool[n - i - 1]), else the set algorithm (j = randbelow(n),
 * redrawn while already selected).  Writes the k selected POSITIONS to out_pos; scratch holds n int32.
 * Returns the number of words consumed (>= 0), -1 when the window is too short (call again with more words), -2 on
 * bad arguments.  hgrnet_b200/sampling.py (SampleStream) keeps the generator state identical to the reference's.
 */
int64_t hgr_sample_replay(const uint32_t* words, int64_t n_words, int64_t n, int64_t k, int64_t setsize,
                          int32_t* out_pos, int32_t* scratch);
/* `count` consecutive calls random.sample(range(n[c]), k[c]) in one go (an OM step's 17 draws): positions of call c at
 * out_pos[k[0] + ... + k[c-1] ...]; scratch holds max(n) int32; setsize is computed here.  Same return values. */
int64_t hgr_sample_replay_many(const uint32_t* words, int64_t n_words, int64_t count, const int64_t* n, const int64_t* k,
                               int32_t* out_pos, int32_t* scratch);
/* The whole host-side plan of one OM training step (model/clip_tree.py:116-141 per iteration, :241-262 over the T
 * iterations) in one call: for iteration t the candidate list cand[t] (n_cand[t] node ids, already without the anchor
 * chain) is sub-sampled to num_compare ids exactly like `random.sample` would (only when it is longer), the anchor is
 * appended when the draw missed it (label_pos[t] = its position), the union of all sets is formed in ascending node id
 * (what numpy.unique gives) and every set is rewritten as positions in that union.
 *   set_ptr [T + 1], set_col [>= T * (num_compare + 1)], label_pos [T], union_ids [>= T * (num_compare + 1)] int32;
 *   counts[0] = entries of set_col, counts[1] = size of the union; scratch: n_nodes + max(n_cand) + num_compare int32.
 * Returns the generator words consumed (>= 0), -1 when the window is too short, -2 on bad arguments. */
int64_t hgr_om_plan(const uint32_t* words, int64_t n_words, int64_t T, const int64_t* const* cand, const int64_t* n_cand,
                    const int64_t* anchor, int64_t num_compare, int64_t n_nodes, int32_t* set_ptr, int32_t* set_col,
                    int32_t* label_pos, int32_t* union_ids, int64_t* counts, int32_t* scratch);

/*
 * Dense logits, out[b, c] = scale * <X[b], bank[c]>, fp32, leading dimension ldo >= C.
 * Same TMA/tcgen05 main loop as hgr_score_topk with a plain store epilogue.  Keeps
 * tree_model.forward()'s contract (model/clip_tree.py:328-333: returns [B, N] logits) for
 * callers that need the matrix (TOR/POR, main.py:143,162-176) and the training-step logits
 * `(img_feats_ @ text_feats.t()) * logit_scale.exp()` (model/clip_tree.py:263).
 */
int hgr_logits_dense(const void* X, const void* bank, int64_t B, int64_t C, int64_t D,
                     float scale, float* out, int64_t ldo, int impl, void* stream);

/*
 * TOR / POR hierarchical metrics (main.py:143,152-191; SURVEY.md 8-f1) of a batch in which every row is matched
 * against the chain of ITS OWN label, without the dense matrix.  For a single-label batch this is exactly the
 * reference's metric, whose per-batch edge / (L-1) and point / L are sums of per-row terms.  Replaces the L clone +
 * index_fill + gather + topk passes over [B, N] and the Python B x L loop with device->host copies of the reference's
 * test().  Needs no host work per batch and no memset, so it can be captured in a CUDA graph.
 *
 * The train rows of the bank are handed over SORTED BY LEVEL (stable: inside a level in train_index order);
 * X . bank_sorted^T runs on the tcgen05 main loop and the epilogue keeps, per image row, a running arg-max of the
 * current level -- the level of a column is warp-uniform and changes n_levels - 1 times over the whole bank -- and
 * publishes it with one 64-bit atomicMax per (row, level, worker).  A second, tiny kernel decodes the winners, maps
 * sorted rows back to train POSITIONS (positions in train_index; chain_pos / first_out / lvl_idx / top1 are positions
 * too), applies the -1 rule and counts.
 *
 *  X            [B, D] bf16, row-normalised          bank_sorted [M, D] bf16, train rows sorted by level
 *  level_end    [n_levels] int32 HOST array: level l = sorted rows [level_end[l-1], level_end[l]); last entry = M;
 *               n_levels <= 32
 *  sorted_to_pos [M] int32 (device): position in train_index of sorted row s
 *  first_out    [n_levels] int32: first position j whose column is NOT at level l (a masked column holds -1.0, so that
 *               position wins when no in-level logit exceeds -1; >= M when there is none)
 *  workspace    B * n_levels * 8 bytes (device): ZERO on first use; the call hands it back zeroed (no memset per batch)
 *  lvl_idx      [B, n_levels] int32 per-level arg-max position after the -1 rule (optional), top1 [B] int32 arg-max
 *               position over the train columns (optional); neither depends on the labels
 *  targets      [B] int32 node id of each row's label
 *  chain table  CSR over all n_nodes nodes, built once per model: the chain of node n is c2p[n] + [n], entries
 *               [chain_ptr[n], chain_ptr[n+1]); per entry chain_pos = its position in train_index (-1: not a train
 *               class) and chain_level = its depth.  chain_ptr [n_nodes + 1] int32, chain_pos / chain_level int32.
 *  counts       [HGR_HIER_MAX_CHAIN + 1][4] int64, INCREMENTED: bin L (chain length) holds {rows, TOR hits (#{k: top1 ==
 *               chain[k]}), points (#{k: lvl[chain_level[k]] == chain[k]}), edges (#{k: matches at k and k+1}; L == 1:
 *               match[0])} of the rows whose chain has L entries (bin 0 stays zero).  The reference's totals follow on
 *               the host: hits = sum_L tor_L, path = sum_L edges_L / max(L-1, 1), point = sum_L points_L / L.
 *  node_splits  NULL: n_sets must be 1 and counts is as above.  Otherwise [n_nodes] uint8 and 1 <= n_sets <= 8: counts
 *               is [n_sets][HGR_HIER_MAX_CHAIN + 1][4] and a row is added to set s for every bit s of
 *               node_splits[targets[row]] (main.py:143,152-191 run once per test split, from one GEMM per batch)
 * A row whose target lies outside [0, n_nodes), or whose chain length lies outside [1, HGR_HIER_MAX_CHAIN], is counted
 * nowhere (its lvl_idx / top1 are still written): callers pad a fixed-shape batch with target -1.
 * Ties: first position in train_index (the CPU arg-max rule; torch's CUDA top-k leaves it unspecified).
 */
#define HGR_HIER_MAX_CHAIN 32 /* = the 32-level limit of the per-level arg-max epilogue */
int hgr_hier_metrics_fused_rows(const void* X, const void* bank_sorted, int64_t B, int64_t M, int64_t D,
                                const int32_t* level_end, int n_levels, const int32_t* sorted_to_pos,
                                const int32_t* first_out, const int32_t* targets, int64_t n_nodes,
                                const int32_t* chain_ptr, const int32_t* chain_pos, const int32_t* chain_level,
                                const uint8_t* node_splits, int n_sets, void* workspace, size_t workspace_bytes,
                                int32_t* lvl_idx, int32_t* top1, int64_t* counts, void* stream);

/*
 * Several test splits of one hierarchy in ONE scoring pass (the reference prints one line per run of main.py:104-222
 * with --model_test / --data_test = 2-hops, 3-hops, all).  The bank [C, D] is the union of the splits' classes, ordered
 * so that the classes of equal split membership form contiguous GROUPS; the scoring kernel's partial lists never cross
 * a group, so for every split the merge takes exactly the lists of its groups -- certified against that split's own
 * K-th value and repaired exactly like hgr_score_topk.  Per split the result is hgr_score_topk on the split's rows of
 * the bank (same values, same (value desc, bank row asc) order).
 *
 *  n_groups, group_end   HOST [n_groups] int32 (n_groups <= 16): group g = bank rows [group_end[g-1], group_end[g]),
 *                        strictly ascending, group_end[n_groups-1] == C.  Copied into the kernel parameters: the call
 *                        can be captured in a CUDA graph.
 *  group_splits          HOST [n_groups] uint8: bit s set = the group's classes belong to split s (n_splits <= 8)
 *  node_splits           [n_nodes] uint8 split bits of every node id: a row counts toward split s only if bit s of
 *                        node_splits[targets[row]] is set (its label is a class of s); NULL with counts == NULL
 *  topk_val / topk_idx   [n_splits, B, K] fp32 / int32 node ids (col_id applied), as hgr_score_topk per split
 *  counts                [n_splits][HGR_NUM_HITS + 1] int64, INCREMENTED: Hit@{1,2,5,10,20} and the number of rows
 *                        counted -- the numerator and denominator of the split's line; NULL to skip
 *  impl                  HGR_IMPL_AUTO / HGR_IMPL_TCGEN05 / HGR_IMPL_TCGEN05_EXACT; others: HGR_ERR_UNSUPPORTED
 *  workspace             hgr_score_topk_splits_workspace_bytes(...) bytes, 16-byte aligned, ZERO on first use, left
 *                        reusable (no memset per batch); the rows re-scanned exactly are counted in its first word
 */
size_t hgr_score_topk_splits_workspace_bytes(int64_t B, int64_t C, int64_t D, int K, int n_groups, const int32_t* group_end);
int hgr_score_topk_splits(const void* X, const void* bank, const int32_t* col_id, int32_t id_base, const int32_t* targets,
                          const uint8_t* node_splits, int64_t n_nodes, int64_t B, int64_t C, int64_t D, float scale, int K,
                          int n_groups, const int32_t* group_end, const uint8_t* group_splits, int n_splits,
                          void* workspace, size_t workspace_bytes, float* topk_val, int32_t* topk_idx, int64_t* counts,
                          int impl, void* stream);

/*
 * hgr_hier_metrics_fused_rows for the CLASS-SHARDED head (main.py:143,152-191): the level-sorted train bank [M, D] is
 * cut into contiguous row ranges, one per rank, and image rows are owned block-wise as in hgr_score_topk_scatter.  The
 * result is bit-identical to hgr_hier_metrics_fused_rows on the whole batch on one GPU: a winner word is
 * (order key << 32 | ~global sorted row), larger = larger value or else smaller row, the stable level sort keeps
 * train_index order inside a level across shard boundaries, and max is associative -- so the max over the shards'
 * words is the word the single-GPU epilogue keeps, whatever the number of shards or the order of arrival.
 *
 * hgr_hier_level_scatter          producer: the per-level arg-max GEMM of X [B, D] against this rank's shard
 *                                 bank_shard [M_r, D] = sorted rows [row_base, row_base + M_r), level_end_local
 *                                 [n_levels] (HOST) = the global level ends clipped to the shard (non-decreasing, last
 *                                 = M_r).  Every word of rows [g * block_rows, (g + 1) * block_rows) is rebased to the
 *                                 global sorted row and stored, zeros included, at dst_blocks[g]
 *                                 [block_rows][n_levels] uint64 (HOST array of n_blocks device pointers, local or peer,
 *                                 8-byte aligned).  M_r == 0 runs no GEMM and stores zeros (X / bank_shard unused).
 *                                 workspace: B * n_levels * 8 bytes, zero on first use, handed back zeroed.  Enqueue it
 *                                 before hgr_peer_signal: the owner's hgr_peer_wait then covers these words too.
 * hgr_hier_finish_rows_gathered   owner: for its n_rows rows, the max over the n_parts word arrays parts[p *
 *                                 part_stride + row * n_levels + level] (part_stride in words), then the decode, -1
 *                                 rule, tie rule and chain matching of hgr_hier_metrics_fused_rows.  targets, lvl_idx,
 *                                 top1 cover the owner's rows; M, sorted_to_pos, first_out and the chain table are the
 *                                 GLOBAL ones; node_splits / n_sets / counts as hgr_hier_metrics_fused_rows.  parts
 *                                 is only read.
 */
int hgr_hier_level_scatter(const void* X, const void* bank_shard, int64_t B, int64_t M_r, int64_t D,
                           const int32_t* level_end_local, int n_levels, int64_t row_base, void* workspace,
                           size_t workspace_bytes, int64_t block_rows, int n_blocks, uint64_t* const* dst_blocks,
                           void* stream);
int hgr_hier_finish_rows_gathered(const uint64_t* parts, int n_parts, int64_t part_stride, int64_t n_rows, int64_t M,
                                  int n_levels, const int32_t* sorted_to_pos, const int32_t* first_out,
                                  const int32_t* targets, int64_t n_nodes, const int32_t* chain_ptr,
                                  const int32_t* chain_pos, const int32_t* chain_level, const uint8_t* node_splits,
                                  int n_sets, int32_t* lvl_idx, int32_t* top1, int64_t* counts, void* stream);

/*
 * Several test splits in one scoring pass on the CLASS-SHARDED head (main.py:104-222 run once per split, as
 * hgr_score_topk_splits, over G ranks).  Every rank holds about 1/G of EVERY group of the union bank (its slice of each
 * group, concatenated in group order, with the clipped group ends as its own group table), so every rank holds about
 * 1/G of every split.  Image rows are owned block-wise as in hgr_score_topk_scatter.
 *
 * Result and tie order: for split s the top-K of s's classes in the order (value desc, rank asc, local bank row asc) --
 * hgr_score_topk on s's rows of the ranks' banks concatenated rank after rank.  At G = 1 that is the union bank's own
 * order: the result is hgr_score_topk_splits's, bit for bit when neither call repairs a row (a repaired list carries
 * the CUDA cores' values of its re-scanned rows, which may differ from the GEMM's in the last bits).
 *
 * hgr_score_topk_splits_scatter_bounded   producer: the grouped scoring kernel of hgr_score_topk_splits on this rank's
 *                                 bank [C, D] (group table n_groups / group_end / group_splits as there), lists sized
 *                                 for each split's GLOBAL stream of split_C_total[s] classes (HOST [n_splits] int64;
 *                                 hgr_score_topk_splits_global_list_len), then per split s and row: the rank's top-K of
 *                                 s (node ids, values times scale) at val_blocks[g] / idx_blocks[g] + s * split_stride +
 *                                 (row - g * block_rows) * K and the bound -- scale * the largest last entry of its FULL
 *                                 narrow lists of s, -inf when none dropped anything -- at bound_blocks[g] + s *
 *                                 split_stride + row - g * block_rows (HOST arrays of n_blocks device pointers, local or
 *                                 peer; split_stride in 4-byte elements, >= n_blocks * block_rows * (2K + 1):
 *                                 a split's lists and bounds of all producers).  No local certificate, no repair, no counting.
 *                                 C == 0 (a rank without rows) and splits without rows here store (-inf, -1) lists and
 *                                 -inf bounds.  impl: HGR_IMPL_AUTO / HGR_IMPL_TCGEN05.  workspace:
 *                                 hgr_score_topk_splits_scatter_bounded_workspace_bytes(...), as hgr_score_topk_splits.
 * hgr_topk_merge_splits_certified owner: for its B rows and every split s, the merge of the P = G shard lists of s at
 *                                 part_val / part_idx + s * split_stride + p * part_stride + row * K in the order above,
 *                                 certified when the merged K-th value beats every shard's bound of s (part_bound + s *
 *                                 split_stride + p * bound_stride + row) STRICTLY.  A doubtful (row, split, shard) is
 *                                 re-scanned exactly on the CUDA cores: the rows of shards[p] whose node (col_id or
 *                                 id_base + row) has bit s in node_splits, over NVLink for a peer's bank.  topk_val /
 *                                 topk_idx [n_splits, B, K]; counts [n_splits][HGR_NUM_HITS + 1] int64, INCREMENTED as
 *                                 in hgr_score_topk_splits (optional); *repair_count (optional) counts (row, split) pairs
 *                                 repaired.  split_stride >= 2 * P * part_stride + P * bound_stride: a split's
 *                                 value lists, id lists and bounds all sit at + s * split_stride.
 */
size_t hgr_score_topk_splits_scatter_bounded_workspace_bytes(int64_t B, int64_t C, int64_t D, int K, int n_groups,
                                                             const int32_t* group_end);
int hgr_score_topk_splits_global_list_len(int64_t B, int64_t C, int64_t D, int K, int n_groups, const int32_t* group_end,
                                          const uint8_t* group_splits, int n_splits, const int64_t* split_C_total);
int hgr_score_topk_splits_scatter_bounded(const void* X, const void* bank, const int32_t* col_id, int32_t id_base,
                                          int64_t B, int64_t C, int64_t D, float scale, int K, int n_groups,
                                          const int32_t* group_end, const uint8_t* group_splits, int n_splits,
                                          const int64_t* split_C_total, void* workspace, size_t workspace_bytes,
                                          int64_t block_rows, int n_blocks, float* const* val_blocks,
                                          int32_t* const* idx_blocks, float* const* bound_blocks, int64_t split_stride,
                                          int impl, void* stream);
int hgr_topk_merge_splits_certified(const float* part_val, const int32_t* part_idx, const float* part_bound, int64_t P,
                                    int64_t B, int K, int n_splits, int64_t part_stride, int64_t bound_stride,
                                    int64_t split_stride, const int32_t* targets, const uint8_t* node_splits,
                                    int64_t n_nodes, float* topk_val, int32_t* topk_idx, int64_t* counts, const void* X,
                                    int64_t D, const hgr_shard_t* shards, float scale, unsigned int* repair_count,
                                    void* stream);

/*
 * Hierarchical mistake severity and LCA distance@k (Bertinetto et al., "Making Better Mistakes", CVPR 2020) of top-K
 * lists already on the device -- the lists of hgr_score_topk / hgr_score_topk_splits / the certified merges.  It
 * extends the Hit@k count of the reference's test() (main.py:135-148) from "is the label in the first k" to "how far
 * from the label are the first k".  Chain table as in hgr_hier_metrics_fused_rows, with the NODE ids per entry:
 * chain(n) = c2p[n] + [n] = chain_node[chain_ptr[n] .. chain_ptr[n+1]), depth(n) = len(c2p[n]).  Every c2p[n] is a
 * shortest root path, so the entry at index i of a chain has depth i.  For a label t and a prediction p:
 *   lca(t, p) = the largest index i with chain(t)[i] == chain(p)[i] (on a DAG the deepest match, not the end of the
 *               common prefix); -1 (a virtual super-root) without one
 *   h(t, p)   = depth(t) - depth(lca)          d(t, p) = depth(t) + depth(p) - 2 depth(lca)
 * A list entry outside [0, n_nodes) (-1: an empty entry when C < K) counts as the super-root: h = d = depth(t) + 1.
 * A row counts when 0 <= targets[row] < n_nodes and its chain has 1 .. HGR_HIER_MAX_CHAIN entries (the TOR / POR rule).
 *
 *  topk_idx    n_sets lists [B, K] int32 node ids, list set s at topk_idx + s * set_stride; K <= HGR_TOPK_MAX
 *  node_splits NULL: n_sets must be 1.  Otherwise [n_nodes] uint8 and n_sets <= 8: list set s counts a row only when
 *              bit s of node_splits[targets[row]] is set (the rule of hgr_score_topk_splits)
 *  counts      [n_sets][HGR_MISTAKE_COUNTERS] int64, INCREMENTED, per set:
 *                0      rows
 *                1      mistakes: rows whose first entry is not the label
 *                2..6   sum over rows of sum_{j < min(k, K)} h(t, p_j), k in {1, 2, 5, 10, 20}
 *                7..11  the same sums of d
 *                12..   histogram of d(t, p_0): bins 0 .. 2 * HGR_HIER_MAX_CHAIN, then one overflow bin
 * One warp per row, one ballot per list entry.  No allocation, no host work per batch: capturable in a CUDA graph.
 */
#define HGR_MISTAKE_COUNTERS (2 + 2 * HGR_NUM_HITS + 2 * HGR_HIER_MAX_CHAIN + 2)
int hgr_hier_mistakes(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                      const uint8_t* node_splits, const int32_t* chain_ptr, const int32_t* chain_node, int64_t n_nodes,
                      int64_t* counts, void* stream);

/*
 * Per-class Hit@{1,2,5,10,20} of top-K lists already on the device -- the lists of hgr_score_topk /
 * hgr_score_topk_splits / the certified merges: the reference's Hit@k count (main.py:135-148) kept per label, from
 * which the class-averaged accuracy (the mean over classes of Hit@k / rows) follows.
 * A row counts when 0 <= targets[row] < n_nodes: it adds 1 to `rows` of its label and, when the label is at position
 * pos of its list (first match), 1 to every Hit@k with pos < k (the rule of the hits / counts of hgr_score_topk).
 *
 *  topk_idx    n_sets lists [B, K] int32 node ids, list set s at topk_idx + s * set_stride; K <= HGR_TOPK_MAX
 *  node_splits NULL: n_sets must be 1.  Otherwise [n_nodes] uint8 and n_sets <= 8: list set s counts a row only when
 *              bit s of node_splits[targets[row]] is set (the rule of hgr_score_topk_splits)
 *  counts      [n_sets][n_nodes][HGR_NUM_HITS + 1] int64, INCREMENTED; row t of set s holds
 *              {Hit@1, Hit@2, Hit@5, Hit@10, Hit@20, rows} of the rows labelled t
 * One thread per row; the rows of a warp with equal labels are combined before they reach global memory (one atomic per
 * non-zero counter, label and warp).  No allocation, no host work per batch: capturable in a CUDA graph.
 */
int hgr_class_hits(const int32_t* topk_idx, int64_t B, int K, int64_t set_stride, int n_sets, const int32_t* targets,
                   const uint8_t* node_splits, int64_t n_nodes, int64_t* counts, void* stream);

/*
 * Fused masked cross-entropy of the OM training step over T sampled class sets
 * (model/clip_tree.py:241-277 with nn.CrossEntropyLoss, :49,:275).
 *
 *  logits   [B, U] fp32 (ld = ldl): scale * img_n @ text_n(union)^T, scale already applied
 *  set_ptr  [T+1] int32 offsets into set_col; set_col [set_ptr[T]] int32 columns (< U) of
 *           iteration t's sampled classes (`compare_idx`, :257); label_pos [T] int32 position
 *           of the positive inside its set (:139); weight [T] fp32 = w_in[m] * w_out[k] (:275)
 *  loss     [T] fp32: weight[t] * mean_b( logsumexp_j - logit_label )   (overwritten)
 *  dlogits  [B, U] fp32 (ld = ldl): sum_t weight[t]/B * (softmax_t - onehot_t), zero outside
 *           every set (overwritten, all zero when T == 0); NULL to skip the backward.
 *  workspace at least hgr_masked_ce_workspace_bytes(B, U, T) bytes.
 */
size_t hgr_masked_ce_workspace_bytes(int64_t B, int64_t U, int64_t T);
int hgr_masked_ce(const float* logits, int64_t ldl, int64_t B, int64_t U,
                  const int32_t* set_ptr, const int32_t* set_col, const int32_t* label_pos,
                  const float* weight, int64_t T, float* loss, float* dlogits,
                  void* workspace, size_t workspace_bytes, void* stream);

/*
 * Backward of the OM step's logits (model/clip_tree.py:276 through :263, :225/:262, then :280): with dlogits from
 * hgr_masked_ce (the T iterations already summed over the union of the sampled classes)
 *     d_img  [B, D] fp32 = d/d(raw image features)  of  x  = raw / |raw|,  via  d_x  = scale * dlogits   @ tn
 *     d_text [U, D] fp32 = d/d(raw text features)   of  tn = raw / |raw|,  via  d_tn = scale * dlogits^T @ x
 *     d_log_scale[0] += sum(dlogits * logits)        (d/d logit_scale of scale = exp(logit_scale); may be NULL)
 * Both gradient GEMMs run on the tcgen05 kernel of the scoring head (bf16 operands, fp32 accumulation).
 *  dlogits, logits [B, U] fp32 (ld = ldl); x [B, D], tn [U, D] bf16 unit rows with their pre-normalisation norms
 *  x_norm [B], t_norm [U] fp32 (hgr_aggregate_normalize's out_norm); D % 8 == 0.
 *  workspace at least hgr_om_backward_workspace_bytes(B, U, D) bytes.
 */
size_t hgr_om_backward_workspace_bytes(int64_t B, int64_t U, int64_t D);
int hgr_om_backward(const float* dlogits, const float* logits, int64_t ldl, int64_t B, int64_t U, int64_t D,
                    const void* x, const float* x_norm, const void* tn, const float* t_norm, float scale,
                    float* d_img, float* d_text, float* d_log_scale, void* workspace, size_t workspace_bytes,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HGR_B200_H */
