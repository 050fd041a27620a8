/*
 * pia_b200.h -- C ABI of libpia_b200.so: the B200 (sm_100a) draft -> verify -> accept hot loop of
 * PIA LOOKAHEAD.
 *
 * The reference path has no FFI: it is plain Python (SURVEY.md 8b).  This ABI therefore sits *below* the
 * Python surface the package keeps (LookaheadCache, lookahead_generation, the per-model forward) and
 * each entry point names the reference code whose work it takes over (paths relative to
 * /root/reference/lookahead/lookahead/).  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - every function returns PIA_OK (0) or a negative pia_status; pia_last_error() gives the text
 *     (thread local).  Nothing here allocates caller-visible memory: all `d_*` pointers are
 *     caller-owned DEVICE buffers, all `h_*` pointers are HOST buffers; `stream` is a cudaStream_t
 *     passed as void*.  Calls are asynchronous on `stream` unless stated otherwise and are legal
 *     inside CUDA-graph capture unless stated otherwise.
 *   - token ids are int32; attention masks are bit rows: row i of a draft of n <= 64*W nodes is W
 *     uint64 words, bit j set <=> node i attends draft node j (i.e. j is i or an ancestor of i).
 */
#ifndef PIA_B200_H_
#define PIA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIA_ABI_VERSION 2

typedef enum {
  PIA_OK = 0,
  PIA_ERR_INVALID = -1,   /* bad argument (python: AssertionError / ValueError)                     */
  PIA_ERR_INDEX = -2,     /* python IndexError of Tree.get (k-th largest beyond the collected list) */
  PIA_ERR_CAPACITY = -3,  /* node / edge / frontier pool exhausted                                   */
  PIA_ERR_CUDA = -4,      /* CUDA runtime error, see pia_last_error()                                */
  PIA_ERR_UNSUPPORTED = -5
} pia_status;

const char *pia_last_error(void);
int pia_abi_version(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches claim) */
unsigned long long pia_launch_count(void);

/* ============================================================================================
 * Trie draft cache   (common/lookahead_cache.py: Tree :24-333, LookaheadCache :336-587)
 * ============================================================================================ */
typedef struct pia_trie pia_trie_t;

enum { PIA_MODE_INPUT = 0, PIA_MODE_OUTPUT = 1, PIA_MODE_MIX = 2 };
enum { PIA_GET_HIER = 0, PIA_GET_ONE = 1 };
/* pia_trie_get flags */
enum {
  PIA_GET_TAIL = 1,      /* d_queries is one growing token sequence per row; the query is its last
                            min(max_query_length, len) tokens (pretrained_model.py:708) */
  PIA_GET_FIRST_ONLY = 2 /* consult only the tree of the first query token: Tree.get(token_ids[1:]) (:65) */
};

typedef struct {
  int32_t vocab_capacity;      /* token ids must be in [0, vocab_capacity)                          */
  int64_t node_capacity;       /* 32-byte node records                                              */
  int64_t edge_capacity;       /* 8-byte (token,node) child entries                                 */
  int32_t n_input_slots;       /* distinct request `idx` values (>=1; bs=1 loop uses idx 0)         */
  int32_t max_node;            /* Tree.max_node          (lookahead_cache.py:337, default 65536)    */
  int32_t max_output_node;     /* Tree.max_output_node   (default 512)                              */
  int32_t max_put_tokens;      /* longest token list of one put/stream_put call                     */
  int32_t frontier_capacity;   /* BFS frontier entries per resident query CTA                       */
  int32_t max_resident_queries;/* query CTAs resident at once (scratch is sized for this many)      */
} pia_trie_config_t;

typedef struct {
  int64_t nodes_used, edges_used;
  int32_t n_trees;
  int32_t n_update_trees;       /* len(_update_trees)       */
  int32_t n_update_input_trees; /* len(_update_input_trees) */
  int32_t error_flags;          /* sticky device-side PIA_ERR_CAPACITY indicators */
  int64_t nodes_visited;        /* cumulative node records read by get kernels (roofline accounting) */
  int64_t edges_visited;
} pia_trie_stats_t;

/* LookaheadCache.__init__ (lookahead_cache.py:337-347). Synchronous; not capturable. */
int pia_trie_create(const pia_trie_config_t *cfg, pia_trie_t **out);
int pia_trie_destroy(pia_trie_t *t);
/* eos_ids / stop_words attributes (written by callers: pretrained_model.py:1088-1089). Synchronous. */
int pia_trie_set_eos(pia_trie_t *t, const int32_t *h_eos, int n);
int pia_trie_set_stop_words(pia_trie_t *t, const int32_t *h_words, int n);
int pia_trie_set_limits(pia_trie_t *t, int max_node, int max_output_node);

/* LookaheadCache.put (lookahead_cache.py:349-373).  d_tokens[n]; if d_n != NULL the live length is
 * min(*d_n, n) read on the device.  mode PIA_MODE_INPUT needs 0 <= idx < n_input_slots.
 * final != 0 runs reset_input_freqs(idx) + squeeze_branch_counts() afterwards (:371-373). */
int pia_trie_put(pia_trie_t *t, const int32_t *d_tokens, int n, const int32_t *d_n, int branch_length, int mode,
                 int idx, int final, void *stream);
/* Tree.put (lookahead_cache.py:33-63) on the tree keyed by `tree_token` alone (created when absent). */
int pia_trie_tree_put(pia_trie_t *t, int tree_token, const int32_t *d_tokens, int n, int mode, int idx, void *stream);
/* LookaheadCache.stream_put (lookahead_cache.py:375-406); the per-idx carry buffer lives on the device.
 * d_idx != NULL: the request idx is read on the device (*d_idx, must be in [0, n_input_slots)) instead of `idx` -
 * the batched loop's slot -> request map changes as requests finish (pretrained_model_batch.py:937-980). */
int pia_trie_stream_put(pia_trie_t *t, const int32_t *d_tokens, int n, const int32_t *d_n, int branch_length, int idx,
                        const int32_t *d_idx, int final, void *stream);

/* LookaheadCache.hier_get / one_get -> Tree.get / get_one_branch (lookahead_cache.py:408-439, 490-517,
 * 65-144, 171-222), `batch` independent queries in one launch.
 *   d_queries : [batch, q_stride] int32;  d_qlen : [batch] valid tokens per row
 *   d_idx     : [batch] request idx per row, or NULL -> `idx` for all rows
 *   max_seq_length > 0 (PIA_GET_TAIL only): branch_length is clamped on the device to
 *               min(branch_length, max_seq_length - len - 1)   (pretrained_model.py:680);
 *               d_max_seq_length != NULL: the limit is read on the device (one CUDA graph for every max_length)
 * outputs (per row b):
 *   d_out_ids  [batch, decoding_length] ; d_out_mask [batch, decoding_length, W], W = ceil(decoding_length/64)
 *   d_out_n    [batch] number of nodes incl. the root (>= 1 unless the query was empty)
 *   d_out_sizes[batch, 2] ; d_out_nsizes[batch] length of python's `sizes` list (0, 1 or 2)
 *   d_status   [batch] PIA_OK or PIA_ERR_INDEX / PIA_ERR_CAPACITY for that row */
int pia_trie_get(pia_trie_t *t, const int32_t *d_queries, const int32_t *d_qlen, int batch, int q_stride,
                 int max_query_length, const int32_t *d_idx, int idx, int decoding_length, int branch_length,
                 int min_input_size, int min_output_size, int mode, int kind, int flags, int max_seq_length,
                 const int32_t *d_max_seq_length, int32_t *d_out_ids, uint64_t *d_out_mask, int32_t *d_out_n,
                 int32_t *d_out_sizes, int32_t *d_out_nsizes, int32_t *d_status, void *stream);

/* Tree.squeeze :295-301 and Tree.reset_input_freq :320-333 of the single tree keyed by `token` (no touched-tree
 * bookkeeping, no 1024-trees threshold: the per-tree methods callers may invoke directly) */
int pia_trie_tree_squeeze(pia_trie_t *t, int token, void *stream);
int pia_trie_tree_reset_input_freq(pia_trie_t *t, int token, int idx, void *stream);
/* reset_input_freqs :566-570 ; squeeze_branch_counts :572-576 ; fresh :563-564 */
int pia_trie_reset_input_freqs(pia_trie_t *t, int idx, void *stream);
int pia_trie_squeeze_branch_counts(pia_trie_t *t, void *stream);
int pia_trie_fresh(pia_trie_t *t, void *stream);
/* Synchronises `stream`. */
int pia_trie_stats(pia_trie_t *t, pia_trie_stats_t *h_out, void *stream);
/* the sticky error bits (pia_trie_stats_t.error_flags: node / edge pool exhausted, carry buffer overflow, ...) copied to
 * *d_out on the stream, capturable: the generation loops put it into their per-step record so that a trie that stopped
 * learning (inserts dropped, lookahead_cache.py has no such failure mode) is reported instead of going unnoticed. */
int pia_trie_copy_error_flags(pia_trie_t *t, int32_t *d_out, void *stream);
/* per-tree counters Tree.n_node / n_output_node (lookahead_cache.py:29-30); -1 when the tree is absent. Synchronous. */
int pia_trie_tree_counters(pia_trie_t *t, int token, int64_t *h_n_node, int64_t *h_n_output_node, void *stream);

/* Storage reclamation (the reference relies on Python's garbage collection after Tree._squeeze pops nodes,
 * lookahead_cache.py:302-310, and on dict growth): copies the reachable forest to the front of the pools (host round
 * trip), child order, counts, per-tree counters and touched-tree lists unchanged; clears the pool-exhausted error bits.
 * h_nodes_before / h_nodes_after (optional) receive the node-pool fill before and after.  Synchronous, between requests. */
int pia_trie_compact(pia_trie_t *t, int64_t *h_nodes_before, int64_t *h_nodes_after, void *stream);

/* Persistence (LookaheadCache.save_mem / load_mem, lookahead_cache.py:578-587): the forest as raw pools in HOST
 * memory.  Node record (32 bytes): {int32 token, int32 n_child, int32 child, int32 cap, double fo, float fi, int32 aux};
 * cap == 0: `child` is the node id of the only child, else the offset of a block of (int32 token, int32 node) entries,
 * children in insertion order.  h_root_of / h_n_node / h_n_out are indexed by first token ([vocab_capacity]).
 * All three synchronise `stream`. */
int pia_trie_export_sizes(pia_trie_t *t, int64_t *n_nodes, int64_t *n_edges, void *stream);
int pia_trie_export(pia_trie_t *t, void *h_nodes, int64_t n_nodes, void *h_edges, int64_t n_edges, int32_t *h_root_of,
                    int32_t *h_n_node, int32_t *h_n_out, void *stream);
int pia_trie_import(pia_trie_t *t, const void *h_nodes, int64_t n_nodes, const void *h_edges, int64_t n_edges,
                    const int32_t *h_root_of, const int32_t *h_n_node, const int32_t *h_n_out, void *stream);

/* ============================================================================================
 * Request slots of one verify step.
 *   - the per-request loop (common/pretrained_model.py:947-1268, bs == 1 :1152) runs ONE slot;
 *   - the batched loop (common/pretrained_model_batch.py:1002-1330) runs one slot per active request: every request
 *     drafts decoding_length // active nodes (:713), so all slots together still fill <= max_nodes activation rows;
 *   - a prefill pass runs one slot per 64-row chain chunk of the same prompt (kv_slot_stride == 0: the chunks share
 *     one cache and chunk c sees the rows chunk c-1 appended).
 * Slot s owns rows [s * rows_per_slot, (s + 1) * rows_per_slot) of every activation buffer (qkv, q, attention out,
 * logits) and of the draft buffers (ids, mask rows); its KV cache starts kv_slot_stride elements after slot s-1's.
 * All arrays are DEVICE memory read at kernel run time, so one captured CUDA graph serves every prompt length,
 * padding and max_length.
 * ============================================================================================ */
typedef struct {
  int32_t batch;                /* number of slots, >= 1                                                       */
  int32_t rows_per_slot;        /* rows reserved per slot; batch * rows_per_slot <= rows of the buffers        */
  const int32_t *d_n;           /* [batch] live draft nodes of the slot (<= rows_per_slot; 0 = idle slot)       */
  const int32_t *d_prefix_len;  /* [batch] P: tokens of the slot already in its KV cache                        */
  const int32_t *d_pad_len;     /* [batch] left-pad columns [0, pad) masked for every row (:1123-1131); NULL = 0 */
  int64_t kv_slot_stride;       /* elements between the [n_layers, n_kv_heads, max_seq, head_dim] caches of
                                   consecutive slots (0: all slots address the same cache)                     */
  int32_t kv_first_slot;        /* TMA-addressed kernels (pia_tree_attn_fwd): cache index slot 0 addresses; the
                                   pointer-addressed ones take the pointer of that cache instead               */
} pia_slots_t;

/* ============================================================================================
 * Tree-masked attention (verify forward)
 *   models/llama/modeling_llama.py:584-588 (mask -> positions) and :243-308 (eager attention);
 *   mistral/modeling_mistral.py:979-982,241-320; pretrained_model.py:725-734 (mask builder).
 * The [n, P+n] 0/1 mask is never materialised: prefix columns [pad_len, P) are visible to every
 * row, the last n columns follow the per-row ancestor bit mask.
 * ============================================================================================ */
typedef struct pia_attn_plan pia_attn_plan_t;

typedef struct {
  int32_t n_q_heads, n_kv_heads, head_dim; /* head_dim 128 or 64                                     */
  int32_t max_seq;                         /* rows of the KV cache (max_length + decoding_length + 1) */
  int32_t max_nodes;                       /* 64 (W=1) or 128 (W=2)                                  */
  int32_t n_layers;
  int32_t kv_split_max;                    /* upper bound of KV splits per head (0 = auto)            */
  int32_t n_slots;                         /* KV caches behind the plan (0/1 = one; batched loop: one per request) */
} pia_attn_config_t;

/* d_k_cache / d_v_cache : [n_slots, n_layers, n_kv_heads, max_seq, head_dim] bf16, owned by the caller for the
 * plan's lifetime (TMA descriptors are encoded over them). Synchronous; not capturable. */
int pia_attn_plan_create(const pia_attn_config_t *cfg, void *d_k_cache, void *d_v_cache, pia_attn_plan_t **out);
int pia_attn_plan_destroy(pia_attn_plan_t *p);
/* diagnostics: per-CTA phase timestamps (16 x uint64 globaltimer values per CTA of the last launch), or NULL to
 * disable; grid geometry of the plan (n_split x n_groups CTAs). */
int pia_attn_plan_set_debug(pia_attn_plan_t *p, void *d_timestamps);
int pia_attn_plan_grid(const pia_attn_plan_t *p, int *n_split, int *n_groups);

/* One layer of tree attention over the cache(s), every slot of the table in one launch (gridDim.z = slot; rows
 * [P_s, P_s + n_s) of slot s's cache must already hold this step's K/V, RoPE applied).
 *   d_q    : [batch * rows_per_slot, n_q_heads, head_dim] bf16 (rows >= n_s of a slot are ignored and not written)
 *   d_mask : [batch * rows_per_slot, W] uint64 ancestor rows (bit j = draft node j of the SAME slot)
 *   d_out  : [batch * rows_per_slot, n_q_heads, head_dim] bf16
 * softmax scale = 1/sqrt(head_dim) * `scale_mul` (1.0 for the reference models).  Needs no workspace: KV splits are
 * merged through the distributed shared memory of a thread-block cluster. */
int pia_tree_attn_fwd(pia_attn_plan_t *p, int layer, const void *d_q, const uint64_t *d_mask, const pia_slots_t *slots,
                      float scale_mul, void *d_out, void *stream);

/* The same attention with RoPE + KV append folded in (modeling_llama.py:261-268 + :272-292 in one launch): d_qkv is the
 * fused projection output [batch * rows_per_slot, (Hq + 2*Hkv) * D] bf16; Q and the draft nodes' K are rotated at the
 * nodes' positions (tables as pia_rope_kv_append), the n draft keys are one extra tile staged in shared memory, the
 * TMA tiles only cover the cached prefix [0, P), and one CTA per KV head appends the rotated K / V rows to cache rows
 * [P, P + n) for the steps to come.  Same arithmetic as pia_rope_kv_append + pia_tree_attn_fwd (the cache rows are bit
 * identical, the output differs by the fp32 summation order of the tiles).  Needs one cache per slot
 * (batch == 1 or kv_slot_stride != 0): prefill chunks that share a cache use the two-kernel path. */
int pia_tree_attn_fused_fwd(pia_attn_plan_t *p, int layer, const void *d_qkv, const void *d_cos, const void *d_sin,
                            int max_pos, const uint64_t *d_mask, const pia_slots_t *slots, float scale_mul, void *d_out,
                            void *stream);

/* ============================================================================================
 * Weight-streaming GEMM of the verify forward: Y[t, n] = sum_k X[t, k] W[n, k]  (X: <= 64 draft rows, W = an
 * nn.Linear weight [N, K] bf16), i.e. the projections of modeling_llama.py:254-256, :303, :185-186, :769.
 * TMA + tcgen05, weights read once; see csrc/gemm_ws.cu.
 * ============================================================================================ */
typedef struct pia_gemm_plan pia_gemm_plan_t;
/* d_x : [x_rows >= 64, K] bf16 activation buffer the plan's TMA descriptor is bound to; K % 64 == 0.
 * split_k > 1 splits the K range over CTAs (for projections with few 128-row weight tiles) and yields fp32 partial
 * slices; split_k == -1 (tiled weights only) selects stream-K: the (tile, k-chunk) units are cut into one equal
 * contiguous range per SM and tiles spanning CTAs are fixed up in-kernel (bf16 output, deterministic); split_k == -2,
 * -4 or -8: the 2 / 4 / 8 K splits of a weight tile run as one thread-block cluster and reduce their fp32 partials through
 * distributed shared memory in split order (bf16 output, deterministic, no fp32 slices in HBM). Synchronous. */
/* w_tiled != 0: d_w holds the same weight re-laid out as [N/128][K/64] contiguous blocks of 128 rows x 64 k
 * (W.view(N/128,128,K/64,64).permute(0,2,1,3)), so that every CTA streams one contiguous slab of HBM. */
int pia_gemm_plan_create(const void *d_w, int N, int K, const void *d_x, int x_rows, int split_k, int w_tiled,
                         pia_gemm_plan_t **out);
/* Grouped GEMM, one launch for all MoE experts (mixtral/modeling_mixtral.py:692-759): for g in [0, groups):
 *   out[g] ([64, N] bf16, consecutive) = X[:, g*K : (g+1)*K] @ W[g]^T,   W : [groups * N, K] bf16 row-major (the stacked
 * expert weights), X : [x_rows >= 64, groups * K] bf16.  N % 128 == 0, K % 64 == 0.  Run with pia_gemm_run. */
int pia_gemm_plan_create_grouped(const void *d_w, int groups, int N, int K, const void *d_x, int x_rows,
                                 pia_gemm_plan_t **out);
int pia_gemm_plan_destroy(pia_gemm_plan_t *g);
int pia_gemm_plan_splits(const pia_gemm_plan_t *g);
/* on == 0: launch this plan without the programmatic-dependent-launch attribute, i.e. as a plain kernel boundary that
 * neither starts before its predecessor has finished nor lets its successor start early (how a library GEMM behaves in
 * the chain); default on. */
int pia_gemm_plan_set_pdl(pia_gemm_plan_t *g, int on);
/* fused SiLU(gate) * up epilogue (modeling_llama.py:185-186): the weight must be laid out so that every 128-row tile
 * holds 64 gate rows followed by the 64 up rows of the same columns; d_out of pia_gemm_run is then [rows, N/2]. */
int pia_gemm_plan_set_silu(pia_gemm_plan_t *g, int on);
/* FP8 weight-only plans: the same projections (modeling_llama.py:254-256, :303, :185-186 and the Mixtral experts,
 * mixtral/modeling_mixtral.py:668-683) with the weight stored as e4m3 plus one fp32 scale per output channel, quantised
 * once at load time:
 *   s[n] = max_k |W[n, k]| / 448 (1 for an all-zero row),   Wq = e4m3(W / s) round-to-nearest-even, saturating at 448,
 *   Y[t, n] = bf16( s[n] * sum_k X[t, k] Wq[n, k]  (+ b[n]) )
 * X is bf16; products and sums are fp32 (MMA accumulation); the bias, where given, is added in fp32 and the result is
 * rounded to bf16 exactly once.  d_w_tiled_f8 holds Wq as [N/128][K/128] contiguous 16 KB blocks of 128 rows x 128 k
 * (Wq.view(N/128,128,K/128,128).permute(0,2,1,3)); N % 128 == 0, K % 128 == 0.  d_scale: [N] fp32; d_bias: [N] bf16 or
 * NULL.  d_x: [x_rows, K] bf16 with 1 <= x_rows <= 256; the plan launches 64, 128 or 256 token rows (the smallest that
 * covers x_rows).  split_k as for pia_gemm_plan_create except stream-K (-1); fp32 slices are [splits][64|128|256][N],
 * every slice scaled and the bias in slice 0.  SiLU*up is not available on these plans. */
int pia_gemm_plan_create_fp8(const void *d_w_tiled_f8, const float *d_scale, const void *d_bias, int N, int K,
                             const void *d_x, int x_rows, int split_k, pia_gemm_plan_t **out);
/* grouped fp8 plan (MoE experts): d_w_tiled_f8 = the groups' tiled e4m3 weights back to back, d_scale [groups, N],
 * X [x_rows, groups * K]; out[g] is [64|128|256, N] bf16, consecutive.  No bias, no K split. */
int pia_gemm_plan_create_grouped_fp8(const void *d_w_tiled_f8, const float *d_scale, int groups, int N, int K,
                                     const void *d_x, int x_rows, pia_gemm_plan_t **out);
/* splits == 1: d_out is bf16 [rows_cap, N]; splits > 1: d_out is fp32 [splits][64][N] partial slices (sum them in
 * slice order, e.g. with pia_rmsnorm_partials).  rows <= 64 rows are written (rows <= x_rows for fp8 plans). */
int pia_gemm_run(pia_gemm_plan_t *g, int rows, void *d_out, void *stream);

/* ============================================================================================
 * Fused elementwise pieces of the verify forward (all bf16 I/O, fp32 math)
 * ============================================================================================ */
/* RMSNorm (modeling_llama.py:76-90): y = (w * (x * rsqrt(mean(x^2)+eps)).to(bf16)) ; rows x hidden.
 * If d_residual_in != NULL: x <- x + residual_in first and the sum is written to d_residual_out. */
int pia_rmsnorm(const void *d_x, const void *d_residual_in, const void *d_weight, float eps, int rows, int hidden,
                void *d_residual_out, void *d_y, void *stream);
/* same, with x given as `n_parts` fp32 split-K slices of pia_gemm_run ([n_parts][part_stride] floats, row-major
 * [rows, hidden] inside a slice): x = bf16(sum of slices), i.e. what a bf16 GEMM output would have held */
int pia_rmsnorm_partials(const float *d_x_parts, int n_parts, int64_t part_stride, const void *d_residual_in,
                         const void *d_weight, float eps, int rows, int hidden, void *d_residual_out, void *d_y,
                         void *stream);
/* RoPE at tree positions + KV append (modeling_llama.py:261-268, 93-169; batched: modeling_llama_batch.py:375-405;
 * position of node i of slot s = max(P_s - pad_s, 0) + depth_i = rowsum(mask) - 1, :587).
 * d_qkv : [batch * rows_per_slot, (Hq + 2*Hkv) * D] bf16 (fused projection output).  d_cos / d_sin : [max_pos, D/2]
 * bf16 tables (cos/sin already rounded to the model dtype exactly as LlamaRotaryEmbedding.forward :111-127 returns
 * them).  Writes q (rotated) to d_q_out [batch * rows_per_slot, Hq, D] and K (rotated) / V to cache rows P_s + i of
 * the layer's [Hkv, max_seq, D] planes of slot s (d_*_cache_layer + s * kv_slot_stride). */
int pia_rope_kv_append(const void *d_qkv, const uint64_t *d_mask, int mask_words, const pia_slots_t *slots,
                       int n_q_heads, int n_kv_heads, int head_dim, const void *d_cos, const void *d_sin, int max_pos,
                       void *d_q_out, void *d_k_cache_layer, void *d_v_cache_layer, int max_seq, void *stream);
/* SiLU(gate) * up (modeling_llama.py:185-186). d_gate_up : [rows, 2*inter] (gate | up) -> d_out [rows, inter] */
int pia_silu_mul(const void *d_gate_up, int rows, int inter, void *d_out, void *stream);
/* embedding gather for the draft nodes: d_out[i] = table[d_ids[i]] (rows >= *d_n are zero filled) */
int pia_embed_gather(const void *d_table, const int32_t *d_ids, const int32_t *d_n, int rows, int hidden, void *d_out,
                     void *stream);
/* MoE combine (mixtral/modeling_mixtral.py:734-759, dense restatement): d_out[t] = sum_e d_expert_out[e][t] * w[t][e]
 * in expert-index order, product and partial sums rounded to bf16 as the eager bf16 loop does.
 * d_expert_out : [n_experts, rows_cap, hidden] bf16; d_weights : [rows, n_experts] bf16 routing weights (0 = expert not
 * selected by that token); d_out : [rows, hidden] bf16. */
int pia_moe_combine(const void *d_expert_out, const void *d_weights, int n_experts, int rows, int rows_cap, int hidden,
                    void *d_out, void *stream);
/* MoE router (mixtral/modeling_mixtral.py:721-727): gate Linear (bf16) -> fp32 softmax -> top-k -> renormalise -> bf16,
 * written densely: d_dense_out [rows, n_experts] holds the routing weight of the selected experts and 0 elsewhere.
 * d_y [rows, hidden] bf16, d_gate_weight [n_experts, hidden] bf16. */
int pia_moe_router(const void *d_y, const void *d_gate_weight, int rows, int hidden, int n_experts, int top_k,
                   void *d_dense_out, void *stream);
/* L2 prefetch of immutable weights (no reference counterpart: the reference's eager loop leaves HBM idle while the
 * small kernels of a layer - RoPE, attention, norms - run; modeling_llama.py:272-292 sits between the qkv and the o
 * projection).  Issues cp.async.bulk.prefetch.L2 for n_ranges ranges of range_bytes (multiple of 16) that start
 * stride_bytes apart at d_base, chunk-interleaved across the ranges (every range gets its first bytes first), paced
 * to gbytes_per_s (0 = as fast as the grid - one warp per SM - issues).  A hint only: no result, nothing to wait for; meant for a side
 * stream / parallel graph branch next to the kernels whose HBM idle time it fills. */
int pia_l2_prefetch(const void *d_base, int64_t n_ranges, int64_t stride_bytes, int64_t range_bytes, float gbytes_per_s,
                    void *stream);

/* ============================================================================================
 * Accept + KV compaction + sequence update
 *   pretrained_model.py:764-892 (longest-prefix accept walk, greedy), :894-945 (KV compaction),
 *   RepetitionPenaltyLogitsProcessor semantics of the installed transformers (call sites :786,:834).
 * ============================================================================================ */
typedef struct {
  int32_t vocab;               /* logits row length                                              */
  int32_t max_nodes;
  float repetition_penalty;    /* 1.0 = none                                                     */
  int32_t n_eos; int32_t eos[8];
  int32_t max_length;          /* generation stops when seq_len >= max_length (MaxLengthCriteria); overridden by
                                  *d_max_length when that pointer is given                          */
  int32_t bound_walk;          /* 1: the walk accepts at most max_length - seq_len tokens, the batched loop's
                                  range(-1, min(max_branch_length, max_length - cur - 2)) (pretrained_model_batch.py:862);
                                  0: unbounded (the per-request loop clamps the draft depth instead, :680) */
} pia_accept_config_t;

/* Row arg-max of the (penalised) logits of every draft node, then the walk of :827-860 (batched loop:
 * pretrained_model_batch.py:810-905), one slot per request (slot layout as pia_slots_t).
 *   d_logits : [batch * rows_per_slot, vocab] bf16 ; d_ids [batch * rows_per_slot] / d_mask / d_n [batch] : the drafts
 *   d_seq : [batch, seq_stride] int32 token sequences (prompt + generated), d_seq_len [batch] their lengths; the
 *           accepted tokens are appended and d_seq_len advanced.
 *   d_max_length : device int overriding cfg->max_length, or NULL
 *   d_rng : NULL = greedy arg-max (:839).  Else multinomial accept (do_sample, :835-837): {seed, step counter} in
 *           device memory; every node draws from softmax(its penalised logits) by the Gumbel-max construction and the
 *           counter is advanced once per call.  The draws are not torch.multinomial's stream: parity is distributional.
 *   d_accept_tokens [batch, cfg->max_nodes] accepted tokens (draft matches + bonus); d_accept_count [batch] (edl)
 *   d_accept_nodes  [batch, cfg->max_nodes] draft node index (slot relative) whose logits produced each token
 *                   (logit_indices :845)
 *   d_prefix_len [batch] : P, advanced to P + count on return
 *   d_finished   [batch] : set to 1 when an eos was accepted or max_length reached (:1225-1231)
 * batch * rows_per_slot <= cfg->max_nodes.  A slot with d_n == 0 is idle (count 0). */
int pia_accept(const pia_accept_config_t *cfg, const void *d_logits, const int32_t *d_ids, const uint64_t *d_mask,
               int mask_words, int batch, int rows_per_slot, const int32_t *d_n, int32_t *d_seq, int32_t *d_seq_len,
               int seq_stride, const int32_t *d_max_length, uint32_t *d_rng, int32_t *d_accept_tokens,
               int32_t *d_accept_count,
               int32_t *d_accept_nodes, int32_t *d_prefix_len, int32_t *d_finished, void *d_workspace, void *stream);
int64_t pia_accept_workspace_bytes(const pia_accept_config_t *cfg);

/* KV compaction (pretrained_model.py:863-875, 894-907; batched :907-918, 986-989) in place: cache row
 * P_old + node -> row P_old + k for the k-th accepted draft node, all layers, K and V, every slot.
 * d_*_cache : [batch (stride kv_slot_stride elements), n_layers, n_kv_heads, max_seq, head_dim];
 * d_accept_nodes [batch, nodes_stride]; d_prefix_len [batch] holds the values *after* pia_accept. */
int pia_kv_compact(void *d_k_cache, void *d_v_cache, int n_layers, int n_kv_heads, int max_seq, int head_dim, int batch,
                   int64_t kv_slot_stride, const int32_t *d_accept_nodes, int nodes_stride,
                   const int32_t *d_accept_count, const int32_t *d_prefix_len, void *stream);

/* ============================================================================================
 * FLOOD `Spec` integration (SURVEY.md 8f-4): the hash-table lookahead draft of flood/flood/utils/speculative.py:23-124
 * (class Lookahead) whose Triton kernels live in flood/flood/ops/draft.py.  Tables are FLOOD's own: freq_table
 * float32 [table_size], draft_table int32 [table_size, branch_length]; a 2-token context (p0, p1) owns the
 * branch_count slots from bucket (p0 * vocab + p1) % (table_size - branch_count).
 * ============================================================================================ */
/* update_draft_table (draft.py:168-204, kernel :92-165): every position p of d_tokens[token_count] with p + 4 <=
 * token_count inserts / reinforces the branch tokens[p+2 : p+2+branch_length] under context (tokens[p], tokens[p+1]);
 * all slots of the bucket decay by 1/2 per update.  Positions are applied in order. */
int pia_flood_update_draft_table(const int32_t *d_tokens, int token_count, float *d_freq_table, int32_t *d_draft_table,
                                 int64_t table_size, int branch_length, int branch_count, int vocab, void *stream);
/* retrieve_draft_table (draft.py:352-402, kernel :278-349): d_queries [batch, 2] -> d_out_tokens
 * [batch, retrieve_count * branch_length + 1] (zero-filled by the caller): [p1, branch 0, branch 1, ...], the
 * retrieve_count most established branches by the 64, 32, ..., 0.5 frequency ladder. */
int pia_flood_retrieve_draft_table(const int32_t *d_queries, int batch, const float *d_freq_table,
                                   const int32_t *d_draft_table, int64_t table_size, int vocab, int branch_length,
                                   int branch_count, int retrieve_count, int32_t *d_out_tokens, void *stream);
/* verify_draft (draft.py:491-543, kernel :406-488): d_input_ids / d_next_ids [batch, branch_count * branch_length] (the
 * flattened draft layout of retrieve_draft_table and the model's next token at each of its positions) -> the longest
 * accepted branch: d_output_ids [batch, branch_length + 1], d_cache_src / d_cache_dst [batch * branch_length]
 * (all three filled with -1 by the caller); d_cache_offsets [batch] = first cache row of each request's draft. */
int pia_flood_verify_draft(const int32_t *d_input_ids, const int32_t *d_next_ids, const int32_t *d_cache_offsets, int batch,
                           int branch_count, int branch_length, int32_t *d_output_ids, int32_t *d_cache_src,
                           int32_t *d_cache_dst, void *stream);
/* update_draft_cache (draft.py:562-570, kernel :547-559): cache row d_src[i] -> row d_dst[i] for every i with
 * d_src[i] >= 0 and d_src[i] != d_dst[i]; d_cache is [rows, row_bytes]. */
int pia_flood_update_draft_cache(void *d_cache, int64_t row_bytes, const int32_t *d_src, const int32_t *d_dst, int count,
                                 void *stream);

#ifdef __cplusplus
}
#endif
#endif /* PIA_B200_H_ */
