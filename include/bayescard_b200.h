/*
 * bayescard_b200 -- C ABI of the B200-native exact-inference hot path of wuziniu/BayesCard.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI: its seam for this
 * path is the Python object assigned to ``Bayescard_BN.infer_machine`` (reference
 * Models/Bayescard_BN.py:141), whose two methods are
 *     VariableEliminationJIT.query(query, n_distinct)                 Pgmpy/inference/ExactInference.py:112-197
 *     VariableEliminationJIT.expectation(query, fanout_attrs, n_distinct)            ...:199-287
 * and whose constructor consumes the topologically aligned CPD list
 *     VariableEliminationJIT.__init__(model, cpds, topological_order, ...)           ...:25-40
 *     Bayescard_BN.align_cpds_in_topological()                        Models/Bayescard_BN.py:340-358
 * Each entry point below names the reference interface it replaces.  All pointers are plain
 * host or device addresses; no torch / numpy / C++ types cross this boundary.  The host side above
 * it (bayescard_b200 / *.py) binds these symbols with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every function returning int returns BC_OK (0) on success, a negative BC_E* code otherwise;
 *     bc_last_error() then holds a human-readable message (thread local).
 *   - there is NO CPU fallback: if no CUDA device / kernel image is usable the call fails.
 *   - a bc_model's tree is fixed at creation and its CPTs change only through bc_model_update;
 *     bc_query_batch* are stream ordered and may be called
 *     concurrently on different models / devices (one host thread per GPU).
 *   - node indices are TOPOLOGICAL (parents before children, node 0 = root), the order of
 *     align_cpds_in_topological() restricted to the root's component.
 */
#ifndef BAYESCARD_B200_H
#define BAYESCARD_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define BC_API __attribute__((visibility("default")))
#else
#define BC_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define BC_OK 0
#define BC_EINVAL (-1)   /* bad argument                                   */
#define BC_ECUDA (-2)    /* CUDA runtime / driver error                    */
#define BC_ENOMEM (-3)   /* host or device allocation failed               */
#define BC_ECOMPILE (-4) /* NVRTC unavailable or specialised build failed  */
#define BC_ELIMIT (-5)   /* model exceeds what the selected kernel supports */

/* ---- query descriptor formats (one row per query, nodes in topological order) ------------------
 * RANGE_U8   2*n_nodes bytes, row stride = round_up(2*n_nodes, 4):  lo_0,hi_0,lo_1,hi_1,...
 *            w_v[c] = 1 for lo_v <= c <= hi_v, else 0 (an unconstrained column is [0, card-1];
 *            lo > hi selects nothing).  Requires card <= 256.  This is the compact form of a
 *            conjunction of range / equality predicates over the discretised bins, i.e. the output
 *            of Bayescard_BN.query_decoding (Models/Bayescard_BN.py:279-325) when every predicate
 *            is a contiguous bin interval with n_distinct weights 1.
 * RANGE_U16  same with uint16 bounds (card <= 65536), row stride 4*n_nodes bytes.
 * DENSE_F32  one fp32 weight per (node, state): node v occupies round_up(card_v,4) floats starting
 *            at bc_model_dense_offset(v); row stride = bc_model_dense_width() floats.  Carries the
 *            general output of query_decoding (IN lists, fractional n_distinct weights).
 * BITS       one bit per (node, state): node v owns bits [bc_model_bits_offset(v), +card_v) of the row,
 *            nodes tightly packed in topological order, row stride = bc_model_desc_stride() bytes
 *            (a multiple of 16).  w_v[c] = bit ? 1 : 0; an unconstrained column has all bits set
 *            (bc_model_bits_default() returns that row).  Carries every predicate whose n_distinct
 *            weights are all 1: ranges, equality and IN lists over the discretised bins.  This is
 *            the format the specialised kernel is fastest on.
 * SPARSE     (host-facing, bc_query_batch_sparse*) CSR: row_off[nq+1] (uint32, in entries) and 32-bit
 *            entries  col[0:15) | cont<<15 | lo<<16 | hi<<24 : states lo..hi of column col; cont=1
 *            ORs into the column's mask built so far (IN lists), cont=0 replaces it.  Columns that
 *            are not mentioned are unconstrained -- the shape of the reference's query dict
 *            (Evaluation/cardinality_estimation.py:60-111).  Needs card <= 256.  Expanded to BITS
 *            rows on the device; only PCIe sees this form.
 * For every format an optional fan-out bitmask (mask_words = ceil(n_nodes/32) uint32 per query,
 * bit v set = multiply w_v by fanouts[v]) implements expectation(); a predicate on a fan-out
 * column wins (ExactInference.py:209,:238), so the host clears the bit for predicated columns.
 */
#define BC_DESC_RANGE_U8 0
#define BC_DESC_RANGE_U16 1
#define BC_DESC_DENSE_F32 2
#define BC_DESC_BITS 3

/* ---- kernel selection ------------------------------------------------------------------------- */
#define BC_KERNEL_AUTO 0     /* fused tensor-core kernel for models of > 15k CPT entries, else the
                                specialised kernel if the model has one, else generic        */
#define BC_KERNEL_GENERIC 1  /* K1: warp per query, CPT arena staged in shared memory by TMA  */
#define BC_KERNEL_SPEC 2     /* K-spec: per-model straight-line kernel, thread per query      */
#define BC_KERNEL_GEMM 3     /* K2: per-edge batched path for large domains, tcgen05 3xTF32 GEMM
                                where the edge shape allows, FP32 SIMT GEMM otherwise; RANGE_* rows */
#define BC_KERNEL_GEMM_SIMT 4 /* K2 with the FP32 SIMT GEMM only (the comparator for K2)      */
#define BC_KERNEL_FUSED 5    /* K3: whole tree per 128-query tile on the tensor cores (tcgen05 3xTF32), messages in
                                tensor memory; trees of <= 128 columns with domains <= 256 states (<= 128 below the root) whose
                                live messages fit the 512 TMEM columns, else BC_ELIMIT */

typedef struct bc_model bc_model;

/* Replaces VariableEliminationJIT.__init__ + align_cpds_in_topological (ExactInference.py:25-40,
 * Bayescard_BN.py:340-358): uploads the topologically ordered CPTs as ONE 16 B-aligned fp32 arena.
 *   parent[v]   topological index of the parent, -1 for v = 0 (the root); parent[v] < v
 *   card[v]     number of states
 *   cpt_off[v]  offset (in floats) of T_v in cpt_arena; T_v[c][p] at cpt_off[v] + c*stride[v] + p
 *   stride[v]   row stride in floats (>= card[parent[v]], multiple of 4); root: one row of card[0]
 *   fan_off[v]  offset (floats) of fanouts[v] (card[v] floats) in fan_arena, or -1
 * Host pointers; the arrays are copied.  device = CUDA ordinal. */
BC_API int bc_model_create(int device, int n_nodes, const int32_t* parent, const int32_t* card,
                    const int64_t* cpt_off, const int32_t* stride, const float* cpt_arena,
                    size_t arena_floats, const int64_t* fan_off, const float* fan_arena,
                    size_t fan_floats, bc_model** out);
/* The same model from a flat, versioned, mmap-able file written once from the pickle (bayescard_b200/loader.py:
 * TreeModel.save_flat; layout in csrc/bc_modelfile.cc): replaces `pickle.load` of the Bayescard_BN object
 * (Models/BN_single_model.py:207-223) + init_inference_method (Models/Bayescard_BN.py:122-142) for a serving process
 * that must not unpickle third-party classes.  Validates magic, version and every section bound. */
BC_API int bc_model_create_from_file(int device, const char* path, bc_model** out);
BC_API void bc_model_destroy(bc_model* m);

BC_API int bc_model_n_nodes(const bc_model* m);
BC_API int bc_model_device(const bc_model* m);
/* DENSE_F32 row geometry */
BC_API int64_t bc_model_dense_width(const bc_model* m);
BC_API int64_t bc_model_dense_offset(const bc_model* m, int node);
/* BITS row geometry: first bit of node v; the all-selected row (row stride bytes, host copy) */
BC_API int64_t bc_model_bits_offset(const bc_model* m, int node);
BC_API int bc_model_bits_default(const bc_model* m, void* row_host, size_t row_bytes);
/* row stride in BYTES of a descriptor format for this model */
BC_API int64_t bc_model_desc_stride(const bc_model* m, int desc_format);
/* ALGORITHMIC flop per query of the dense tree: 2 * sum_{v != root} card(v)*card(parent(v)) */
BC_API int64_t bc_model_flops_dense(const bc_model* m);

/* Build (or load from the on-disk cache) the per-model specialised kernel (K-spec): straight-line
 * sm_100a code for this tree with the CPT entries as FFMA immediates, compiled with NVRTC.
 * cache_dir may be NULL (no cache).  Returns BC_ECOMPILE if NVRTC is missing or the build fails;
 * the generic kernel keeps working. */
BC_API int bc_model_specialize(bc_model* m, const char* cache_dir);
BC_API int bc_model_has_spec(const bc_model* m);
/* Plan of the fused tensor-core kernel (K3) for this model, for inspection and tests (works on host-only models):
 *   info[8]  = {edges, TMEM columns allocated per CTA, CTAs per SM, shared memory bytes per CTA, first accumulator
 *               column, accumulator columns, column of the root's message, operand images in KB}
 *   edges    = per edge in schedule order {child, card(child), card(parent), parent states padded to 16, TMEM column of
 *               the child's message (-1: leaf), TMEM column of the parent's message, first message into the parent,
 *               ring steps}; may be NULL.
 * BC_ELIMIT (with the reason in bc_last_error) when K3 does not serve the model. */
BC_API int bc_model_fused_plan(bc_model* m, int32_t* info, int32_t* edges, size_t edges_capacity);
/* ... and its step sequence: sequence[i] = edge index (position in the schedule above) | 128 for a TAIL edge, which a CTA runs for
 * its PREVIOUS tile (the chain at the top of the tree is interleaved with the next tile's body); flags[e] per edge: bit 0 first /
 * bit 1 last edge of a run of consecutive edges into one parent, bit 2 the parent's message stays in the epilogue warps' registers
 * over the run.  *n_tail = number of tail edges (the last ones of the schedule).  Both arrays hold `edges` entries. */
BC_API int bc_model_fused_sequence(bc_model* m, uint8_t* sequence, uint8_t* flags, size_t capacity, int32_t* n_tail);
/* Write the generated CUDA source of the specialised kernel (host only, no GPU needed; used by the
 * ahead-of-time build and by tests).  Returns the number of bytes needed including the NUL. */
BC_API int64_t bc_model_spec_source(const bc_model* m, char* buf, size_t buf_bytes);
/* Hash that names the cache entry "<hash>.cubin" for this model + code generator version. */
BC_API uint64_t bc_model_spec_hash(const bc_model* m);
/* Attach an already compiled cubin (ahead-of-time build). */
BC_API int bc_model_load_cubin(bc_model* m, const void* image, size_t bytes);

/* Replaces the per-query loop `for q: infer_machine.query(q, nd)` / `.expectation(q, fan, nd)`
 * (Testing/BN_testing.py:21-46, Models/BN_ensemble_model.py:228-252) with ONE launch over a batch.
 * DEVICE pointers.  desc: n_queries rows in desc_format; fanout_mask: NULL or n_queries*mask_words
 * uint32; out_prob: n_queries fp32 = sum_x prod_v w_v[x_v] T_v[x_v, x_pa(v)].
 * stream: a cudaStream_t (NULL = legacy default stream). */
BC_API int bc_query_batch(bc_model* m, const void* desc, size_t n_queries, int desc_format,
                   const uint32_t* fanout_mask, float* out_prob, int kernel, void* stream);

/* Same with HOST buffers: chunks the batch, overlaps H2D / kernel / D2H on internal streams with
 * pinned staging buffers, returns when out_prob (host) is complete.  This is the end-to-end path
 * a caller of the reference-facing Python API goes through. */
BC_API int bc_query_batch_host(bc_model* m, const void* desc, size_t n_queries, int desc_format,
                        const uint32_t* fanout_mask, float* out_prob, int kernel);

/* ---- GROUP BY one column: per-state counts of a target node under each query's predicates ---------------------------
 * Replaces the per-value loop `[bn.query({**P, a: v}) for v in values]` over Bayescard_BN.query (Models/Bayescard_BN.py:496)
 * with ONE pass per query: for the target node t (topological index) and each row's weights w_v,
 *     out[q][b] = sum_{x : x_t = b} prod_v w_v[x_v] T_v[x_v, x_pa(v)]          b = 0 .. card(t) - 1
 * so w_t restricts the groups and sum_b out[q][b] is the out_prob[q] of bc_query_batch on the same row.  out is contiguous
 * fp32 [n_queries][card(t)].  Rows are BITS or DENSE_F32; there is no fan-out mask (fan-out columns are unconstrained:
 * bc_expectation_marginal_batch below with a NULL mask, which is what this call is).
 * DEVICE pointers, stream ordered.  kernel:
 *   BC_KERNEL_AUTO   the specialised marginal kernel of t when it is attached, otherwise the expansion below
 *   BC_KERNEL_SPEC   the specialised marginal kernel of t; BC_ECOMPILE when it is not attached
 *   any other id     the expansion through that kernel: every row becomes card(t) rows (the target's weights restricted
 *                    to one state each, built on the device in chunks of <= 256 MB), evaluated q-major by bc_query_batch
 * BC_EINVAL for a target outside [0, n_nodes), a RANGE_* or unknown format, or a host-only model; n_queries == 0 is BC_OK
 * with no launch.  Results below the fp32 range are not carried (no scaled form). */
BC_API int bc_marginal_batch(bc_model* m, const void* desc, size_t n_queries, int desc_format, int target, float* out,
                             int kernel, void* stream);
/* GROUP BY one column of an EXPECTATION: replaces `[bn.expectation({**P, a: v}, fan) for v in values]` over
 * Bayescard_BN.expectation (Models/Bayescard_BN.py:559) -- the per-value loop of a GROUP BY over a join, where every factor
 * is weighted by fan-out columns -- with ONE pass per query.  fanout_mask has bc_query_batch's layout and meaning: NULL or
 * n_queries * mask_words uint32, bit v of row q multiplies w_v by fanouts[v] (w'_v), and
 *     out[q][b] = sum_{x : x_t = b} prod_v w'_v[x_v] T_v[x_v, x_pa(v)]
 * so sum_b out[q][b] is bc_query_batch's out_prob[q] on the same row and mask.  Formats, kernel ids, argument checks and
 * error codes are bc_marginal_batch's; a NULL mask is exactly bc_marginal_batch.  The specialised marginal kernel reads the
 * mask in place (still one launch); the expansion repeats each mask row card(t) times next to the expanded rows (counted
 * in the 256 MB chunk bound) and passes it to bc_query_batch. */
BC_API int bc_expectation_marginal_batch(bc_model* m, const void* desc, size_t n_queries, int desc_format,
                                         const uint32_t* fanout_mask, int target, float* out, int kernel, void* stream);
/* Build (or load "<cache_dir>/marg_<hash>.cubin") the specialised marginal kernel of one target node: straight-line sm_100a
 * code like bc_model_specialize's, attached through the driver JIT; one module per target, kept on the model. */
BC_API int bc_model_specialize_marginal(bc_model* m, int target, const char* cache_dir);
/* Its generated PTX (host-only models too; returns the bytes needed including the NUL) and the hash that names its cache
 * entry (model, target and marginal generator version; 0 for a target out of range). */
BC_API int64_t bc_model_marginal_source(const bc_model* m, int target, char* buf, size_t buf_bytes);
BC_API uint64_t bc_model_marginal_hash(const bc_model* m, int target);

/* ---- GROUP BY two columns: per-(state, state) counts of two nodes a != b under each query's predicates ----------------
 * Replaces `[bn.query({**P, a: va, b: vb}) for va, vb in pairs]` -- card(a) * card(b) full evaluations per query -- with ONE
 * pass per query.  With bc_expectation_marginal_batch's weights w'_v (fan-out mask bit v multiplies w_v by fanouts[v];
 * NULL: no mask)
 *     out[q][i][j] = sum_{x : x_a = i, x_b = j} prod_v w'_v[x_v] T_v[x_v, x_pa(v)]        contiguous fp32 [n][card(a)][card(b)]
 * Both targets' own weights apply.  Summing over j gives bc_expectation_marginal_batch(a) on the same row and mask, over i
 * the same for b, over both bc_query_batch.  Rows are BITS or DENSE_F32.  DEVICE pointers, stream ordered.  kernel:
 *   BC_KERNEL_AUTO   the joint module of (a, b) when it is attached, otherwise the expansion below
 *   BC_KERNEL_SPEC   the joint module of (a, b); BC_ECOMPILE when it is not attached
 *   any other id     the expansion: every row becomes card(a) rows (a's weights restricted to one state each, the mask row
 *                    repeated; chunks of <= 256 MB), evaluated by bc_expectation_marginal_batch(b) with that kernel id
 * BC_EINVAL for a == b, a node outside [0, n_nodes), a RANGE_* or unknown format, NULL pointers or a host-only model;
 * n_queries == 0 is BC_OK with no launch.  Results below the fp32 range are not carried. */
BC_API int bc_joint_marginal_batch(bc_model* m, const void* desc, size_t n_queries, int desc_format, const uint32_t* fanout_mask,
                                   int a, int b, float* out, int kernel, void* stream);
/* Build (or load "<cache_dir>/joint_<hash>.cubin") the joint module of the ordered pair (a, b): straight-line sm_100a code
 * unrolled over the states of one of the two nodes, attached through the driver JIT and kept on the model.  BC_ELIMIT (with
 * the instruction count and the cap in bc_last_error) for a pair whose body would exceed BC_JOINT_MAX_FFMA = 32768 FMA-pipe
 * instructions per entry point; AUTO then expands. */
BC_API int bc_model_specialize_joint(bc_model* m, int a, int b, const char* cache_dir);
/* Its generated PTX (host-only models too; the bytes needed including the NUL, or BC_ELIMIT as above) and the hash that names
 * its cache entry (model, ordered pair and joint generator version; 0 for an invalid pair). */
BC_API int64_t bc_model_joint_source(const bc_model* m, int a, int b, char* buf, size_t buf_bytes);
BC_API uint64_t bc_model_joint_hash(const bc_model* m, int a, int b);

/* Device-side descriptor conversion (stream ordered, DEVICE pointers): RANGE_U8 / RANGE_U16 -> BITS. */
BC_API int bc_convert_desc(bc_model* m, const void* src, int src_format, void* dst, int dst_format, size_t n_queries,
                    void* stream);
/* SPARSE queries.  bc_expand_sparse: DEVICE pointers, writes n_queries BITS rows (stream ordered).
 * bc_query_batch_sparse_host: HOST pointers (pinned or pageable); chunks the batch and overlaps
 * H2D(row_off, entries) / expand / inference kernel / D2H(out) on internal streams.  This is the
 * end-to-end call behind Bayescard_BN.query_batch: per query it moves 4 + 4*k bytes in and 4 out. */
BC_API int bc_expand_sparse(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t n_queries,
                     void* dst_bits, void* stream);
BC_API int bc_query_batch_sparse_host(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t n_queries,
                               const uint32_t* fanout_mask, float* out_prob, int kernel);

/* WSPARSE: the sparse (query, n_distinct) dicts of query_decoding (Models/Bayescard_BN.py:279-325) WITH fractional
 * weights, as they cross PCIe: CSR over the batch, row q = words[row_off[q] .. row_off[q+1]), a list of runs
 *   header = column (bits 0-14) | continuation (bit 15) | first state (bits 16-23) | count (bits 24-31)
 * each followed by `count` fp32 weights for the states first .. first+count-1.  The first run of a column clears the
 * column (states that are not listed get weight 0); continuation runs add states; columns without a run are
 * unconstrained.  Expanded to DENSE_F32 rows on the device (bc_expand_wsparse: device buffers, stream ordered), then
 * evaluated like bc_query_batch_host; the IMDB expectation factors shrink from 1.5-1.8 KB to ~50-100 B per factor. */
BC_API int bc_expand_wsparse(bc_model* m, const uint32_t* row_off_dev, const uint32_t* words_dev, size_t n_queries,
                      float* dst_dense_dev, void* stream);
BC_API int bc_query_batch_wsparse_host(bc_model* m, const uint32_t* row_off, const uint32_t* words, size_t n_queries,
                                const uint32_t* fan_mask, float* out_prob, int kernel);

/* ---- PACKED: the densest wire form of unit-weight range / IN-list queries (what SPARSE carries), for PCIe ------------
 * The reference's query is a sparse dict {column: bins} (Evaluation/cardinality_estimation.py:60-111); over PCIe every
 * byte of it counts (the end-to-end rate of bc_query_batch_*_host is the copy rate divided by bytes per query):
 *     klen[n]                        uint8   entries of each query (<= 255)
 *     blk_off[ceil(n / 128) + 1]     uint32  index of the first entry of every block of 128 queries
 *     payload                        bit stream, entry e at bits [e*w, (e+1)*w), little endian in 32-bit words, rounded
 *                                    up to whole words + 2 words of padding; w = cb + 2*sb, cb = bits(n_nodes - 1), sb = bits(max_card - 1)
 *                                    (bc_model_packed_geometry); entry = col | lo << cb | hi << (cb + sb)
 * Entries of a query are grouped by column; an entry with its predecessor's column ORs into that column's mask (IN lists).
 * Census: 17 bits per entry, ~17 B per query (SPARSE: ~35 B).  Expanded to BITS rows on the device. */
BC_API int bc_model_packed_geometry(const bc_model* m, int* entry_bits, int* col_bits, int* state_bits);
/* HOST: SPARSE (CSR) -> PACKED.  klen[n], blk_off[ceil(n/128)+1], payload[payload_capacity]; *payload_bytes = bytes used
 * (also set when the capacity is too small: call once with capacity 0 to size the buffer). */
BC_API int bc_pack_sparse(const bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t n_queries, uint8_t* klen,
                          uint32_t* blk_off, void* payload, size_t payload_capacity, size_t* payload_bytes);
/* DEVICE buffers, stream ordered: PACKED -> BITS rows. */
BC_API int bc_expand_packed(bc_model* m, const uint8_t* klen_dev, const uint32_t* blk_off_dev, const void* payload_dev, size_t n_queries,
                            void* dst_bits_dev, void* stream);
/* HOST buffers (pinned for full speed) in, fp32 probabilities out: chunks of 1 M queries flow through three slots on
 * three streams (H2D | expansion + inference | D2H overlap across chunks of a larger batch). */
BC_API int bc_query_batch_packed_host(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload, size_t payload_bytes,
                                      size_t n_queries, const uint32_t* fanout_mask, float* out_prob, int kernel);
/* Asynchronous form: returns when the batch is ENQUEUED (copies, expansion, inference, read-back on the model's three streams) and
 * stores a ticket; `out` (PINNED host memory) is complete after bc_pipe_wait(m, ticket).  klen / blk_off / payload / fan_mask / out
 * must stay untouched until then.  Consecutive submissions overlap: the H2D copy of batch i + 1 runs under the kernels and the
 * read-back of batch i (a serving loop keeps two batches in flight).  Tickets complete in order; any synchronous *_host call on the
 * same model first waits for everything submitted. */
BC_API int bc_query_batch_packed_host_submit(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload,
                                             size_t payload_bytes, size_t nq, const uint32_t* fan_mask, float* out, int kernel,
                                             uint64_t* ticket);
BC_API int bc_pipe_wait(bc_model* m, uint64_t ticket);

/* ---- results beyond the fp32 range --------------------------------------------------------------------------------
 * The reference computes every product in fp64 (Pgmpy/inference/ExactInference.py:157-177, np.dot / np.prod on fp64
 * factors): ten narrow predicates on 1 000 - 10 000-bin domains give probabilities below 1e-38, which an fp32 result
 * flushes to zero.  The *_scaled entry points carry one power-of-two exponent per query: the kernels renormalise a
 * message row (exactly, by a power of two) every time an edge has been multiplied in, and return
 *     probability[q] = out_mantissa[q] * 2^out_exponent[q]          (combine in fp64: ldexp(mantissa, exponent)).
 * Served by the generic kernel (K1: every descriptor format, fan-out masks), the fused tensor-core kernel (K3: every
 * format, fan-out masks, the models it plans) and the batched large-domain path (K2: RANGE_* rows); BC_KERNEL_AUTO picks
 * between them the way bc_query_batch does for a model without an image.
 * DEVICE pointers, stream ordered. */
BC_API int bc_query_batch_scaled(bc_model* m, const void* desc, size_t n_queries, int desc_format,
                                 const uint32_t* fanout_mask, float* out_mantissa, int32_t* out_exponent, int kernel,
                                 void* stream);
/* HOST buffers in, fp64 probabilities out (the library combines mantissa and exponent). */
BC_API int bc_query_batch_scaled_host(bc_model* m, const void* desc, size_t n_queries, int desc_format,
                                      const uint32_t* fanout_mask, double* out_prob, int kernel);

/* Synthetic workload generator (BASELINE.json configs 2 and 5; SURVEY.md section 8d): writes
 * RANGE_U8 descriptors for query indices [first, first+n) from a counter-based RNG keyed by
 * (seed, query index), so any query can be regenerated on the host for oracle spot checks
 * (bc_gen_range_queries_host is the bit-identical host twin).  Per query k ~ U{kmin..kmax}
 * distinct columns are constrained, each with lo ~ U{0..card-1}, hi ~ U{lo..card-1}. */
BC_API int bc_gen_range_queries(bc_model* m, uint64_t seed, uint64_t first, size_t n, int kmin, int kmax,
                         void* desc_dev, void* stream);
BC_API int bc_gen_range_queries_host(int n_nodes, const int32_t* card, uint64_t seed, uint64_t first,
                              size_t n, int kmin, int kmax, void* desc_host);
/* The same queries in SPARSE form (host): row_off[n+1], entries (capacity n*kmax); entries of a query
 * are in ascending column order.  Returns the number of entries written in *n_entries. */
BC_API int bc_gen_sparse_queries_host(int n_nodes, const int32_t* card, uint64_t seed, uint64_t first, size_t n,
                               int kmin, int kmax, uint32_t* row_off, uint32_t* entries, size_t* n_entries);

/* ---- batched SQL -> descriptor compiler (HOST only, no GPU; SURVEY.md section 8f item 1) -------------------------
 * Replaces the per-query Python in front of the hot path: parse_query_single_table
 * (Evaluation/cardinality_estimation.py:22-119) followed by Bayescard_BN.query_decoding
 * (Models/Bayescard_BN.py:279-325, with realign :53-72, continuous_range_map :180-239 and
 * BN_single_model.apply_encoding_to_value / apply_ndistinct_to_value :98-139), for a BATCH of SQL texts, writing the
 * descriptor rows bc_query_batch* read.  The column tables are handed over once per model:
 *   categorical / boolean column: the encoding dict as parallel arrays in dict order (original value, numeric or
 *     string, -> bin and n_in_bin weight) and BN.domain[attr] in stored order (inequalities are evaluated on it);
 *   continuous column: BN.domain[attr] = (lo, hi), the bin edges of BN.mapping[attr] and n_distinct_mapping[attr].
 *   node = topological index of the column in the tree, or -1 for a column of the table that the tree does not hold
 *   (still decoded -- an undecodable predicate on it zeroes the estimate -- but it constrains nothing).
 * bc_sqlc_compile classifies every query:
 *   BC_SQLC_BITS    every weight is 1: BITS row written to bits_rows + i * bc_sqlc_bits_stride()
 *   BC_SQLC_DENSE   fractional n_distinct weights: DENSE_F32 row appended to dense_rows, dense_index[k] = i
 *   BC_SQLC_ZERO    undecodable predicate or no reachable column: the estimate is 0 (Bayescard_BN.py:517-521,
 *                   ExactInference.py:197); no row is written
 *   BC_SQLC_PYTHON  a predicate shape this compiler does not restate (anything the reference raises on, operands whose
 *                   Python parsing is subtle): the caller evaluates the query through the Python mirror
 *   BC_SQLC_OVERFLOW  a DENSE query that did not fit dense_capacity rows: compile it again with more room */
#define BC_SQLC_BITS 0
#define BC_SQLC_DENSE 1
#define BC_SQLC_ZERO 2
#define BC_SQLC_PYTHON 3
#define BC_SQLC_OVERFLOW 4
typedef struct bc_sqlc bc_sqlc;
BC_API int bc_sqlc_create(int n_nodes, const int32_t* card, bc_sqlc** out);
BC_API void bc_sqlc_destroy(bc_sqlc* c);
BC_API int64_t bc_sqlc_bits_stride(const bc_sqlc* c);   /* bytes per BITS row   (== bc_model_desc_stride(BITS))   */
BC_API int64_t bc_sqlc_dense_width(const bc_sqlc* c);   /* floats per DENSE row (== bc_model_dense_width())       */
BC_API int bc_sqlc_add_categorical(bc_sqlc* c, const char* name, int node, int has_encoding, int n_enc,
                                   const uint8_t* enc_is_str, const double* enc_num, const char* const* enc_str,
                                   const int32_t* enc_bin, const double* enc_weight, int n_dom,
                                   const uint8_t* dom_is_str, const double* dom_num, const char* const* dom_str);
BC_API int bc_sqlc_add_continuous(bc_sqlc* c, const char* name, int node, double dom_lo, double dom_hi, int n_bins,
                                  const double* edge_lo, const double* edge_hi, int n_ndmap, const double* nd_key,
                                  const double* nd_mult);
BC_API int bc_sqlc_compile(const bc_sqlc* c, size_t n_queries, const char* const* sql, uint8_t* kind, void* bits_rows,
                           float* dense_rows, size_t dense_capacity, uint32_t* dense_index, size_t* n_dense);

/* ---- CPT fitting for a fixed tree (SURVEY.md section 8f item 3) --------------------------------------------------
 * Replaces `self.model.fit(discrete_table)` (Models/Bayescard_BN.py:108-110): BayesianModel.fit
 * (Pgmpy/models/BayesianModel.py:278-323) -> MaximumLikelihoodEstimator.estimate_cpd (Pgmpy/estimators/MLE.py:61-104)
 * -> state_counts (Pgmpy/estimators/base.py:63-135).  One pass over the discretised table counts, for every node v,
 * how often (state of v, state of parent(v)) occurs:
 *   table_dev   DEVICE pointer, n_rows rows of bin ids, row-major, column v = topological node v, elements of
 *               elem_bytes (1: uint8, card <= 256; 2: uint16), row stride row_stride_elems (>= n_nodes) elements
 *   counts_dev  DEVICE pointer to n_counters + 1 64-bit counters: n_counters = sum_v card[v] * card[parent(v)] (root:
 *               card[0]), node after node in topological order, counter of (c, p) at off_v + c * card[parent(v)] + p
 *               -- the layout of TabularCPD.values -- followed by ONE extra counter, the number of skipped rows;
 *               zeroed by the call
 *   bad_rows_host  (nullable) number of rows skipped because a bin id was >= card; reading it synchronises the stream
 * The column normalisation (all-zero column -> uniform, MLE.py:77-79; values / values.sum(axis=0), CPD.normalize) is a
 * few thousand fp64 divisions and is left to the caller (bayescard_b200/fit.py), which keeps the CPTs bit-identical to
 * the reference's. */
BC_API int bc_fit_counts(int device, int n_nodes, const int32_t* parent, const int32_t* card, const void* table_dev,
                         int elem_bytes, size_t n_rows, size_t row_stride_elems, unsigned long long* counts_dev,
                         size_t n_counters, uint32_t* bad_rows_host, void* stream);

/* ---- Incremental update of a served model: rows inserted into / deleted from the table -------------------------
 * Replaces rerunning `self.model.fit(discrete_table)` of build_from_data (Models/Bayescard_BN.py:108-110) on the changed
 * table.  The tree stays as it is; only the CPTs follow the counts.  A model keeps u64 counts on the device once they are
 * attached; an update counts its rows into +/-1 deltas, adds them, and normalises again only the CPT columns (node, parent
 * state) whose counts moved, in fp64 with bc_fit_counts' caller's rule, so that the arena equals a fresh bc_model_create
 * of the refitted CPTs bit for bit.
 *
 * bc_model_set_counts: counts_host holds n_counters u64 counts in bc_fit_counts' layout (node after node, (c, p) at
 *   off_v + c * card[parent(v)] + p); n_counters must be the tree's total (checked before any device work).  The CPTs are
 *   NOT derived from them: the caller attaches counts that match the arena (bayescard_b200/fit.py checks this).  Replaces
 *   counts attached earlier.  Synchronous.
 * bc_model_get_counts: the counters of nodes [node_first, node_first + node_count) into counts_host.  Synchronous. */
BC_API int bc_model_set_counts(bc_model* m, const uint64_t* counts_host, size_t n_counters);
BC_API int bc_model_get_counts(const bc_model* m, int node_first, int node_count, uint64_t* counts_host);
/* The fp32 CPT arena as the kernels read it (from_device = 1, synchronous) or its host copy (0; BC_ELIMIT for models too large
 * to keep one): the arena bc_model_create was given, zero-padded.  Returns the number of floats; with out == NULL or a capacity
 * below that, nothing is copied. */
BC_API int64_t bc_model_arena(const bc_model* m, int from_device, float* out, size_t capacity);
/* One batch: ins_dev / del_dev are DEVICE tables of n_ins / n_del rows of bin ids (bc_fit_counts' convention: row-major,
 * column v = topological node v, elem_bytes 1 (uint8) or 2 (uint16), row stride row_stride_elems >= n_nodes elements).
 *   - counts become counts + count(ins) - count(del), integer-exact;
 *   - the call is rejected with BC_EINVAL, and NOTHING on the model changes, when a row of either table holds a bin id
 *     outside its node's domain (*bad_rows_host = how many) or when a delete would take a count below zero (the error
 *     names the node, own bin and parent bin); deleting rows that were never counted is only detected through such an
 *     underflow;
 *   - the touched CPT columns are re-normalised in the device arena and mirrored into the host copy, so bc_model_spec_hash
 *     changes with them; then, if any count changed, the specialised and marginal modules are unloaded (has_spec becomes
 *     0: call bc_model_specialize again) and the K2 / K3 plans are dropped (rebuilt on their next use).  An update with no
 *     rows, or whose deltas cancel, changes nothing and keeps every module attached;
 *   - touched_nodes_host (nullable, n_nodes bytes): 1 for every node whose counts changed; bad_rows_host nullable.
 * Stream ordered on `stream`: query batches enqueued on it before the call see the old CPTs, those enqueued after it the new
 * ones (the call synchronises the stream twice: once to validate, once when the host copy of the arena is complete).  No
 * call on the same model may run concurrently from another stream or host thread.
 * BC_EINVAL before any device work for: an element size other than 1 / 2, a short row stride, NULL rows, a node whose
 * card does not fit the element type, or a model without counts. */
BC_API int bc_model_update(bc_model* m, const void* ins_dev, size_t n_ins, const void* del_dev, size_t n_del, int elem_bytes,
                           size_t row_stride_elems, uint8_t* touched_nodes_host, uint32_t* bad_rows_host, void* stream);

/* ---- Structure learning: all-pairs counts, mutual information, Chow-Liu tree ------------------------------------
 * Replaces pomegranate's BayesianNetwork.from_samples(algorithm='chow-liu', root=0) (Models/BN_single_model.py:141-202).
 *   table_dev   DEVICE pointer, n_rows rows of bin ids, row-major, columns in ANY order, elem_bytes 1 (uint8) or 2
 *               (uint16), row stride row_stride_elems (>= n_cols) elements; n_cols >= 2; 1 <= card[i] <= 256 (uint8)
 *               or 65536 (uint16); sum of the cards, padded to a multiple of 256, at most 16384 (BC_ELIMIT beyond)
 *   counts_dev  DEVICE pointer to n_counters + 1 64-bit counters, zeroed by the call.  Layout: per column i its
 *               marginal counts (card[i] counters, at C_i = sum_{k<i} card[k]); then for every pair i < j in
 *               row-major pair order (0,1), (0,2), ..., (1,2), ... the block card[i] x card[j], row-major ([a][b] =
 *               rows with bin a in column i and bin b in column j); then ONE extra counter, the number of skipped rows
 *   bad_rows_host  (nullable) rows skipped because a bin id was >= its column's card (a skipped row counts nowhere,
 *               as in bc_fit_counts); reading it synchronises the stream
 * The counting is one int8 tensor-core GEMM (one-hot(table)^T . one-hot(table)) with s32 accumulation: exact. */
BC_API int bc_pair_counts(int device, int n_cols, const int32_t* card, const void* table_dev, int elem_bytes, size_t n_rows,
                          size_t row_stride_elems, unsigned long long* counts_dev, size_t n_counters,
                          uint32_t* bad_rows_host, void* stream);
/* The Chow-Liu tree of the table: bc_pair_counts, then MI[i][j] = sum_ab (n_ab/N) log(N n_ab / (n_a n_b)) over
 * n_ab > 0 in fp64 on the device (N = rows kept; pomegranate's mutual information with pseudocount 0, scaled by N),
 * then Prim's maximum spanning tree on the host, rooted at `root`.  Tie rule (pomegranate's discrete_chow_liu_tree):
 * the next edge is the (in-tree x, outside y) pair of largest MI, x scanned in the order the nodes joined, y
 * ascending, only a strictly larger MI replacing the best so far.
 *   parent_host  int32[n_cols]: parent column of every column, -1 for the root (table column order)
 *   counts_dev   (nullable) receives the counts as bc_pair_counts writes them (n_counters + 1 counters); when NULL
 *                the counts live in a temporary buffer and n_counters is ignored
 *   mi_host      (nullable) fp64[n_cols * n_cols], symmetric, zero diagonal
 * Synchronous: returns when the tree is known. */
BC_API int bc_chow_liu(int device, int n_cols, const int32_t* card, const void* table_dev, int elem_bytes, size_t n_rows,
                       size_t row_stride_elems, int root, unsigned long long* counts_dev, size_t n_counters,
                       int32_t* parent_host, double* mi_host, uint32_t* bad_rows_host, void* stream);

/* Measured FP32 FFMA peak of the device (TFLOP/s), the roofline denominator SURVEY.md section 8d
 * asks to measure in the same run rather than quote. */
BC_API int bc_measure_fp32_peak(int device, double* tflops, double* sm_clock_mhz);

/* Number of kernel launches issued by this library on behalf of the calling process. */
BC_API uint64_t bc_launch_count(void);

BC_API const char* bc_last_error(void);
BC_API const char* bc_version(void);

/* ---- factor lists of join queries, natively (HOST only; BASELINE.json config 3) -----------------------------------------
 * The IMDB ensemble answers a join query as join_size * prod(p_f | 1 / p_f) over FACTORS, each a query()/expectation() of one
 * BN with a dict {column: scalar | (lo, hi)} (Models/BN_ensemble_model.py:192-252, Evaluation/parse_query_imdb.py:54-325).
 * bc_sqlc_compile_factors restates Bayescard_BN.query_decoding (Models/Bayescard_BN.py:279-325) for those two value shapes
 * (numeric values) and writes the BITS / DENSE rows; factor f owns predicates pred_off[f] .. pred_off[f+1]: the column index
 * inside this compiler (bc_sqlc_column_index), kind 0 = scalar a / 1 = tuple (a, b).  ids (nullable) selects factors of a
 * larger table (the factors of one BN); fan_mask (nullable, one word per factor) marks factors that carry fan-out columns.
 * kind[] as for bc_sqlc_compile.  With ws_words != NULL the factors with fractional weights are written as WSPARSE rows
 * (ws_row_off[k] .. ws_row_off[k+1] for dense_index[k]; ~100 B instead of a 1.5 KB DENSE row) and dense_rows is not used. */
BC_API int bc_sqlc_set_null(bc_sqlc* c, const char* name, double null_value);   /* BN.null_values[name] */
BC_API int bc_sqlc_column_index(const bc_sqlc* c, const char* name);            /* -1: not a column of this BN */
BC_API int bc_sqlc_compile_factors(const bc_sqlc* c, size_t n_factors, const uint32_t* ids, const uint32_t* pred_off,
                                   const int32_t* pred_col, const uint8_t* pred_kind, const double* pred_a, const double* pred_b,
                                   const uint32_t* fan_mask, uint8_t* kind, void* bits_rows, float* dense_rows, size_t dense_capacity,
                                   uint32_t* dense_index, size_t* n_dense, uint32_t* ws_row_off, uint32_t* ws_words, size_t ws_capacity,
                                   size_t* n_ws_words);
/* The job-light star planner: a batch of SQL texts -> factor table (what Evaluation/parse_query_imdb.py:54-325 produces for a
 * star on title.id over the two-table models title x X; first model by the pairwise-RDC vector).  sqlc[b] / tables[b] /
 * join_sizes[b]: the model of title x tables[b]; fan_node[a * n_bn + b]: node of title.mul_<tables[b]>.movie_id in model a.
 * status[q] = 0 planned, 1 not a job-light star query (plan it with the Python mirror).  Factors of query q:
 * first_factor[q] .. first_factor[q+1].  BC_ELIMIT with *n_factors / *n_preds set when the buffers are too small. */
typedef struct bc_joblight bc_joblight;
BC_API int bc_joblight_create(int n_bn, const bc_sqlc* const* sqlc, const char* const* tables, const double* join_sizes,
                              const int32_t* fan_node, int n_rdc, const char* const* rdc_a, const char* const* rdc_b,
                              const double* rdc_val, double epsilon, bc_joblight** out);
BC_API void bc_joblight_destroy(bc_joblight* h);
BC_API int bc_joblight_plan(const bc_joblight* h, size_t n, const char* const* sqls, uint8_t* status, double* join_size,
                            uint32_t* first_factor, size_t factor_capacity, int32_t* factor_bn, uint8_t* factor_inverse,
                            uint32_t* factor_fan_mask, uint32_t* pred_off, size_t pred_capacity, int32_t* pred_col, uint8_t* pred_kind,
                            double* pred_a, double* pred_b, size_t* n_factors, size_t* n_preds);
/* The same over one text buffer: query q is text[text_off[q], text_off[q+1]) (n + 1 offsets; separators between queries are
 * whitespace / ';' to the parser).  Turning a batch of host-language strings into a char* array costs about as much as planning
 * them; a joined buffer does not. */
BC_API int bc_joblight_plan_text(const bc_joblight* h, size_t n, const char* text, const uint64_t* text_off, uint8_t* status,
                                 double* join_size, uint32_t* first_factor, size_t factor_capacity, int32_t* factor_bn,
                                 uint8_t* factor_inverse, uint32_t* factor_fan_mask, uint32_t* pred_off, size_t pred_capacity,
                                 int32_t* pred_col, uint8_t* pred_kind, double* pred_a, double* pred_b, size_t* n_factors,
                                 size_t* n_preds);
/* BN_ensemble.cardinality (Models/BN_ensemble_model.py:228-252): join_size * prod(p | 1/p), a zero factor gives 1, clamp >= 1. */
BC_API int bc_joblight_combine(size_t n, const uint8_t* status, const double* join_size, const uint32_t* first_factor,
                               const uint8_t* factor_inverse, const double* factor_prob, double* out);

#ifdef __cplusplus
}
#endif
#endif /* BAYESCARD_B200_H */
