// CPT fitting for a FIXED tree: the step right before the inference path (SURVEY.md section 8f item 3).
//
// Replaces `self.model.fit(discrete_table)` of Bayescard_BN.build_from_data (Models/Bayescard_BN.py:108-110), i.e.
// BayesianModel.fit (Pgmpy/models/BayesianModel.py:278-323) -> MaximumLikelihoodEstimator.estimate_cpd
// (Pgmpy/estimators/MLE.py:61-104) -> state_counts (Pgmpy/estimators/base.py:63-135): for every node a 2-D histogram
// of (own state, parent state) over the discretised table, then column normalisation (an all-zero column becomes
// uniform, MLE.py:77-79).  The reference spends 140 s (DMV, 11.6 M rows) to 717 s (Census) in pandas group-bys
// (logs/dmv_20210112-101604.log:6, logs/census_20210112-103814.log:6).
//
// Here the table (n_rows x n_cols bin ids, row-major, columns in topological order, uint8 or uint16) is read ONCE:
// each thread walks rows, every CTA keeps a private copy of ALL the count tables in shared memory (DMV 10 882
// counters = 43 KB, IMDB <= 122 KB) and adds into it with shared-memory atomics; tables of <= 64 counters (boolean
// columns) get one copy per lane so that the 32 lanes of a warp never collide on them.  At the
// end every CTA adds its private tables into the global 64-bit counters.  Models whose tables do not fit shared
// memory count straight into the global counters.  The counts are integers, so the result is bit-exact whatever the
// order of the atomics; the normalisation (a few thousand divisions) is done by the caller in fp64, exactly as the
// reference does it.  Bound: HBM (n_rows x n_cols x element size bytes, read once).
//
// The same kernel serves bc_model_update (DESIGN.md section 9e): a served model keeps its counts on the device, a batch of
// inserted / deleted rows is counted into +/-1 deltas, and only the CPT columns whose counts moved are normalised again --
// the reference's alternative is rerunning the whole fit on the changed table.
#include <cstring>

#include "bc_internal.h"

namespace {

struct FitNode {
    int parent;     // topological index of the parent column, -1 for the root
    int card;
    int card_pa;    // 1 for the root
    int off;        // first counter of this node; counter of (c, p) = off + c * card_pa + p
    int rep;        // tiny tables: first word of the lane-replicated copy in shared memory, else -1
};

constexpr int kMaxParamNodes = 160;  // the node table travels as a kernel parameter (3.2 KB) up to this many columns
struct FitParams {
    int n_nodes;
    FitNode nodes[kMaxParamNodes];
};

// Lane-replicated counters for tiny tables: a boolean-by-boolean edge has four counters that all 32 lanes of a warp
// hammer; with one copy per lane (counter i of a small table lives at rep + i * 32 + lane) there is no conflict.
constexpr int kSmallTable = 64;

constexpr int kRowsPerIter = 4;  // rows in flight per thread: their byte loads overlap

// NEG: the pass counts rows with -1 into two's-complement 64-bit deltas (bc_model_update's deleted rows): the flush adds
// 0 - x, the direct path adds ~0 (and undoes a skipped row's increments with +1).  NEG = false is bc_fit_counts' kernel.
template <typename T, bool SHARED, bool NEG = false>
__global__ void __launch_bounds__(256) fit_count_kernel(const T* __restrict__ table, size_t n_rows, size_t row_stride,
                                                         const __grid_constant__ FitParams prm, const FitNode* __restrict__ nodes_dev,
                                                         int n_nodes, int n_counters, int n_shared, unsigned long long* __restrict__ counts) {
    unsigned long long* bad_rows = counts + n_counters;  // one extra 64-bit counter behind the tables
    // dynamic shared memory: [node table (5 ints per node)] [private counters + lane replicas]
    extern __shared__ __align__(16) unsigned int smem_u[];
    int* s_nodes = reinterpret_cast<int*>(smem_u);
    unsigned int* s_cnt = smem_u + ((n_nodes * 5 + 3) & ~3);
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < n_nodes * 5; i += blockDim.x)
        s_nodes[i] = nodes_dev ? reinterpret_cast<const int*>(nodes_dev)[i] : reinterpret_cast<const int*>(prm.nodes)[i];
    if (SHARED)
        for (int i = threadIdx.x; i < n_shared; i += blockDim.x) s_cnt[i] = 0;
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t r0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r0 < n_rows; r0 += stride * kRowsPerIter) {
        const T* row[kRowsPerIter];
        int badv[kRowsPerIter];  // first node whose bin id is outside its domain (n_nodes: none); -1: no such row
#pragma unroll
        for (int k = 0; k < kRowsPerIter; ++k) {
            const size_t r = r0 + (size_t)k * stride;
            row[k] = table + (r < n_rows ? r : r0) * row_stride;
            badv[k] = r < n_rows ? n_nodes : -1;
        }
        for (int v = 0; v < n_nodes; ++v) {
            const int parent = s_nodes[5 * v], card = s_nodes[5 * v + 1], card_pa = s_nodes[5 * v + 2];
            const int off = s_nodes[5 * v + 3], rep = s_nodes[5 * v + 4];
            int c[kRowsPerIter], p[kRowsPerIter];
#pragma unroll
            for (int k = 0; k < kRowsPerIter; ++k) {
                c[k] = (int)row[k][v];
                p[k] = parent >= 0 ? (int)row[k][parent] : 0;  // validated earlier: parents come first
            }
#pragma unroll
            for (int k = 0; k < kRowsPerIter; ++k) {
                if (v >= badv[k]) continue;
                if (c[k] >= card) {  // rare: the row is skipped and reported, its earlier increments are undone below
                    badv[k] = v;
                    continue;
                }
                const int li = c[k] * card_pa + p[k];
                if (SHARED) atomicAdd(&s_cnt[rep >= 0 ? rep + (li << 5) + lane : off + li], 1u);
                else atomicAdd(&counts[off + li], NEG ? ~0ull : 1ull);
            }
        }
#pragma unroll
        for (int k = 0; k < kRowsPerIter; ++k) {
            if (badv[k] < 0 || badv[k] >= n_nodes) continue;
            atomicAdd(bad_rows, 1ull);
            for (int u = 0; u < badv[k]; ++u) {
                const int parent = s_nodes[5 * u], card_pa = s_nodes[5 * u + 2], off = s_nodes[5 * u + 3], rep = s_nodes[5 * u + 4];
                const int li = (int)row[k][u] * card_pa + (parent >= 0 ? (int)row[k][parent] : 0);
                if (SHARED) atomicSub(&s_cnt[rep >= 0 ? rep + (li << 5) + lane : off + li], 1u);
                else atomicAdd(&counts[off + li], NEG ? 1ull : ~0ull);
            }
        }
    }
    if (SHARED) {
        __syncthreads();
        // private tables -> global 64-bit counters; the lane replicas of a tiny table are summed first
        for (int v = 0; v < n_nodes; ++v) {
            const int card = s_nodes[5 * v + 1], card_pa = s_nodes[5 * v + 2], off = s_nodes[5 * v + 3], rep = s_nodes[5 * v + 4];
            if (rep < 0) continue;
            for (int li = threadIdx.x; li < card * card_pa; li += blockDim.x) {
                unsigned int x = 0;
                for (int l = 0; l < 32; ++l) x += s_cnt[rep + (li << 5) + l];
                s_cnt[off + li] = x;  // the plain slot of a replicated table is otherwise unused
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n_counters; i += blockDim.x) {
            const unsigned int x = s_cnt[i];
            if (x) atomicAdd(&counts[i], NEG ? 0ull - (unsigned long long)x : (unsigned long long)x);
        }
    }
}

template <typename T, bool SH, bool NEG>
int fit_launch(int device, unsigned grid, size_t smem, cudaStream_t st, const void* table_dev, size_t n_rows,
               size_t row_stride_elems, const FitParams& prm, const FitNode* d_nodes, int n_nodes, int total, int n_shared,
               unsigned long long* counts_dev) {
    static int attr_bytes[64] = {};  // per device: raise the dynamic shared-memory limit only when it grows
    if (device >= 64 || attr_bytes[device] < (int)smem) {
        BC_CUDA_CHECK(cudaFuncSetAttribute(fit_count_kernel<T, SH, NEG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (device < 64) attr_bytes[device] = (int)smem;
    }
    fit_count_kernel<T, SH, NEG><<<grid, 256, smem, st>>>(static_cast<const T*>(table_dev), n_rows, row_stride_elems, prm, d_nodes,
                                                         n_nodes, total, n_shared, counts_dev);
    return BC_OK;
}

// One counting pass of a table into counts_dev (n_counters + 1 counters, the last one counts skipped rows).  zero: the
// counters are cleared first (bc_fit_counts); neg: every row counts -1 (bc_model_update's deleted rows).  `who` prefixes
// the error messages; the caller has checked the pointers, the element size and the row stride.
int fit_pass(const char* who, int device, int n_nodes, const int32_t* parent, const int32_t* card, const void* table_dev,
             int elem_bytes, size_t n_rows, size_t row_stride_elems, unsigned long long* counts_dev, size_t n_counters,
             bool zero, bool neg, cudaStream_t st) {
    std::vector<FitNode> nodes(n_nodes);
    long long total = 0;
    for (int v = 0; v < n_nodes; ++v) {
        if (card[v] <= 0 || card[v] > (elem_bytes == 1 ? 256 : 65536) || parent[v] >= v || (v == 0) != (parent[v] < 0)) {
            bc_set_error("%s: node %d: card %d, parent %d (topological order, one root, card within the element type)",
                         who, v, card[v], parent[v]);
            return BC_EINVAL;
        }
        nodes[v].parent = parent[v];
        nodes[v].card = card[v];
        nodes[v].card_pa = parent[v] >= 0 ? card[parent[v]] : 1;
        nodes[v].off = (int)total;
        nodes[v].rep = -1;
        total += (long long)card[v] * nodes[v].card_pa;
        if (total > (1ll << 30)) {
            bc_set_error("%s: more than 2^30 counters", who);
            return BC_ELIMIT;
        }
    }
    if ((size_t)total != n_counters) {
        bc_set_error("%s: counts buffer holds %zu counters, the tree needs %lld", who, n_counters, total);
        return BC_EINVAL;
    }
    BC_CUDA_CHECK(cudaSetDevice(device));
    int sm_count = 0, smem_optin = 0;
    BC_CUDA_CHECK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    BC_CUDA_CHECK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    // shared-memory plan: all private tables + lane replicas of the tiny ones
    size_t n_shared = (size_t)total;
    for (int v = 0; v < n_nodes; ++v)
        if (nodes[v].card * nodes[v].card_pa <= kSmallTable) {
            nodes[v].rep = (int)n_shared;
            n_shared += (size_t)nodes[v].card * nodes[v].card_pa * 32;
        }
    bool shared = (n_shared + (size_t)n_nodes * 5 + 4) * 4 + 1024 <= (size_t)smem_optin;
    if (!shared && (size_t)total * 4 + 1024 <= (size_t)smem_optin) {  // the tables fit, their replicas do not
        for (int v = 0; v < n_nodes; ++v) nodes[v].rep = -1;
        n_shared = (size_t)total;
        shared = true;
    }
    const size_t node_words = ((size_t)n_nodes * 5 + 3) & ~(size_t)3;
    const size_t smem = (node_words + (shared ? n_shared : 0)) * 4;
    // the node table travels as a kernel parameter; only trees wider than that need a device copy
    const bool by_param = n_nodes <= kMaxParamNodes;
    FitNode* d_nodes = nullptr;
    if (!by_param) {
        BC_CUDA_CHECK(cudaMallocAsync(&d_nodes, sizeof(FitNode) * n_nodes, st));
        // pageable source: the copy is staged by the runtime before the call returns
        BC_CUDA_CHECK(cudaMemcpyAsync(d_nodes, nodes.data(), sizeof(FitNode) * n_nodes, cudaMemcpyHostToDevice, st));
    }
    if (zero) BC_CUDA_CHECK(cudaMemsetAsync(counts_dev, 0, sizeof(unsigned long long) * (n_counters + 1), st));
    if (n_rows) {
        static FitParams prm;  // filled under the lock below; passed by value at launch
        static std::mutex prm_mu;
        std::lock_guard<std::mutex> lock(prm_mu);
        prm.n_nodes = n_nodes;
        if (by_param) std::copy(nodes.begin(), nodes.end(), prm.nodes);
        // persistent grid: as many 256-thread CTAs per SM as the private tables allow (at most 4)
        int per_sm = shared ? (int)((size_t)smem_optin / (smem + 1024)) : 4;
        if (per_sm > 4) per_sm = 4;
        if (per_sm < 1) per_sm = 1;
        long long grid = (long long)sm_count * per_sm;
        const long long needed = (long long)((n_rows + 256 * kRowsPerIter - 1) / (256 * kRowsPerIter));
        if (grid > needed) grid = needed;
        auto launch = [&](auto fn) {
            return fn(device, (unsigned)grid, smem, st, table_dev, n_rows, row_stride_elems, prm, d_nodes, n_nodes, (int)total,
                      (int)n_shared, counts_dev);
        };
        int rc;
        if (elem_bytes == 1) {
            if (shared) rc = neg ? launch(fit_launch<uint8_t, true, true>) : launch(fit_launch<uint8_t, true, false>);
            else rc = neg ? launch(fit_launch<uint8_t, false, true>) : launch(fit_launch<uint8_t, false, false>);
        } else {
            if (shared) rc = neg ? launch(fit_launch<uint16_t, true, true>) : launch(fit_launch<uint16_t, true, false>);
            else rc = neg ? launch(fit_launch<uint16_t, false, true>) : launch(fit_launch<uint16_t, false, false>);
        }
        if (rc) return rc;
        BC_CUDA_CHECK(cudaGetLastError());
        bc_count_launch();
    }
    if (d_nodes) cudaFreeAsync(d_nodes, st);
    return BC_OK;
}

// ------------------------------------------------------------------------------------ incremental update
// Per node: where its counters, its columns (node, parent state) and its CPT live.
struct UpdNode {
    long long off;       // first counter (bc_fit_counts layout: off + c * card_pa + p)
    long long col_off;   // first column in the flat column index
    long long cpt_off;   // T_v in the arena: cpt_off + c * stride + p (root: cpt_off + c)
    int card, card_pa, stride, root;
};

// the node owning counter (by_col = false) or column (by_col = true) i: every node owns at least one of each
__device__ __forceinline__ int upd_node_of(const UpdNode* __restrict__ nd, int n, long long i, bool by_col) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((by_col ? nd[mid].col_off : nd[mid].off) <= i) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// Marks the nodes with a non-zero delta and records the first counter that counts + delta would take below zero.
__global__ void __launch_bounds__(256) upd_check_kernel(const UpdNode* __restrict__ nd, int n, const unsigned long long* __restrict__ counts,
                                                        const unsigned long long* __restrict__ delta, long long n_counters,
                                                        unsigned long long* first_bad, unsigned char* node_touched) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_counters; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long d = delta[i];
        if (!d) continue;
        node_touched[upd_node_of(nd, n, i, false)] = 1;
        if ((long long)d < 0 && counts[i] < 0ull - d) atomicMin(first_bad, (unsigned long long)i);
    }
}

// counts += delta (two's complement); marks the column of every changed counter.
__global__ void __launch_bounds__(256) upd_apply_kernel(const UpdNode* __restrict__ nd, int n, unsigned long long* __restrict__ counts,
                                                        const unsigned long long* __restrict__ delta, long long n_counters,
                                                        unsigned char* col_touched) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_counters; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long d = delta[i];
        if (!d) continue;
        counts[i] += d;
        const int v = upd_node_of(nd, n, i, false);
        col_touched[nd[v].col_off + (i - nd[v].off) % nd[v].card_pa] = 1;
    }
}

// Re-normalises every marked column exactly as fit.counts_to_cpts does (MLE.py:77-79, CPD.normalize): an all-zero column
// becomes 1 / card, otherwise count / column sum.  The sum of integer counts below 2^53 is exact in any order and the fp64
// division and the fp32 store round to nearest even, so the entries are bit-identical to numpy's followed by pack_arena's.
__global__ void __launch_bounds__(256) upd_norm_kernel(const UpdNode* __restrict__ nd, int n, const unsigned long long* __restrict__ counts,
                                                       long long n_cols, const unsigned char* __restrict__ col_touched, float* arena) {
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_cols; j += (long long)gridDim.x * blockDim.x) {
        if (!col_touched[j]) continue;
        const UpdNode r = nd[upd_node_of(nd, n, j, true)];
        const long long p = j - r.col_off;
        const unsigned long long* c0 = counts + r.off + p;
        double sum = 0.0;
        for (int c = 0; c < r.card; ++c) sum += __ull2double_rn(c0[(long long)c * r.card_pa]);
        float* t = arena + r.cpt_off + (r.root ? 0 : p);
        const long long step = r.root ? 1 : r.stride;
        for (int c = 0; c < r.card; ++c) {
            const double x = sum == 0.0 ? __ddiv_rn(1.0, (double)r.card) : __ddiv_rn(__ull2double_rn(c0[(long long)c * r.card_pa]), sum);
            t[c * step] = __double2float_rn(x);
        }
    }
}

long long model_counters(const bc_model* m) {
    long long total = 0;
    for (const BcNodeRec& r : m->nodes) total += (long long)r.card * r.card_pa;
    return total;
}

unsigned upd_grid(const bc_model* m, long long work) {
    long long g = (work + 255) / 256;
    if (g > (long long)m->sm_count * 8) g = (long long)m->sm_count * 8;
    return (unsigned)(g < 1 ? 1 : g);
}

}  // namespace

extern "C" int bc_fit_counts(int device, int n_nodes, const int32_t* parent, const int32_t* card, const void* table_dev,
                             int elem_bytes, size_t n_rows, size_t row_stride_elems, unsigned long long* counts_dev,
                             size_t n_counters, uint32_t* bad_rows_host, void* stream) {
    if (n_nodes <= 0 || !parent || !card || (!table_dev && n_rows) || !counts_dev || (elem_bytes != 1 && elem_bytes != 2) ||
        row_stride_elems < (size_t)n_nodes) {
        bc_set_error("bc_fit_counts: bad arguments");
        return BC_EINVAL;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = fit_pass("bc_fit_counts", device, n_nodes, parent, card, table_dev, elem_bytes, n_rows, row_stride_elems, counts_dev,
                      n_counters, true, false, st);
    if (rc) return rc;
    if (bad_rows_host) {
        unsigned long long bad = 0;
        BC_CUDA_CHECK(cudaMemcpyAsync(&bad, counts_dev + n_counters, sizeof(bad), cudaMemcpyDeviceToHost, st));
        BC_CUDA_CHECK(cudaStreamSynchronize(st));
        *bad_rows_host = (uint32_t)(bad > 0xffffffffull ? 0xffffffffull : bad);
    }
    return BC_OK;
}

extern "C" int bc_model_set_counts(bc_model* m, const uint64_t* counts_host, size_t n_counters) {
    if (!m) { bc_set_error("bc_model_set_counts: model is NULL"); return BC_EINVAL; }
    const long long total = model_counters(m);
    if ((size_t)total != n_counters) {
        bc_set_error("bc_model_set_counts: %zu counters given, the tree needs %lld", n_counters, total);
        return BC_EINVAL;
    }
    if (!counts_host) { bc_set_error("bc_model_set_counts: counts is NULL"); return BC_EINVAL; }
    if (m->device < 0) { bc_set_error("bc_model_set_counts: host-only model"); return BC_EINVAL; }
    if (total > (1ll << 30)) { bc_set_error("bc_model_set_counts: more than 2^30 counters"); return BC_ELIMIT; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    if (!m->d_counts) {
        std::vector<UpdNode> nd(m->n);
        std::vector<int64_t> cnt_off(m->n + 1), col_off(m->n + 1);
        long long off = 0, col = 0;
        for (int v = 0; v < m->n; ++v) {
            const BcNodeRec& r = m->nodes[v];
            nd[v] = UpdNode{off, col, (long long)r.cpt_off, r.card, r.card_pa, r.stride, v == 0 ? 1 : 0};
            cnt_off[v] = off;
            col_off[v] = col;
            off += (long long)r.card * r.card_pa;
            col += r.card_pa;
        }
        cnt_off[m->n] = off;
        col_off[m->n] = col;
        unsigned long long* d_counts = nullptr;
        void* d_upd = nullptr;
        BC_CUDA_CHECK(cudaMalloc(&d_counts, sizeof(unsigned long long) * (size_t)total));
        if (cudaMalloc(&d_upd, sizeof(UpdNode) * nd.size()) != cudaSuccess ||
            cudaMemcpy(d_upd, nd.data(), sizeof(UpdNode) * nd.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
            bc_set_error("bc_model_set_counts: %s", cudaGetErrorString(cudaGetLastError()));
            cudaFree(d_counts);
            cudaFree(d_upd);
            return BC_ECUDA;
        }
        m->d_counts = d_counts;
        m->d_upd = d_upd;
        m->cnt_off = std::move(cnt_off);
        m->col_off = std::move(col_off);
    }
    m->has_counts = false;   // (a failed copy leaves no counts attached)
    BC_CUDA_CHECK(cudaDeviceSynchronize());   // no update or query still reads the counters being replaced
    BC_CUDA_CHECK(cudaMemcpy(m->d_counts, counts_host, sizeof(uint64_t) * n_counters, cudaMemcpyHostToDevice));
    m->has_counts = true;
    return BC_OK;
}

extern "C" int bc_model_get_counts(const bc_model* m, int node_first, int node_count, uint64_t* counts_host) {
    if (!m) { bc_set_error("bc_model_get_counts: model is NULL"); return BC_EINVAL; }
    if (node_first < 0 || node_count < 0 || node_first + node_count > m->n) {
        bc_set_error("bc_model_get_counts: nodes [%d, %d + %d) outside the model's %d nodes", node_first, node_first, node_count, m->n);
        return BC_EINVAL;
    }
    if (!m->has_counts) { bc_set_error("bc_model_get_counts: no counts attached (bc_model_set_counts)"); return BC_EINVAL; }
    if (node_count == 0) return BC_OK;
    if (!counts_host) { bc_set_error("bc_model_get_counts: counts is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    const int64_t a = m->cnt_off[node_first], b = m->cnt_off[node_first + node_count];
    BC_CUDA_CHECK(cudaMemcpy(counts_host, m->d_counts + a, sizeof(uint64_t) * (size_t)(b - a), cudaMemcpyDeviceToHost));
    return BC_OK;
}

extern "C" int bc_model_update(bc_model* m, const void* ins_dev, size_t n_ins, const void* del_dev, size_t n_del, int elem_bytes,
                               size_t row_stride_elems, uint8_t* touched_nodes_host, uint32_t* bad_rows_host, void* stream) {
    if (!m) { bc_set_error("bc_model_update: model is NULL"); return BC_EINVAL; }
    if (elem_bytes != 1 && elem_bytes != 2) {
        bc_set_error("bc_model_update: element size %d (1: uint8, 2: uint16 bin ids)", elem_bytes);
        return BC_EINVAL;
    }
    if (row_stride_elems < (size_t)m->n) {
        bc_set_error("bc_model_update: row stride of %zu elements is shorter than a row of %d columns", row_stride_elems, m->n);
        return BC_EINVAL;
    }
    if ((n_ins && !ins_dev) || (n_del && !del_dev)) { bc_set_error("bc_model_update: rows are NULL"); return BC_EINVAL; }
    for (int v = 0; v < m->n; ++v)
        if (m->nodes[v].card > (elem_bytes == 1 ? 256 : 65536)) {
            bc_set_error("bc_model_update: node %d has %d states, more than %d-byte bin ids hold", v, m->nodes[v].card, elem_bytes);
            return BC_EINVAL;
        }
    if (!m->has_counts) { bc_set_error("bc_model_update: no counts attached (bc_model_set_counts)"); return BC_EINVAL; }
    if (touched_nodes_host) std::memset(touched_nodes_host, 0, (size_t)m->n);
    if (bad_rows_host) *bad_rows_host = 0;
    if (n_ins == 0 && n_del == 0) return BC_OK;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = bc_pipe_quiesce_model(m);   // asynchronous host submissions in flight still read the old CPTs
    if (rc) return rc;
    const int n = m->n;
    const long long n_counters = m->cnt_off[n], n_cols = m->col_off[n];
    // scratch: [delta x n_counters][skipped rows][first underflowing counter][node flags x n][column flags x n_cols]
    const size_t flag_bytes = (size_t)n + (size_t)n_cols;
    const size_t bytes = sizeof(unsigned long long) * ((size_t)n_counters + 2) + flag_bytes;
    unsigned long long* delta = nullptr;
    BC_CUDA_CHECK(cudaMallocAsync(&delta, bytes, st));
    struct Scratch {
        void* p;
        cudaStream_t st;
        ~Scratch() { cudaFreeAsync(p, st); }
    } scratch{delta, st};
    unsigned char* node_t = reinterpret_cast<unsigned char*>(delta + n_counters + 2);
    unsigned char* col_t = node_t + n;
    BC_CUDA_CHECK(cudaMemsetAsync(delta, 0, bytes, st));
    BC_CUDA_CHECK(cudaMemsetAsync(delta + n_counters + 1, 0xff, sizeof(unsigned long long), st));
    std::vector<int32_t> parent(n), card(n);
    for (int v = 0; v < n; ++v) {
        parent[v] = m->nodes[v].parent;
        card[v] = m->nodes[v].card;
    }
    // 1. delta counts: inserted rows +1, deleted rows -1, one buffer (the skipped-row counter collects both)
    if (n_ins && (rc = fit_pass("bc_model_update", m->device, n, parent.data(), card.data(), ins_dev, elem_bytes, n_ins,
                                row_stride_elems, delta, (size_t)n_counters, false, false, st)))
        return rc;
    if (n_del && (rc = fit_pass("bc_model_update", m->device, n, parent.data(), card.data(), del_dev, elem_bytes, n_del,
                                row_stride_elems, delta, (size_t)n_counters, false, true, st)))
        return rc;
    const UpdNode* nd = static_cast<const UpdNode*>(m->d_upd);
    // 2. validate: one read-back of {skipped rows, first underflow} and the touched nodes
    upd_check_kernel<<<upd_grid(m, n_counters), 256, 0, st>>>(nd, n, m->d_counts, delta, n_counters, delta + n_counters + 1, node_t);
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch();
    unsigned long long flags[2] = {0, 0};
    std::vector<uint8_t> touched(n, 0);
    BC_CUDA_CHECK(cudaMemcpyAsync(flags, delta + n_counters, sizeof(flags), cudaMemcpyDeviceToHost, st));
    BC_CUDA_CHECK(cudaMemcpyAsync(touched.data(), node_t, (size_t)n, cudaMemcpyDeviceToHost, st));
    BC_CUDA_CHECK(cudaStreamSynchronize(st));
    if (bad_rows_host) *bad_rows_host = (uint32_t)(flags[0] > 0xffffffffull ? 0xffffffffull : flags[0]);
    if (flags[0]) {
        bc_set_error("bc_model_update: %llu rows hold a bin id outside the model's domains; nothing was applied", flags[0]);
        return BC_EINVAL;
    }
    if (flags[1] != ~0ull) {
        const long long i = (long long)flags[1];
        int v = n - 1;
        while (m->cnt_off[v] > i) --v;
        const long long li = i - m->cnt_off[v];
        bc_set_error("bc_model_update: the deleted rows would take a count below zero (node %d, own bin %lld, parent bin %lld); "
                     "nothing was applied", v, li / m->nodes[v].card_pa, v == 0 ? -1ll : li % m->nodes[v].card_pa);
        return BC_EINVAL;
    }
    bool any = false;
    for (uint8_t t : touched) any = any || t;
    if (!any) return BC_OK;   // the deltas cancel: nothing moves, every module stays attached
    // 3. apply, re-normalise the touched columns in the device arena, mirror the touched nodes into the host arena
    upd_apply_kernel<<<upd_grid(m, n_counters), 256, 0, st>>>(nd, n, m->d_counts, delta, n_counters, col_t);
    BC_CUDA_CHECK(cudaGetLastError());
    upd_norm_kernel<<<upd_grid(m, n_cols), 256, 0, st>>>(nd, n, m->d_counts, n_cols, col_t, m->d_arena);
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch(2);
    if (!m->arena.empty())
        for (int v = 0; v < n; ++v) {
            if (!touched[v]) continue;
            const BcNodeRec& r = m->nodes[v];
            const size_t floats = (size_t)(v == 0 ? 1 : r.card) * r.stride;
            BC_CUDA_CHECK(cudaMemcpyAsync(m->arena.data() + r.cpt_off, m->d_arena + r.cpt_off, floats * sizeof(float),
                                          cudaMemcpyDeviceToHost, st));
        }
    BC_CUDA_CHECK(cudaStreamSynchronize(st));
    // 4. everything that cached the old CPTs goes; K2 / K3 plans and modules are rebuilt on their next use
    bc_model_drop_cached(m);
    if (touched_nodes_host) std::memcpy(touched_nodes_host, touched.data(), (size_t)n);
    return BC_OK;
}
