// GROUP BY on one column: out[q][b] = sum_{x : x_t = b} prod_v w_v[x_v] T_v[x_v, x_pa(v)] for every state b of a target node t,
// with w_v multiplied by fanouts[v] where bit v of query q's fan-out mask is set (bc_expectation_marginal_batch).
// GROUP BY on two columns (bc_joint_marginal_batch): out[q][i][j], the same sum over x_a = i, x_b = j.
//
// Two paths (see include/bayescard_b200.h, bc_marginal_batch):
//   - the specialised marginal kernel of (model, t) (spec_codegen.cc / spec_jit.cu): one upward pass plus one downward
//     chain along the root -> t path per query, card(t) results per thread;
//   - the expansion, for every model the existing kernels serve: each row becomes card(t) rows, row b with the target's
//     weights restricted to state b (and the query's mask row), evaluated q-major by bc_query_batch, so its results already
//     are out[q][b].
// The joint marginal has the same two paths: its generated module of (a, b), or the expansion of each row into card(a) rows
// (a's weights restricted to one state each) evaluated by bc_expectation_marginal_batch(b), whose card(b) results per row
// already are out[q][i][j].
#include <cstring>
#include <functional>

#include "bc_internal.h"

namespace {

// BITS: row (q, b) = row q with the target's bits [off, off + card) ANDed with the one-hot of bit off + b.
__global__ void expand_bits_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, size_t nq, int words, int card,
                                   int off) {
    const size_t total = nq * (size_t)card * words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int w = (int)(i % words);
        const size_t r = i / words;
        const size_t q = r / card;
        const int b = (int)(r % card);
        uint32_t x = src[q * words + w];
        const int lo = w * 32, hi = lo + 32;   // bits of this word: [lo, hi)
        const int a = off > lo ? off : lo, e = off + card < hi ? off + card : hi;
        if (a < e) {
            const uint32_t tmask = (uint32_t)((((uint64_t)1 << (e - a)) - 1) << (a - lo));
            const int bit = off + b;
            const uint32_t keep = (bit >= lo && bit < hi) ? 1u << (bit - lo) : 0u;
            x &= ~tmask | keep;
        }
        dst[i] = x;
    }
}

// DENSE_F32: row (q, b) = row q with every weight of the target except state b set to 0.
__global__ void expand_dense_kernel(const float* __restrict__ src, float* __restrict__ dst, size_t nq, int width, int card, int off) {
    const size_t total = nq * (size_t)card * width;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(i % width);
        const size_t r = i / width;
        const size_t q = r / card;
        const int b = (int)(r % card);
        float x = src[q * width + j];
        if (j >= off && j < off + card && j != off + b) x = 0.f;
        dst[i] = x;
    }
}

// Fan-out mask: row (q, b) = mask row q, for each of the card rows of query q.
__global__ void expand_mask_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, size_t nq, int words, int card) {
    const size_t total = nq * (size_t)card * words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[(i / ((size_t)card * words)) * words + i % words];
}

constexpr size_t kExpandBytes = 256u << 20;   // bound on the expanded rows (and mask rows) of one chunk

// Each row becomes card(target) rows, row (q, b) with the target's weights restricted to state b and the mask row of q; the
// chunk's rows go q-major through `eval(rows, n_rows, mask_rows, out)`, which writes `per_row` floats per row.
using ExpandEval = std::function<int(const void*, size_t, const uint32_t*, float*)>;
int expand_path(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, int target, float* out, size_t per_row,
                const ExpandEval& eval, cudaStream_t st) {
    const int card = m->nodes[target].card;
    const size_t stride = (size_t)bc_model_desc_stride(m, fmt);
    const size_t mask_stride = fan_mask ? 4 * (size_t)m->mask_words : 0;
    const size_t row_bytes = (stride + mask_stride) * card;   // expanded bytes per query
    size_t chunk = kExpandBytes / row_bytes;
    if (chunk < 1) chunk = 1;
    if (chunk > nq) chunk = nq;
    void* scratch = nullptr;
    BC_CUDA_CHECK(cudaMallocAsync(&scratch, chunk * row_bytes, st));
    // the expanded mask rows follow the descriptor rows (stride is a multiple of 16 bytes)
    uint32_t* mask_scratch = fan_mask ? reinterpret_cast<uint32_t*>(static_cast<unsigned char*>(scratch) + chunk * stride * card) : nullptr;
    const int threads = 256;
    auto grid_of = [&](size_t elems) {
        long long grid = (long long)((elems + threads - 1) / threads);
        return (unsigned)(grid > (long long)m->sm_count * 16 ? (long long)m->sm_count * 16 : grid);
    };
    int rc = BC_OK;
    for (size_t q0 = 0; q0 < nq && rc == BC_OK; q0 += chunk) {
        const size_t cq = nq - q0 < chunk ? nq - q0 : chunk;
        const unsigned grid = grid_of(cq * card * stride / 4);
        const unsigned char* src = static_cast<const unsigned char*>(desc) + q0 * stride;
        if (fmt == BC_DESC_BITS)
            expand_bits_kernel<<<grid, threads, 0, st>>>(reinterpret_cast<const uint32_t*>(src), static_cast<uint32_t*>(scratch), cq,
                                                         (int)(stride / 4), card, m->bits[target].bit_off);
        else
            expand_dense_kernel<<<grid, threads, 0, st>>>(reinterpret_cast<const float*>(src), static_cast<float*>(scratch), cq,
                                                          (int)(stride / 4), card, m->nodes[target].lam_off);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess && fan_mask) {
            bc_count_launch();
            expand_mask_kernel<<<grid_of(cq * card * m->mask_words), threads, 0, st>>>(fan_mask + q0 * m->mask_words, mask_scratch, cq,
                                                                                       m->mask_words, card);
            e = cudaGetLastError();
        }
        if (e != cudaSuccess) {
            bc_set_error("marginal expansion kernel: %s", cudaGetErrorString(e));
            rc = BC_ECUDA;
            break;
        }
        bc_count_launch();
        rc = eval(scratch, cq * card, mask_scratch, out + q0 * card * per_row);
    }
    cudaFreeAsync(scratch, st);
    return rc;
}

bool bad_target(const bc_model* m, int target) {
    if (target < 0 || target >= m->n) {
        bc_set_error("target node %d outside the model's %d nodes", target, m->n);
        return true;
    }
    return false;
}

}  // namespace

extern "C" int bc_model_specialize_marginal(bc_model* m, int target, const char* cache_dir) {
    if (!m || m->device < 0) { bc_set_error("specialize_marginal needs a device model"); return BC_EINVAL; }
    if (bad_target(m, target)) return BC_EINVAL;
    return bc_marg_build(m, target, cache_dir);
}

extern "C" int64_t bc_model_marginal_source(const bc_model* m, int target, char* buf, size_t buf_bytes) {
    if (!m) { bc_set_error("model is NULL"); return BC_EINVAL; }
    if (bad_target(m, target)) return BC_EINVAL;
    if (m->arena.empty()) { bc_set_error("model too large for a specialised kernel"); return BC_ELIMIT; }
    const std::string s = bc_marginal_generate(*m, target);
    if (buf && buf_bytes > 0) {
        const size_t k = s.size() + 1 <= buf_bytes ? s.size() : buf_bytes - 1;
        std::memcpy(buf, s.data(), k);
        buf[k] = 0;
    }
    return (int64_t)s.size() + 1;
}

extern "C" uint64_t bc_model_marginal_hash(const bc_model* m, int target) {
    if (!m || target < 0 || target >= m->n) return 0;
    return bc_marginal_hash_of(*m, target);
}

extern "C" int bc_expectation_marginal_batch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fanout_mask, int target,
                                             float* out, int kernel, void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (bad_target(m, target)) return BC_EINVAL;
    if (fmt != BC_DESC_BITS && fmt != BC_DESC_DENSE_F32) {
        bc_set_error("bc_marginal_batch reads BITS or DENSE_F32 rows, not format %d", fmt);
        return BC_EINVAL;
    }
    if (nq == 0) return BC_OK;
    if (!desc || !out) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (kernel == BC_KERNEL_SPEC || (kernel == BC_KERNEL_AUTO && bc_marg_attached(m, target)))
        return bc_marg_launch(m, desc, nq, fmt, fanout_mask, target, out, st);
    return expand_path(m, desc, nq, fmt, fanout_mask, target, out, 1,
                       [&](const void* rows, size_t n, const uint32_t* mask, float* o) {
                           return bc_query_batch(m, rows, n, fmt, mask, o, kernel, st);
                       }, st);
}

extern "C" int bc_marginal_batch(bc_model* m, const void* desc, size_t nq, int fmt, int target, float* out, int kernel, void* stream) {
    return bc_expectation_marginal_batch(m, desc, nq, fmt, nullptr, target, out, kernel, stream);
}

// ------------------------------------------------------------------------------------ GROUP BY two columns
static bool bad_pair(const bc_model* m, int a, int b) {
    if (bad_target(m, a) || bad_target(m, b)) return true;
    if (a == b) {
        bc_set_error("a joint marginal needs two distinct nodes, got %d twice", a);
        return true;
    }
    return false;
}

extern "C" int bc_model_specialize_joint(bc_model* m, int a, int b, const char* cache_dir) {
    if (!m || m->device < 0) { bc_set_error("specialize_joint needs a device model"); return BC_EINVAL; }
    if (bad_pair(m, a, b)) return BC_EINVAL;
    return bc_joint_build(m, a, b, cache_dir);
}

extern "C" int64_t bc_model_joint_source(const bc_model* m, int a, int b, char* buf, size_t buf_bytes) {
    if (!m) { bc_set_error("model is NULL"); return BC_EINVAL; }
    if (bad_pair(m, a, b)) return BC_EINVAL;
    if (m->arena.empty()) { bc_set_error("model too large for a specialised kernel"); return BC_ELIMIT; }
    std::string s;
    const int rc = bc_joint_generate(*m, a, b, &s);
    if (rc != BC_OK) return rc;
    if (buf && buf_bytes > 0) {
        const size_t k = s.size() + 1 <= buf_bytes ? s.size() : buf_bytes - 1;
        std::memcpy(buf, s.data(), k);
        buf[k] = 0;
    }
    return (int64_t)s.size() + 1;
}

extern "C" uint64_t bc_model_joint_hash(const bc_model* m, int a, int b) {
    if (!m || a < 0 || a >= m->n || b < 0 || b >= m->n || a == b) return 0;
    return bc_joint_hash_of(*m, a, b);
}

extern "C" int bc_joint_marginal_batch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fanout_mask, int a, int b,
                                       float* out, int kernel, void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (bad_pair(m, a, b)) return BC_EINVAL;
    if (fmt != BC_DESC_BITS && fmt != BC_DESC_DENSE_F32) {
        bc_set_error("bc_joint_marginal_batch reads BITS or DENSE_F32 rows, not format %d", fmt);
        return BC_EINVAL;
    }
    if (nq == 0) return BC_OK;
    if (!desc || !out) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (kernel == BC_KERNEL_SPEC || (kernel == BC_KERNEL_AUTO && bc_joint_attached(m, a, b)))
        return bc_joint_launch(m, desc, nq, fmt, fanout_mask, a, b, out, st);
    return expand_path(m, desc, nq, fmt, fanout_mask, a, out, (size_t)m->nodes[b].card,
                       [&](const void* rows, size_t n, const uint32_t* mask, float* o) {
                           return bc_expectation_marginal_batch(m, rows, n, fmt, mask, b, o, kernel, stream);
                       }, st);
}
