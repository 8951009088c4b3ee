// C ABI of libbayescard_b200.so: model lifecycle, kernel dispatch, host-buffer pipeline,
// synthetic query generator, FP32 peak probe.  See include/bayescard_b200.h for the contract.
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>

#include "bc_internal.h"

// ------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static std::atomic<uint64_t> g_launches{0};

void bc_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void bc_count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

extern "C" const char* bc_last_error(void) { return g_err; }
extern "C" const char* bc_version(void) { return BC_VERSION_STRING; }
extern "C" uint64_t bc_launch_count(void) { return g_launches.load(); }

// ------------------------------------------------------------------------------------ host pipe
struct BcHostPipe {
    static constexpr int kSlots = 3;
    cudaStream_t s_in = nullptr, s_k = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[kSlots]{}, ev_k[kSlots]{}, ev_out[kSlots]{};
    void* d_desc[kSlots]{};
    uint32_t* d_mask[kSlots]{};
    float* d_out[kSlots]{};
    void* h_desc[kSlots]{};   // pinned staging, used only when the caller's buffers are pageable
    uint32_t* h_mask[kSlots]{};
    float* h_out[kSlots]{};
    size_t cap_desc = 0, cap_mask = 0, cap_q = 0;
    // SPARSE path: CSR slices in, BITS rows built on the device
    uint32_t* d_rowoff[kSlots]{};
    uint32_t* d_entries[kSlots]{};
    uint32_t* d_bits[kSlots]{};
    uint32_t* h_rowoff[kSlots]{};
    uint32_t* h_entries[kSlots]{};
    size_t cap_sq = 0, cap_entries = 0;
    // WSPARSE path: weighted runs in, DENSE_F32 rows built on the device
    float* d_wdense[kSlots]{};
    size_t cap_wq = 0;
    // PACKED path: klen bytes, block offsets and the entry bit stream
    uint8_t* d_klen[kSlots]{};
    uint32_t* d_blk[kSlots]{};
    uint32_t* d_pay[kSlots]{};
    size_t cap_pq = 0, cap_pay = 0;
    // asynchronous submissions (bc_query_batch_packed_host_submit): chunks take slots round robin ACROSS calls
    uint64_t n_chunks = 0;          // chunks enqueued so far = the ticket of the latest submission
    bool pending = false;           // work of an un-waited submission may still be in flight
    bool slot_used[kSlots]{};
};

// Everything enqueued on the pipe has finished (every chunk ends with its D2H on s_out): the synchronous pipelines start from here.
static int pipe_quiesce(BcHostPipe* p) {
    if (!p || !p->pending) return BC_OK;
    BC_CUDA_CHECK(cudaStreamSynchronize(p->s_out));
    p->pending = false;
    for (bool& u : p->slot_used) u = false;
    return BC_OK;
}

int bc_pipe_quiesce_model(bc_model* m) {
    std::lock_guard<std::mutex> lock(m->pipe_mu);
    return pipe_quiesce(m->pipe);
}

static void pipe_free(BcHostPipe* p) {
    if (!p) return;
    for (int i = 0; i < BcHostPipe::kSlots; ++i) {
        cudaFree(p->d_desc[i]);
        cudaFree(p->d_mask[i]);
        cudaFree(p->d_out[i]);
        cudaFreeHost(p->h_desc[i]);
        cudaFreeHost(p->h_mask[i]);
        cudaFreeHost(p->h_out[i]);
        cudaFree(p->d_rowoff[i]);
        cudaFree(p->d_wdense[i]);
        cudaFree(p->d_klen[i]);
        cudaFree(p->d_blk[i]);
        cudaFree(p->d_pay[i]);
        cudaFree(p->d_entries[i]);
        cudaFree(p->d_bits[i]);
        cudaFreeHost(p->h_rowoff[i]);
        cudaFreeHost(p->h_entries[i]);
        if (p->ev_in[i]) cudaEventDestroy(p->ev_in[i]);
        if (p->ev_k[i]) cudaEventDestroy(p->ev_k[i]);
        if (p->ev_out[i]) cudaEventDestroy(p->ev_out[i]);
    }
    if (p->s_in) cudaStreamDestroy(p->s_in);
    if (p->s_k) cudaStreamDestroy(p->s_k);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    delete p;
}

// ------------------------------------------------------------------------------------ model
extern "C" int bc_model_create(int device, int n_nodes, const int32_t* parent, const int32_t* card,
                               const int64_t* cpt_off, const int32_t* stride, const float* cpt_arena,
                               size_t arena_floats, const int64_t* fan_off, const float* fan_arena,
                               size_t fan_floats, bc_model** out) {
    if (!out) { bc_set_error("out is NULL"); return BC_EINVAL; }
    *out = nullptr;
    if (n_nodes <= 0 || n_nodes > 65535 || !parent || !card || !cpt_off || !stride || !cpt_arena) {
        bc_set_error("bad model arguments (n_nodes=%d)", n_nodes);
        return BC_EINVAL;
    }
    if (arena_floats == 0 || arena_floats > (size_t(1) << 40) || fan_floats > (size_t(1) << 40)) {
        bc_set_error("implausible arena size (%zu CPT floats, %zu fan-out floats)", arena_floats, fan_floats);
        return BC_EINVAL;
    }
    bc_model* m = new (std::nothrow) bc_model();
    if (!m) { bc_set_error("out of host memory"); return BC_ENOMEM; }
    try {   // std::vector allocations below must not throw across the C ABI
    m->device = device;
    m->n = n_nodes;
    m->nodes.resize(n_nodes);
    int64_t lam = 0, max_stride = 4;
    for (int v = 0; v < n_nodes; ++v) {
        BcNodeRec& r = m->nodes[v];
        r.parent = parent[v];
        r.card = card[v];
        r.stride = stride[v];
        r.cpt_off = cpt_off[v];
        r.fan_off = (fan_off && fan_arena && fan_off[v] >= 0) ? (int32_t)fan_off[v] : -1;
        bool ok = card[v] >= 1 && stride[v] >= 1 && cpt_off[v] >= 0 && (cpt_off[v] % 4) == 0 && (stride[v] % 4) == 0;
        if (v == 0) ok = ok && parent[0] == -1;
        else ok = ok && parent[v] >= 0 && parent[v] < v;
        if (!ok) {
            bc_set_error("node %d: invalid parent/card/stride/offset (nodes must be topologically ordered, "
                         "offsets and strides multiples of 4 floats)", v);
            delete m;
            return BC_EINVAL;
        }
        r.card_pa = v == 0 ? 1 : card[parent[v]];
        const int64_t rows = v == 0 ? 1 : card[v];
        const int64_t cols = v == 0 ? card[0] : r.card_pa;
        if (stride[v] < cols || cpt_off[v] + rows * stride[v] > (int64_t)arena_floats) {
            bc_set_error("node %d: CPT [%lld x %lld, stride %d] at %lld exceeds the arena (%zu floats)", v,
                         (long long)rows, (long long)cols, stride[v], (long long)cpt_off[v], arena_floats);
            delete m;
            return BC_EINVAL;
        }
        if (r.fan_off >= 0 && (size_t)r.fan_off + card[v] > fan_floats) {
            bc_set_error("node %d: fan-out vector exceeds the fan arena", v);
            delete m;
            return BC_EINVAL;
        }
        r.lam_off = (int32_t)lam;
        lam += bc_round_up(card[v], 4);
        if (stride[v] > max_stride) max_stride = stride[v];
        if (card[v] > m->max_card) m->max_card = card[v];
        if (v > 0) m->flops_dense += 2LL * card[v] * r.card_pa;
    }
    if (lam > (1LL << 30)) { bc_set_error("sum of domain sizes too large"); delete m; return BC_ELIMIT; }
    m->lam_total = (int)lam;
    m->mask_words = (n_nodes + 31) / 32;
    // BITS rows: one bit per (node, state), tightly packed, row padded to 16 bytes
    m->bits.resize(n_nodes);
    int64_t bit = 0;
    for (int v = 0; v < n_nodes; ++v) {
        m->bits[v].bit_off = (int32_t)bit;
        m->bits[v].card = card[v];
        bit += card[v];
    }
    m->bits_words = (int)bc_round_up((bit + 31) / 32, 4);
    m->bits_default.assign(m->bits_words, 0u);
    for (int64_t b = 0; b < bit; ++b) m->bits_default[b >> 5] |= 1u << (b & 31);
    m->ent_node.resize(m->lam_total);
    for (int v = 0; v < n_nodes; ++v)
        for (int c = 0; c < (int)bc_round_up(card[v], 4); ++c) m->ent_node[m->nodes[v].lam_off + c] = (uint16_t)v;
    // host copy of the arena with a zero tail so that vectorised row loops may over-read safely
    const size_t tail = (size_t)(3 * max_stride + 64);
    m->arena_floats_padded = (size_t)bc_round_up((int64_t)(arena_floats + tail), 4);
    const bool keep_host = arena_floats <= (64u << 20);  // code generation only makes sense for small models
    if (keep_host || device < 0) {
        m->arena.assign(m->arena_floats_padded, 0.f);
        std::memcpy(m->arena.data(), cpt_arena, arena_floats * sizeof(float));
    }
    if (fan_arena && fan_floats) m->fan.assign(fan_arena, fan_arena + fan_floats);
    else m->fan.assign(4, 0.f);

    if (device >= 0) {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || device >= ndev) {
            bc_set_error("CUDA device %d not available (%s); this library has no CPU fallback", device,
                         e == cudaSuccess ? "ordinal out of range" : cudaGetErrorString(e));
            delete m;
            return BC_ECUDA;
        }
#define CK(expr)                                                                                  \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            bc_set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                         \
            bc_model_destroy(m);                                                                  \
            return BC_ECUDA;                                                                      \
        }                                                                                         \
    } while (0)
        CK(cudaSetDevice(device));
        {   // stream-ordered scratch (range rows -> BITS rows inside bc_query_batch) must not go back to the driver at every
            // synchronisation: with the default release threshold of 0 a B = 1 call paid ~0.5 ms of cudaMallocAsync
            cudaMemPool_t pool = nullptr;
            if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
                unsigned long long keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
            }
            cudaGetLastError();
        }
        CK(cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, device));
        CK(cudaDeviceGetAttribute(&m->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
        CK(cudaMalloc(&m->d_arena, m->arena_floats_padded * sizeof(float)));
        CK(cudaMemset(m->d_arena, 0, m->arena_floats_padded * sizeof(float)));
        CK(cudaMemcpy(m->d_arena, cpt_arena, arena_floats * sizeof(float), cudaMemcpyHostToDevice));
        CK(cudaMalloc(&m->d_fan, m->fan.size() * sizeof(float)));
        CK(cudaMemcpy(m->d_fan, m->fan.data(), m->fan.size() * sizeof(float), cudaMemcpyHostToDevice));
        CK(cudaMalloc(&m->d_nodes, m->nodes.size() * sizeof(BcNodeRec)));
        CK(cudaMemcpy(m->d_nodes, m->nodes.data(), m->nodes.size() * sizeof(BcNodeRec), cudaMemcpyHostToDevice));
        CK(cudaMalloc(&m->d_bits, m->bits.size() * sizeof(BcBitsRec)));
        CK(cudaMemcpy(m->d_bits, m->bits.data(), m->bits.size() * sizeof(BcBitsRec), cudaMemcpyHostToDevice));
        CK(cudaMalloc(&m->d_spec_ctr, BC_SPEC_CTR_SLOTS * 16));
        CK(cudaMemset(m->d_spec_ctr, 0, BC_SPEC_CTR_SLOTS * 16));
        CK(cudaMalloc(&m->d_bits_default, m->bits_default.size() * 4));
        CK(cudaMemcpy(m->d_bits_default, m->bits_default.data(), m->bits_default.size() * 4, cudaMemcpyHostToDevice));
        {
            std::vector<float> dd(m->lam_total, 0.f);
            for (int v = 0; v < m->n; ++v)
                for (int c = 0; c < m->nodes[v].card; ++c) dd[m->nodes[v].lam_off + c] = 1.f;
            CK(cudaMalloc(&m->d_dense_default, dd.size() * sizeof(float)));
            CK(cudaMemcpy(m->d_dense_default, dd.data(), dd.size() * sizeof(float), cudaMemcpyHostToDevice));
        }
        CK(cudaMalloc(&m->d_ent_node, m->ent_node.size() * sizeof(uint16_t)));
        CK(cudaMemcpy(m->d_ent_node, m->ent_node.data(), m->ent_node.size() * sizeof(uint16_t),
                      cudaMemcpyHostToDevice));
#undef CK
    }
    } catch (const std::bad_alloc&) {
        bc_set_error("out of host memory while building the model");
        bc_model_destroy(m);
        return BC_ENOMEM;
    }
    *out = m;
    return BC_OK;
}

extern "C" void bc_model_destroy(bc_model* m) {
    if (!m) return;
    if (m->device >= 0) {
        cudaSetDevice(m->device);
        pipe_free(m->pipe);
        bc_k2_free(m);
        bc_k3_free(m);
        if (m->spec_lib) cudaLibraryUnload(m->spec_lib);
        bc_marg_free(m);
        cudaFree(m->d_arena);
        cudaFree(m->d_fan);
        cudaFree(m->d_nodes);
        cudaFree(m->d_bits);
        cudaFree(m->d_bits_default);
        cudaFree(m->d_dense_default);
        cudaFree(m->d_spec_ctr);
        cudaFree(m->d_ent_node);
        cudaFree(m->d_counts);
        cudaFree(m->d_upd);
    }
    delete m;
}

void bc_model_drop_cached(bc_model* m) {
    if (m->spec_lib) cudaLibraryUnload(m->spec_lib);
    m->spec_lib = nullptr;
    m->spec_range8 = m->spec_dense = m->spec_bits = nullptr;
    {
        std::lock_guard<std::mutex> lock(m->marg_mu);
        bc_marg_free(m);
    }
    {
        std::lock_guard<std::mutex> lock(m->k2_mu);
        bc_k2_free(m);
    }
    std::lock_guard<std::mutex> lock(m->k3_mu);
    bc_k3_free(m);
}

extern "C" int bc_model_n_nodes(const bc_model* m) { return m ? m->n : 0; }
extern "C" int bc_model_device(const bc_model* m) { return m ? m->device : -1; }
extern "C" int64_t bc_model_dense_width(const bc_model* m) { return m ? m->lam_total : 0; }
extern "C" int64_t bc_model_dense_offset(const bc_model* m, int node) {
    if (!m || node < 0 || node >= m->n) return -1;
    return m->nodes[node].lam_off;
}
extern "C" int64_t bc_model_desc_stride(const bc_model* m, int fmt) {
    if (!m) return 0;
    switch (fmt) {
        case BC_DESC_RANGE_U8: return bc_round_up(2LL * m->n, 4);
        case BC_DESC_RANGE_U16: return 4LL * m->n;
        case BC_DESC_DENSE_F32: return 4LL * m->lam_total;
        case BC_DESC_BITS: return 4LL * m->bits_words;
    }
    return 0;
}
extern "C" int64_t bc_model_bits_offset(const bc_model* m, int node) {
    if (!m || node < 0 || node >= m->n) return -1;
    return m->bits[node].bit_off;
}
extern "C" int bc_model_bits_default(const bc_model* m, void* row_host, size_t row_bytes) {
    if (!m || !row_host || row_bytes < (size_t)m->bits_words * 4) { bc_set_error("bad arguments"); return BC_EINVAL; }
    std::memcpy(row_host, m->bits_default.data(), (size_t)m->bits_words * 4);
    return BC_OK;
}
extern "C" int64_t bc_model_flops_dense(const bc_model* m) { return m ? m->flops_dense : 0; }
extern "C" int64_t bc_model_arena(const bc_model* m, int from_device, float* out, size_t capacity) {
    if (!m) { bc_set_error("model is NULL"); return BC_EINVAL; }
    const size_t floats = m->arena_floats_padded;
    if (!out || capacity < floats) return (int64_t)floats;
    if (!from_device) {
        if (m->arena.empty()) { bc_set_error("the model keeps no host copy of its arena"); return BC_ELIMIT; }
        std::memcpy(out, m->arena.data(), floats * sizeof(float));
        return (int64_t)floats;
    }
    if (m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    BC_CUDA_CHECK(cudaMemcpy(out, m->d_arena, floats * sizeof(float), cudaMemcpyDeviceToHost));
    return (int64_t)floats;
}
extern "C" int bc_model_has_spec(const bc_model* m) {
    return m && (m->spec_range8 || m->spec_bits || m->spec_dense) ? 1 : 0;
}

extern "C" int64_t bc_model_spec_source(const bc_model* m, char* buf, size_t buf_bytes) {
    if (!m) { bc_set_error("model is NULL"); return BC_EINVAL; }
    if (m->arena.empty()) { bc_set_error("model too large for a specialised kernel"); return BC_ELIMIT; }
    std::string s = bc_spec_generate(*m);
    if (buf && buf_bytes > 0) {
        size_t k = s.size() + 1 <= buf_bytes ? s.size() : buf_bytes - 1;
        std::memcpy(buf, s.data(), k);
        buf[k] = 0;
    }
    return (int64_t)s.size() + 1;
}
extern "C" uint64_t bc_model_spec_hash(const bc_model* m) { return m ? bc_spec_hash_of(*m) : 0; }
extern "C" int bc_model_specialize(bc_model* m, const char* cache_dir) {
    if (!m || m->device < 0) { bc_set_error("specialize needs a device model"); return BC_EINVAL; }
    return bc_spec_build(m, cache_dir);
}
extern "C" int bc_model_load_cubin(bc_model* m, const void* image, size_t bytes) {
    if (!m || m->device < 0 || !image || !bytes) { bc_set_error("bad arguments"); return BC_EINVAL; }
    return bc_spec_attach(m, image, bytes);
}

// ------------------------------------------------------------------------------------ dispatch
static int check_format(const bc_model* m, int fmt) {
    if (fmt == BC_DESC_RANGE_U8 && m->max_card > 256) {
        bc_set_error("RANGE_U8 needs every domain <= 256 states (max is %d); use RANGE_U16", m->max_card);
        return BC_ELIMIT;
    }
    if (fmt < 0 || fmt > BC_DESC_BITS) { bc_set_error("unknown descriptor format %d", fmt); return BC_EINVAL; }
    return BC_OK;
}

// K3 reads BITS or DENSE_F32 rows: range rows are converted into stream-ordered scratch first
static int fused_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out, cudaStream_t st,
                        int32_t* out_exp) {
    if (fmt != BC_DESC_RANGE_U8 && fmt != BC_DESC_RANGE_U16) return bc_k3_launch(m, desc, nq, fmt, fan_mask, out, st, out_exp);
    {   // (decline before allocating anything when the model is not served)
        int32_t info[8];
        int rc = bc_model_fused_plan(m, info, nullptr, 0);
        if (rc) return rc;
    }
    void* scratch = nullptr;
    BC_CUDA_CHECK(cudaMallocAsync(&scratch, nq * (size_t)m->bits_words * 4, st));
    int rc = bc_convert_launch(m, desc, fmt, scratch, BC_DESC_BITS, nq, st);
    if (rc == BC_OK) rc = bc_k3_launch(m, scratch, nq, BC_DESC_BITS, fan_mask, out, st, out_exp);
    cudaFreeAsync(scratch, st);
    return rc;
}

extern "C" int bc_query_batch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask,
                              float* out, int kernel, void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq == 0) return BC_OK;
    if (!desc || !out) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    int rc = check_format(m, fmt);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool is_range = fmt == BC_DESC_RANGE_U8 || fmt == BC_DESC_RANGE_U16;
    const bool spec_direct = (fmt == BC_DESC_RANGE_U8 && m->spec_range8) || (fmt == BC_DESC_DENSE_F32 && m->spec_dense) ||
                             (fmt == BC_DESC_BITS && m->spec_bits);
    const bool spec_via_bits = is_range && !spec_direct && m->spec_bits;
    // AUTO: models whose straight-line code outgrows the instruction caches (IMDB: > 20k CPT entries) are faster on the
    // fused tensor-core kernel in every format (profiles/r1_k3_*.txt); it declines (BC_ELIMIT) what it cannot serve
    // (also for models without a specialised image from ~20k dense flops: measured faster than K1 / K2 on the synthetic
    // 10 x 100 and 20 x 50 trees, profiles/r1_config4_small_domains_k3.jsonl)
    const bool has_image = m->spec_bits || m->spec_dense || m->spec_range8;
    if (kernel == BC_KERNEL_AUTO && m->flops_dense >= (has_image ? 30000 : 20000) && m->n <= 128 && m->max_card <= 256) {
        // a handful of queries (the scalar drop-in call is B = 1): the warp-per-query kernel answers in 33 us where the
        // tile kernel needs 46 us and the straight-line kernel 94 us (400 KB of cold code); tools/latency_probe.py
        if (nq <= 32) return bc_k1_launch(m, desc, nq, fmt, fan_mask, out, st);
        rc = bc_query_batch(m, desc, nq, fmt, fan_mask, out, BC_KERNEL_FUSED, stream);
        if (rc != BC_ELIMIT) return rc;
    }
    if (kernel == BC_KERNEL_SPEC && !spec_direct && !spec_via_bits) {
        bc_set_error("no specialised kernel attached for this model / format (call bc_model_specialize)");
        return BC_ECOMPILE;
    }
    if (kernel == BC_KERNEL_SPEC || kernel == BC_KERNEL_AUTO) {
        if (spec_direct) return bc_spec_launch(m, desc, nq, fmt, fan_mask, out, st);
        if (spec_via_bits) {
            // range rows -> BITS rows in stream-ordered scratch, then the BITS kernel
            void* scratch = nullptr;
            BC_CUDA_CHECK(cudaMallocAsync(&scratch, nq * (size_t)m->bits_words * 4, st));
            rc = bc_convert_launch(m, desc, fmt, scratch, BC_DESC_BITS, nq, st);
            if (rc == BC_OK) rc = bc_spec_launch(m, scratch, nq, BC_DESC_BITS, fan_mask, out, st);
            cudaFreeAsync(scratch, st);
            return rc;
        }
    }
    if (kernel == BC_KERNEL_FUSED) return fused_launch(m, desc, nq, fmt, fan_mask, out, st, nullptr);
    if (kernel == BC_KERNEL_GEMM || kernel == BC_KERNEL_GEMM_SIMT)
        return bc_k2_launch(m, desc, nq, fmt, fan_mask, out, kernel == BC_KERNEL_GEMM, st);
    // no image: large domains go to the batched path (K1 re-reads every CPT once per query)
    if (kernel == BC_KERNEL_AUTO && is_range && !fan_mask && (m->max_card > 256 || m->lam_total > 4096))
        return bc_k2_launch(m, desc, nq, fmt, fan_mask, out, 1, st);
    if (kernel == BC_KERNEL_GENERIC || kernel == BC_KERNEL_AUTO) return bc_k1_launch(m, desc, nq, fmt, fan_mask, out, st);
    bc_set_error("kernel %d not available in this build", kernel);
    return BC_EINVAL;
}

extern "C" int bc_query_batch_scaled(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out_mant,
                                     int32_t* out_exp, int kernel, void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq == 0) return BC_OK;
    if (!desc || !out_mant || !out_exp) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    int rc = check_format(m, fmt);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool is_range = fmt == BC_DESC_RANGE_U8 || fmt == BC_DESC_RANGE_U16;
    if (kernel == BC_KERNEL_AUTO && nq > 32 && m->flops_dense >= 20000 && m->n <= 128 && m->max_card <= 256) {
        // the fused tensor-core kernel where it serves the model (it carries the exponent through its epilogue); it declines what
        // does not fit tensor memory
        rc = fused_launch(m, desc, nq, fmt, fan_mask, out_mant, st, out_exp);
        if (rc != BC_ELIMIT) return rc;
    }
    if (kernel == BC_KERNEL_AUTO)   // large domains: the batched path (K1 re-reads every CPT once per query)
        kernel = (is_range && !fan_mask && (m->max_card > 256 || m->lam_total > 4096)) ? BC_KERNEL_GEMM : BC_KERNEL_GENERIC;
    if (kernel == BC_KERNEL_GEMM || kernel == BC_KERNEL_GEMM_SIMT)
        return bc_k2_launch(m, desc, nq, fmt, fan_mask, out_mant, kernel == BC_KERNEL_GEMM, st, out_exp);
    if (kernel == BC_KERNEL_GENERIC) return bc_k1_launch(m, desc, nq, fmt, fan_mask, out_mant, st, out_exp);
    if (kernel == BC_KERNEL_FUSED) return fused_launch(m, desc, nq, fmt, fan_mask, out_mant, st, out_exp);
    bc_set_error("scaled results are served by BC_KERNEL_GENERIC, BC_KERNEL_FUSED and BC_KERNEL_GEMM(_SIMT), not by kernel %d", kernel);
    return BC_EINVAL;
}

extern "C" int bc_query_batch_scaled_host(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, double* out,
                                          int kernel) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq == 0) return BC_OK;
    if (!desc || !out) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    int rc = check_format(m, fmt);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    // not a throughput path (wide-range results are the rare case): one synchronous round trip in chunks
    const size_t stride = (size_t)bc_model_desc_stride(m, fmt);
    size_t chunk = (64u << 20) / stride;
    if (chunk < 4096) chunk = 4096;
    if (chunk > nq) chunk = nq;
    void* d_desc = nullptr;
    uint32_t* d_mask = nullptr;
    float* d_m = nullptr;
    int32_t* d_e = nullptr;
    auto cleanup = [&]() { cudaFree(d_desc); cudaFree(d_mask); cudaFree(d_m); cudaFree(d_e); };
    std::vector<float> hm;
    std::vector<int32_t> he;
    try {
        hm.resize(chunk);
        he.resize(chunk);
    } catch (const std::bad_alloc&) {
        bc_set_error("out of host memory");
        return BC_ENOMEM;
    }
#define CKS(expr)                                                                        \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            bc_set_error("%s failed: %s", #expr, cudaGetErrorString(_e));                \
            cleanup();                                                                   \
            return BC_ECUDA;                                                             \
        }                                                                                \
    } while (0)
    CKS(cudaMalloc(&d_desc, chunk * stride));
    if (fan_mask) CKS(cudaMalloc(&d_mask, chunk * m->mask_words * 4));
    CKS(cudaMalloc(&d_m, chunk * 4));
    CKS(cudaMalloc(&d_e, chunk * 4));
    for (size_t q0 = 0; q0 < nq; q0 += chunk) {
        const size_t cq = nq - q0 < chunk ? nq - q0 : chunk;
        CKS(cudaMemcpy(d_desc, static_cast<const unsigned char*>(desc) + q0 * stride, cq * stride, cudaMemcpyHostToDevice));
        if (fan_mask) CKS(cudaMemcpy(d_mask, fan_mask + q0 * m->mask_words, cq * m->mask_words * 4, cudaMemcpyHostToDevice));
        rc = bc_query_batch_scaled(m, d_desc, cq, fmt, fan_mask ? d_mask : nullptr, d_m, d_e, kernel, nullptr);
        if (rc) { cleanup(); return rc; }
        CKS(cudaMemcpy(hm.data(), d_m, cq * 4, cudaMemcpyDeviceToHost));
        CKS(cudaMemcpy(he.data(), d_e, cq * 4, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < cq; ++i) out[q0 + i] = std::ldexp((double)hm[i], he[i]);
    }
#undef CKS
    cleanup();
    return BC_OK;
}

static int pipe_streams(bc_model* m) {
    if (!m->pipe) {
        m->pipe = new BcHostPipe();
        BcHostPipe* p = m->pipe;
        BC_CUDA_CHECK(cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking));
        BC_CUDA_CHECK(cudaStreamCreateWithFlags(&p->s_k, cudaStreamNonBlocking));
        BC_CUDA_CHECK(cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            BC_CUDA_CHECK(cudaEventCreateWithFlags(&p->ev_in[i], cudaEventDisableTiming));
            BC_CUDA_CHECK(cudaEventCreateWithFlags(&p->ev_k[i], cudaEventDisableTiming));
            BC_CUDA_CHECK(cudaEventCreateWithFlags(&p->ev_out[i], cudaEventDisableTiming));
        }
    }
    return BC_OK;
}

static int pipe_ensure(bc_model* m, size_t chunk_q, size_t desc_stride) {
    int rc = pipe_streams(m);
    if (rc) return rc;
    BcHostPipe* p = m->pipe;
    const size_t need_desc = chunk_q * desc_stride, need_mask = chunk_q * m->mask_words * 4;
    if (need_desc > p->cap_desc || need_mask > p->cap_mask || chunk_q > p->cap_q) {
        // capacities are zeroed first and set only after every slot is allocated: a cudaMalloc that fails half way must
        // not leave NULL slots behind capacities that a later, smaller request would pass
        p->cap_desc = 0; p->cap_mask = 0; p->cap_q = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_desc[i]); cudaFree(p->d_mask[i]); cudaFree(p->d_out[i]);
            cudaFreeHost(p->h_desc[i]); cudaFreeHost(p->h_mask[i]); cudaFreeHost(p->h_out[i]);
            p->d_desc[i] = nullptr; p->d_mask[i] = nullptr; p->d_out[i] = nullptr;
            p->h_desc[i] = nullptr; p->h_mask[i] = nullptr; p->h_out[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_desc[i], need_desc));
            BC_CUDA_CHECK(cudaMalloc(&p->d_mask[i], need_mask));
            BC_CUDA_CHECK(cudaMalloc(&p->d_out[i], chunk_q * 4));
        }
        p->cap_desc = need_desc; p->cap_mask = need_mask; p->cap_q = chunk_q;
    }
    return BC_OK;
}

// An error return in the middle of a pipelined host call must not leave asynchronous copies running against the caller's
// pinned buffers (the caller may free them on error): the guard drains the three pipe streams on every exit path that
// did not reach the final synchronisation.
struct PipeDrain {
    BcHostPipe* p;
    bool armed = false;
    explicit PipeDrain(BcHostPipe* pipe) : p(pipe) {}
    ~PipeDrain() {
        if (!armed || !p) return;
        cudaStreamSynchronize(p->s_in);
        cudaStreamSynchronize(p->s_k);
        cudaStreamSynchronize(p->s_out);
    }
};

static bool is_pinned(const void* ptr) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

extern "C" int bc_query_batch_host(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask,
                                   float* out, int kernel) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq == 0) return BC_OK;
    if (!desc || !out) { bc_set_error("desc/out is NULL"); return BC_EINVAL; }
    int rc = check_format(m, fmt);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    const size_t stride = (size_t)bc_model_desc_stride(m, fmt);
    // ~16 MiB of descriptors per chunk keeps three slots in flight without hogging memory
    size_t chunk = (16u << 20) / stride;
    chunk = chunk < 4096 ? 4096 : chunk;
    if (chunk > nq) chunk = nq;
    std::lock_guard<std::mutex> lock(m->pipe_mu);
    if ((rc = pipe_quiesce(m->pipe))) return rc;   // (asynchronous PACKED submissions share the slots)
    rc = pipe_ensure(m, chunk, stride);
    if (rc) return rc;
    BcHostPipe* p = m->pipe;
    PipeDrain drain(p);
    const bool pin_desc = is_pinned(desc), pin_out = is_pinned(out), pin_mask = !fan_mask || is_pinned(fan_mask);
    auto ensure_host = [&](void** h, size_t bytes) -> int {
        if (!*h) BC_CUDA_CHECK(cudaHostAlloc(h, bytes, cudaHostAllocDefault));
        return BC_OK;
    };
    const size_t nchunks = (nq + chunk - 1) / chunk;
    for (size_t ci = 0; ci < nchunks; ++ci) {
        const int s = (int)(ci % BcHostPipe::kSlots);
        const size_t q0 = ci * chunk, cq = (q0 + chunk <= nq) ? chunk : nq - q0;
        // the slot's previous D2H (and with it its kernel and H2D) must be finished before reuse
        if (ci >= (size_t)BcHostPipe::kSlots) {
            BC_CUDA_CHECK(cudaEventSynchronize(p->ev_out[s]));
            if (!pin_out) {
                const size_t pq0 = (ci - BcHostPipe::kSlots) * chunk;
                std::memcpy(out + pq0, p->h_out[s], chunk * 4);
            }
        }
        const unsigned char* src = static_cast<const unsigned char*>(desc) + q0 * stride;
        if (!pin_desc) {
            if ((rc = ensure_host(&p->h_desc[s], p->cap_desc))) return rc;
            std::memcpy(p->h_desc[s], src, cq * stride);
            src = static_cast<const unsigned char*>(p->h_desc[s]);
        }
        drain.armed = true;
        BC_CUDA_CHECK(cudaMemcpyAsync(p->d_desc[s], src, cq * stride, cudaMemcpyHostToDevice, p->s_in));
        const uint32_t* dmask = nullptr;
        if (fan_mask) {
            const uint32_t* msrc = fan_mask + q0 * m->mask_words;
            if (!pin_mask) {
                if ((rc = ensure_host((void**)&p->h_mask[s], p->cap_mask))) return rc;
                std::memcpy(p->h_mask[s], msrc, cq * m->mask_words * 4);
                msrc = p->h_mask[s];
            }
            BC_CUDA_CHECK(cudaMemcpyAsync(p->d_mask[s], msrc, cq * m->mask_words * 4, cudaMemcpyHostToDevice, p->s_in));
            dmask = p->d_mask[s];
        }
        BC_CUDA_CHECK(cudaEventRecord(p->ev_in[s], p->s_in));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_k, p->ev_in[s], 0));
        rc = bc_query_batch(m, p->d_desc[s], cq, fmt, dmask, p->d_out[s], kernel, p->s_k);
        if (rc) return rc;
        BC_CUDA_CHECK(cudaEventRecord(p->ev_k[s], p->s_k));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_out, p->ev_k[s], 0));
        float* dst = out + q0;
        if (!pin_out) {
            if ((rc = ensure_host((void**)&p->h_out[s], p->cap_q * 4))) return rc;
            dst = p->h_out[s];
        }
        BC_CUDA_CHECK(cudaMemcpyAsync(dst, p->d_out[s], cq * 4, cudaMemcpyDeviceToHost, p->s_out));
        BC_CUDA_CHECK(cudaEventRecord(p->ev_out[s], p->s_out));
    }
    BC_CUDA_CHECK(cudaStreamSynchronize(p->s_out));
    drain.armed = false;   // s_out waited for every kernel and copy of the call
    if (!pin_out) {
        const size_t first = nchunks > (size_t)BcHostPipe::kSlots ? nchunks - BcHostPipe::kSlots : 0;
        for (size_t ci = first; ci < nchunks; ++ci) {
            const int s = (int)(ci % BcHostPipe::kSlots);
            const size_t q0 = ci * chunk, cq = (q0 + chunk <= nq) ? chunk : nq - q0;
            std::memcpy(out + q0, p->h_out[s], cq * 4);
        }
    }
    return BC_OK;
}


// ------------------------------------------------------------------------------------ conversion / sparse
extern "C" int bc_convert_desc(bc_model* m, const void* src, int src_fmt, void* dst, int dst_fmt, size_t nq,
                               void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq && (!src || !dst)) { bc_set_error("src/dst is NULL"); return BC_EINVAL; }
    int rc = check_format(m, src_fmt);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    return bc_convert_launch(m, src, src_fmt, dst, dst_fmt, nq, static_cast<cudaStream_t>(stream));
}

extern "C" int bc_expand_sparse(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t nq,
                                void* dst_bits, void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq && (!row_off || !dst_bits)) { bc_set_error("row_off/dst is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    return bc_expand_sparse_launch(m, row_off, entries, nq, dst_bits, static_cast<cudaStream_t>(stream));
}

static int sparse_ensure(bc_model* m, size_t chunk_q, size_t chunk_entries) {
    int rc = pipe_streams(m);
    if (rc) return rc;
    BcHostPipe* p = m->pipe;
    if (chunk_q > p->cap_sq) {
        p->cap_sq = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_rowoff[i]); cudaFree(p->d_bits[i]);
            cudaFreeHost(p->h_rowoff[i]);
            p->d_rowoff[i] = nullptr; p->d_bits[i] = nullptr; p->h_rowoff[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_rowoff[i], (chunk_q + 1) * 4));
            BC_CUDA_CHECK(cudaMalloc(&p->d_bits[i], chunk_q * (size_t)m->bits_words * 4));
        }
        p->cap_sq = chunk_q;
    }
    if (chunk_entries > p->cap_entries) {
        p->cap_entries = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_entries[i]);
            cudaFreeHost(p->h_entries[i]);
            p->d_entries[i] = nullptr; p->h_entries[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_entries[i], chunk_entries * 4));
        }
        p->cap_entries = chunk_entries;
    }
    const size_t need_mask = chunk_q * m->mask_words * 4;
    if (chunk_q > p->cap_q || need_mask > p->cap_mask) {
        p->cap_q = 0; p->cap_mask = 0; p->cap_desc = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_mask[i]); cudaFree(p->d_out[i]);
            cudaFreeHost(p->h_mask[i]); cudaFreeHost(p->h_out[i]);
            p->d_mask[i] = nullptr; p->d_out[i] = nullptr; p->h_mask[i] = nullptr; p->h_out[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_mask[i], need_mask));
            BC_CUDA_CHECK(cudaMalloc(&p->d_out[i], chunk_q * 4));
        }
        p->cap_q = chunk_q; p->cap_mask = need_mask;
        // the RANGE/DENSE staging of this pipe is sized per (cap_q, cap_desc): force it to be rebuilt
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_desc[i]); cudaFreeHost(p->h_desc[i]);
            p->d_desc[i] = nullptr; p->h_desc[i] = nullptr;
        }
        p->cap_desc = 0;
    }
    return BC_OK;
}

static int sparse_host_impl(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t nq, const uint32_t* fan_mask,
                            float* out, int kernel, bool weighted) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq == 0) return BC_OK;
    if (!row_off || !out) { bc_set_error("row_off/out is NULL"); return BC_EINVAL; }
    if (row_off[nq] > row_off[0] && !entries) { bc_set_error("entries is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    // chunks of 1M queries (~30 MB of CSR): measured on B200 (profiles/r1_e2e_chunk_sweep.txt) every extra
    // chunk costs ~50 us of copy / event latency, more than the overlap wins back below a few million
    // queries; larger batches pipeline H2D | expand+infer | D2H over three slots (BC_SPARSE_CHUNK overrides)
    size_t chunk = weighted ? 128 * 1024 : 1024 * 1024;   // weighted rows expand to 4 * sum(card) bytes each on the device
    if (const char* env = std::getenv(weighted ? "BC_WSPARSE_CHUNK" : "BC_SPARSE_CHUNK")) {
        const long long v = std::atoll(env);
        if (v >= 1024) chunk = (size_t)v;
    }
    if (chunk > nq) chunk = nq;
    const size_t nchunks = (nq + chunk - 1) / chunk;
    size_t max_entries = 1;
    for (size_t ci = 0; ci < nchunks; ++ci) {
        const size_t q0 = ci * chunk, q1 = q0 + chunk < nq ? q0 + chunk : nq;
        if (row_off[q1] < row_off[q0]) { bc_set_error("row_off is not monotone at query %zu", q0); return BC_EINVAL; }
        const size_t ne = row_off[q1] - row_off[q0];
        if (ne > max_entries) max_entries = ne;
    }
    std::lock_guard<std::mutex> lock(m->pipe_mu);
    int rc = pipe_quiesce(m->pipe);   // (asynchronous PACKED submissions share the slots)
    if (rc) return rc;
    rc = sparse_ensure(m, chunk, max_entries);
    if (rc) return rc;
    BcHostPipe* p = m->pipe;
    PipeDrain drain(p);
    if (weighted && chunk > p->cap_wq) {
        p->cap_wq = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_wdense[i]);
            p->d_wdense[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_wdense[i], chunk * (size_t)m->lam_total * 4));
        }
        p->cap_wq = chunk;
    }
    const bool pin_off = is_pinned(row_off), pin_ent = !entries || is_pinned(entries), pin_out = is_pinned(out),
               pin_mask = !fan_mask || is_pinned(fan_mask);
    auto ensure_host = [&](void** h, size_t bytes) -> int {
        if (!*h) BC_CUDA_CHECK(cudaHostAlloc(h, bytes, cudaHostAllocDefault));
        return BC_OK;
    };
    for (size_t ci = 0; ci < nchunks; ++ci) {
        const int s = (int)(ci % BcHostPipe::kSlots);
        const size_t q0 = ci * chunk, cq = (q0 + chunk <= nq) ? chunk : nq - q0;
        if (ci >= (size_t)BcHostPipe::kSlots) {
            BC_CUDA_CHECK(cudaEventSynchronize(p->ev_out[s]));
            if (!pin_out) std::memcpy(out + (ci - BcHostPipe::kSlots) * chunk, p->h_out[s], chunk * 4);
        }
        const uint32_t e0 = row_off[q0];
        const size_t ne = row_off[q0 + cq] - e0;
        const uint32_t* osrc = row_off + q0;
        if (!pin_off) {
            if ((rc = ensure_host((void**)&p->h_rowoff[s], (p->cap_sq + 1) * 4))) return rc;
            std::memcpy(p->h_rowoff[s], osrc, (cq + 1) * 4);
            osrc = p->h_rowoff[s];
        }
        drain.armed = true;
        BC_CUDA_CHECK(cudaMemcpyAsync(p->d_rowoff[s], osrc, (cq + 1) * 4, cudaMemcpyHostToDevice, p->s_in));
        if (ne) {
            const uint32_t* esrc = entries + e0;
            if (!pin_ent) {
                if ((rc = ensure_host((void**)&p->h_entries[s], p->cap_entries * 4))) return rc;
                std::memcpy(p->h_entries[s], esrc, ne * 4);
                esrc = p->h_entries[s];
            }
            BC_CUDA_CHECK(cudaMemcpyAsync(p->d_entries[s], esrc, ne * 4, cudaMemcpyHostToDevice, p->s_in));
        }
        const uint32_t* dmask = nullptr;
        if (fan_mask) {
            const uint32_t* msrc = fan_mask + q0 * m->mask_words;
            if (!pin_mask) {
                if ((rc = ensure_host((void**)&p->h_mask[s], p->cap_mask))) return rc;
                std::memcpy(p->h_mask[s], msrc, cq * m->mask_words * 4);
                msrc = p->h_mask[s];
            }
            BC_CUDA_CHECK(cudaMemcpyAsync(p->d_mask[s], msrc, cq * m->mask_words * 4, cudaMemcpyHostToDevice, p->s_in));
            dmask = p->d_mask[s];
        }
        BC_CUDA_CHECK(cudaEventRecord(p->ev_in[s], p->s_in));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_k, p->ev_in[s], 0));
        // row_off values are absolute entry indices: bias the entries pointer instead of rewriting them
        if (weighted) {
            rc = bc_expand_wsparse_launch(m, p->d_rowoff[s], p->d_entries[s] - e0, cq, p->d_wdense[s], p->s_k);
            if (rc) return rc;
            rc = bc_query_batch(m, p->d_wdense[s], cq, BC_DESC_DENSE_F32, dmask, p->d_out[s], kernel, p->s_k);
        } else {
            rc = bc_expand_sparse_launch(m, p->d_rowoff[s], p->d_entries[s] - e0, cq, p->d_bits[s], p->s_k);
            if (rc) return rc;
            rc = bc_query_batch(m, p->d_bits[s], cq, BC_DESC_BITS, dmask, p->d_out[s], kernel, p->s_k);
        }
        if (rc) return rc;
        BC_CUDA_CHECK(cudaEventRecord(p->ev_k[s], p->s_k));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_out, p->ev_k[s], 0));
        float* dst = out + q0;
        if (!pin_out) {
            if ((rc = ensure_host((void**)&p->h_out[s], p->cap_q * 4))) return rc;
            dst = p->h_out[s];
        }
        BC_CUDA_CHECK(cudaMemcpyAsync(dst, p->d_out[s], cq * 4, cudaMemcpyDeviceToHost, p->s_out));
        BC_CUDA_CHECK(cudaEventRecord(p->ev_out[s], p->s_out));
    }
    BC_CUDA_CHECK(cudaStreamSynchronize(p->s_out));
    drain.armed = false;   // s_out waited for every kernel and copy of the call
    if (!pin_out) {
        const size_t first = nchunks > (size_t)BcHostPipe::kSlots ? nchunks - BcHostPipe::kSlots : 0;
        for (size_t ci = first; ci < nchunks; ++ci) {
            const int s = (int)(ci % BcHostPipe::kSlots);
            const size_t q0 = ci * chunk, cq = (q0 + chunk <= nq) ? chunk : nq - q0;
            std::memcpy(out + q0, p->h_out[s], cq * 4);
        }
    }
    return BC_OK;
}

extern "C" int bc_query_batch_sparse_host(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t nq,
                                          const uint32_t* fan_mask, float* out, int kernel) {
    return sparse_host_impl(m, row_off, entries, nq, fan_mask, out, kernel, false);
}

extern "C" int bc_query_batch_wsparse_host(bc_model* m, const uint32_t* row_off, const uint32_t* words, size_t nq,
                                           const uint32_t* fan_mask, float* out, int kernel) {
    return sparse_host_impl(m, row_off, words, nq, fan_mask, out, kernel, true);
}

// ------------------------------------------------------------------------------------ PACKED wire format
extern "C" int bc_model_packed_geometry(const bc_model* m, int* entry_bits, int* col_bits, int* state_bits) {
    if (!m) { bc_set_error("model is NULL"); return BC_EINVAL; }
    int cb, sb;
    bc_packed_geometry(m, &cb, &sb);
    if (entry_bits) *entry_bits = cb + 2 * sb;
    if (col_bits) *col_bits = cb;
    if (state_bits) *state_bits = sb;
    if (cb + 2 * sb > 31) { bc_set_error("PACKED entries hold at most 31 bits; this model needs %d", cb + 2 * sb); return BC_ELIMIT; }
    return BC_OK;
}

extern "C" int bc_pack_sparse(const bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t nq, uint8_t* klen,
                              uint32_t* blk_off, void* payload, size_t payload_capacity, size_t* payload_bytes) {
    if (!m || !row_off || (!klen && nq) || !blk_off || !payload) { bc_set_error("bad arguments"); return BC_EINVAL; }
    int w, cb, sb;
    int rc = bc_model_packed_geometry(m, &w, &cb, &sb);
    if (rc) return rc;
    const size_t ne = nq ? (size_t)row_off[nq] - row_off[0] : 0;
    const size_t need = ((ne * (size_t)w + 31) / 32 + 2) * 4;   // whole 32-bit words + 2: the expansion kernel reads two words per entry
    if (payload_bytes) *payload_bytes = need;
    if (need > payload_capacity) { bc_set_error("payload buffer too small: %zu B needed", need); return BC_EINVAL; }
    if (ne && !entries) { bc_set_error("entries is NULL"); return BC_EINVAL; }
    if (ne >= (1ull << 32)) { bc_set_error("batch too large for 32-bit entry indices: split it"); return BC_ELIMIT; }
    std::memset(payload, 0, need);
    uint32_t* words = static_cast<uint32_t*>(payload);
    const uint32_t e_base = nq ? row_off[0] : 0;
    size_t e = 0;
    for (size_t q = 0; q < nq; ++q) {
        if (q % BC_PACKED_BLOCK == 0) blk_off[q / BC_PACKED_BLOCK] = (uint32_t)e;
        const uint32_t a = row_off[q], b = row_off[q + 1];
        if (b < a || b - a > 255) { bc_set_error("query %zu: %u entries (PACKED holds at most 255 per query)", q, b - a); return BC_ELIMIT; }
        klen[q] = (uint8_t)(b - a);
        int prev = -1;
        for (uint32_t i = a; i < b; ++i, ++e) {
            const uint32_t x = entries[i];
            const int col = (int)(x & 0x7fffu), cont = (int)((x >> 15) & 1u);
            const uint32_t lo = (x >> 16) & 0xffu, hi = x >> 24;
            if (cont != (col == prev)) {   // PACKED has no continuation bit: entries of a column must be adjacent, first one without `cont`
                bc_set_error("query %zu: entries must be grouped by column (continuation entries right behind their column's first)", q);
                return BC_EINVAL;
            }
            if (col >= (1 << cb) || lo >= (1u << sb) || hi >= (1u << sb)) { bc_set_error("query %zu: entry out of range for this model", q); return BC_EINVAL; }
            prev = col;
            const uint64_t v = (uint64_t)col | ((uint64_t)lo << cb) | ((uint64_t)hi << (cb + sb));
            const size_t bit = e * (size_t)w;
            const uint64_t sh = v << (bit & 31);
            words[bit >> 5] |= (uint32_t)sh;
            words[(bit >> 5) + 1] |= (uint32_t)(sh >> 32);
        }
        (void)e_base;
    }
    blk_off[(nq + BC_PACKED_BLOCK - 1) / BC_PACKED_BLOCK] = (uint32_t)e;
    return BC_OK;
}

extern "C" int bc_expand_packed(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload, size_t nq, void* dst_bits,
                                void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq && (!klen || !blk_off || !payload || !dst_bits)) { bc_set_error("klen/blk_off/payload/dst is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    return bc_expand_packed_launch(m, klen, blk_off, static_cast<const uint32_t*>(payload), 0ull, nq, dst_bits, static_cast<cudaStream_t>(stream));
}

// Host buffers in (pinned for full speed), fp32 probabilities out.  Batches beyond one chunk of 1 M queries (BC_PACKED_CHUNK
// overrides; a multiple of 128) flow through three slots on three streams (H2D | expansion + inference | D2H).  Smaller
// chunks were measured and LOSE on this platform (profiles/r2_e2e_packed_chunk_sweep.txt: every chunk costs ~100 us of
// enqueue / event latency -- 1 M queries: one chunk 1.69e9 q/s, four chunks 1.42e9, sixteen 0.60e9), so a 1 M-query call
// is one H2D copy of 15 MB, two kernels and one D2H copy; what it gains over SPARSE is the bytes: 15.4 B instead of 31 B per
// Census query.
// PACKED entries -> H2D -> expand -> infer -> D2H in chunks over the three slots.  `ticket` == nullptr: synchronous (returns when `out`
// is complete).  Otherwise the call returns once everything is ENQUEUED and *ticket identifies the submission for
// bc_pipe_wait: consecutive submissions then overlap (the copy of batch i + 1 runs under the kernels and the read-back of batch i).
static int packed_host_run(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload, size_t payload_bytes, size_t nq,
                           const uint32_t* fan_mask, float* out, int kernel, uint64_t* ticket) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (ticket) *ticket = 0;
    if (nq == 0) return BC_OK;
    if (!klen || !blk_off || !payload || !out) { bc_set_error("klen/blk_off/payload/out is NULL"); return BC_EINVAL; }
    int w, cb, sb;
    int rc = bc_model_packed_geometry(m, &w, &cb, &sb);
    if (rc) return rc;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    // 512 K queries per chunk: a 1 M-query call then overlaps the second chunk's H2D with the first chunk's kernels and read-back
    // (profiles/r2_e2e_packed_chunk_sweep.txt: one chunk 1.41e9, two 2.10e9, four 1.97e9, eight 1.88e9 queries/s on the same box)
    size_t chunk = 512 * 1024;
    if (const char* env = std::getenv("BC_PACKED_CHUNK")) {
        const long long v = std::atoll(env);
        if (v >= BC_PACKED_BLOCK) chunk = (size_t)v / BC_PACKED_BLOCK * BC_PACKED_BLOCK;
    }
    const size_t nblk_total = (nq + BC_PACKED_BLOCK - 1) / BC_PACKED_BLOCK;
    if (chunk > nblk_total * BC_PACKED_BLOCK) chunk = nblk_total * BC_PACKED_BLOCK;
    const size_t nchunks = (nq + chunk - 1) / chunk;
    const size_t total_words = payload_bytes / 4;
    const uint32_t* pay = static_cast<const uint32_t*>(payload);
    // largest payload slice of a chunk (+ 2 words of read-ahead)
    size_t max_words = 4;
    for (size_t ci = 0; ci < nchunks; ++ci) {
        const size_t b0 = ci * chunk / BC_PACKED_BLOCK, q1 = (ci + 1) * chunk < nq ? (ci + 1) * chunk : nq;
        const size_t b1 = (q1 + BC_PACKED_BLOCK - 1) / BC_PACKED_BLOCK;
        if (blk_off[b1] < blk_off[b0]) { bc_set_error("blk_off is not monotone at block %zu", b0); return BC_EINVAL; }
        const size_t w0 = ((size_t)blk_off[b0] * w) >> 5, w1 = (((size_t)blk_off[b1] * w + 31) >> 5) + 2;
        if (w1 > total_words) { bc_set_error("payload shorter than blk_off says (%zu words needed, %zu given)", w1, total_words); return BC_EINVAL; }
        if (w1 - w0 > max_words) max_words = w1 - w0;
    }
    std::lock_guard<std::mutex> lock(m->pipe_mu);
    rc = pipe_streams(m);
    if (rc) return rc;
    BcHostPipe* p = m->pipe;
    const size_t need_mask = chunk * m->mask_words * 4;
    if (chunk > p->cap_sq || chunk > p->cap_q || need_mask > p->cap_mask || chunk > p->cap_pq || max_words * 4 > p->cap_pay)
        if ((rc = pipe_quiesce(p))) return rc;   // buffers are about to be re-allocated: nothing may be in flight
    rc = sparse_ensure(m, chunk, 1);
    if (rc) return rc;
    if (chunk > p->cap_pq || max_words * 4 > p->cap_pay) {
        p->cap_pq = 0;
        p->cap_pay = 0;
        for (int i = 0; i < BcHostPipe::kSlots; ++i) {
            cudaFree(p->d_klen[i]); cudaFree(p->d_blk[i]); cudaFree(p->d_pay[i]);
            p->d_klen[i] = nullptr; p->d_blk[i] = nullptr; p->d_pay[i] = nullptr;
            BC_CUDA_CHECK(cudaMalloc(&p->d_klen[i], chunk));
            BC_CUDA_CHECK(cudaMalloc(&p->d_blk[i], (chunk / BC_PACKED_BLOCK + 2) * 4));
            BC_CUDA_CHECK(cudaMalloc(&p->d_pay[i], max_words * 4));
        }
        p->cap_pq = chunk;
        p->cap_pay = max_words * 4;
    }
    PipeDrain drain(p);
    for (size_t ci = 0; ci < nchunks; ++ci) {
        const int s = (int)(p->n_chunks % BcHostPipe::kSlots);
        const size_t q0 = ci * chunk, cq = (q0 + chunk <= nq) ? chunk : nq - q0;
        const size_t b0 = q0 / BC_PACKED_BLOCK, nb = (cq + BC_PACKED_BLOCK - 1) / BC_PACKED_BLOCK;
        if (p->slot_used[s]) BC_CUDA_CHECK(cudaEventSynchronize(p->ev_out[s]));   // the slot's buffers are free again
        const size_t w0 = ((size_t)blk_off[b0] * w) >> 5, w1 = (((size_t)blk_off[b0 + nb] * w + 31) >> 5) + 2;
        drain.armed = true;
        p->pending = true;
        p->slot_used[s] = true;
        ++p->n_chunks;
        BC_CUDA_CHECK(cudaMemcpyAsync(p->d_klen[s], klen + q0, cq, cudaMemcpyHostToDevice, p->s_in));
        BC_CUDA_CHECK(cudaMemcpyAsync(p->d_blk[s], blk_off + b0, (nb + 1) * 4, cudaMemcpyHostToDevice, p->s_in));
        BC_CUDA_CHECK(cudaMemcpyAsync(p->d_pay[s], pay + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, p->s_in));
        const uint32_t* dmask = nullptr;
        if (fan_mask) {
            BC_CUDA_CHECK(cudaMemcpyAsync(p->d_mask[s], fan_mask + q0 * m->mask_words, cq * m->mask_words * 4, cudaMemcpyHostToDevice, p->s_in));
            dmask = p->d_mask[s];
        }
        BC_CUDA_CHECK(cudaEventRecord(p->ev_in[s], p->s_in));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_k, p->ev_in[s], 0));
        rc = bc_expand_packed_launch(m, p->d_klen[s], p->d_blk[s], p->d_pay[s], (unsigned long long)w0, cq, p->d_bits[s], p->s_k);
        if (rc) return rc;
        rc = bc_query_batch(m, p->d_bits[s], cq, BC_DESC_BITS, dmask, p->d_out[s], kernel, p->s_k);
        if (rc) return rc;
        BC_CUDA_CHECK(cudaEventRecord(p->ev_k[s], p->s_k));
        BC_CUDA_CHECK(cudaStreamWaitEvent(p->s_out, p->ev_k[s], 0));
        BC_CUDA_CHECK(cudaMemcpyAsync(out + q0, p->d_out[s], cq * 4, cudaMemcpyDeviceToHost, p->s_out));
        BC_CUDA_CHECK(cudaEventRecord(p->ev_out[s], p->s_out));
    }
    if (ticket) {
        *ticket = p->n_chunks;
        drain.armed = false;
        return BC_OK;
    }
    BC_CUDA_CHECK(cudaStreamSynchronize(p->s_out));
    p->pending = false;
    for (bool& u : p->slot_used) u = false;
    drain.armed = false;
    return BC_OK;
}

extern "C" int bc_query_batch_packed_host(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload, size_t payload_bytes,
                                          size_t nq, const uint32_t* fan_mask, float* out, int kernel) {
    return packed_host_run(m, klen, blk_off, payload, payload_bytes, nq, fan_mask, out, kernel, nullptr);
}

extern "C" int bc_query_batch_packed_host_submit(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const void* payload,
                                                 size_t payload_bytes, size_t nq, const uint32_t* fan_mask, float* out, int kernel,
                                                 uint64_t* ticket) {
    if (!ticket) { bc_set_error("ticket is NULL"); return BC_EINVAL; }
    if (m && nq && !is_pinned(out)) { bc_set_error("an asynchronous submission reads its results back into PINNED host memory"); return BC_EINVAL; }
    return packed_host_run(m, klen, blk_off, payload, payload_bytes, nq, fan_mask, out, kernel, ticket);
}

extern "C" int bc_pipe_wait(bc_model* m, uint64_t ticket) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (ticket == 0) return BC_OK;
    cudaEvent_t ev;
    {
        std::lock_guard<std::mutex> lock(m->pipe_mu);
        BcHostPipe* p = m->pipe;
        if (ticket > (p ? p->n_chunks : 0)) { bc_set_error("ticket %llu was not issued by this model", (unsigned long long)ticket); return BC_EINVAL; }
        if (!p->pending) return BC_OK;
        BC_CUDA_CHECK(cudaSetDevice(m->device));
        if (ticket == p->n_chunks) return pipe_quiesce(p);
        // chunks finish in order; the slot's event belongs to chunk ticket - 1 or to a later chunk that reused the slot (then it
        // waits for more than it has to, never for less)
        ev = p->ev_out[(ticket - 1) % BcHostPipe::kSlots];
    }
    BC_CUDA_CHECK(cudaEventSynchronize(ev));
    return BC_OK;
}

extern "C" int bc_expand_wsparse(bc_model* m, const uint32_t* row_off, const uint32_t* words, size_t nq, float* dst_dense,
                                 void* stream) {
    if (!m || m->device < 0) { bc_set_error("model has no device (host-only model)"); return BC_EINVAL; }
    if (nq && (!row_off || !dst_dense)) { bc_set_error("row_off/dst is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    return bc_expand_wsparse_launch(m, row_off, words, nq, dst_dense, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------ generator
// Counter-based RNG: splitmix64 keyed by (seed, query index); identical on host and device.
__host__ __device__ static inline uint64_t bc_mix(uint64_t& s) {
    s += 0x9E3779B97F4A7C15ull;
    uint64_t z = s;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__host__ __device__ static inline void bc_gen_row(const int32_t* card, int n, uint64_t seed, uint64_t idx,
                                                  int kmin, int kmax, uint8_t* row) {
    uint64_t s = seed * 0xD1342543DE82EF95ull + idx * 0x2545F4914F6CDD1Dull + 0x1234567ull;
    bc_mix(s);
    for (int v = 0; v < n; ++v) {
        row[2 * v] = 0;
        row[2 * v + 1] = (uint8_t)(card[v] - 1);
    }
    int k = kmin + (int)(bc_mix(s) % (uint64_t)(kmax - kmin + 1));
    if (k > n) k = n;
    uint32_t used[32];
    for (int i = 0; i < 32; ++i) used[i] = 0;
    for (int j = 0; j < k; ++j) {
        int v;
        do {
            v = (int)(bc_mix(s) % (uint64_t)n);
        } while ((used[v >> 5] >> (v & 31)) & 1u);
        used[v >> 5] |= 1u << (v & 31);
        const int c = card[v];
        const int lo = (int)(bc_mix(s) % (uint64_t)c);
        const int hi = lo + (int)(bc_mix(s) % (uint64_t)(c - lo));
        row[2 * v] = (uint8_t)lo;
        row[2 * v + 1] = (uint8_t)hi;
    }
}

__global__ void bc_gen_kernel(const BcNodeRec* nodes, int n, uint64_t seed, uint64_t first, size_t nq, int kmin,
                              int kmax, uint8_t* desc, size_t stride) {
    extern __shared__ int32_t s_card[];
    for (int v = threadIdx.x; v < n; v += blockDim.x) s_card[v] = nodes[v].card;
    __syncthreads();
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (size_t)gridDim.x * blockDim.x) {
        uint8_t* row = desc + q * stride;
        bc_gen_row(s_card, n, seed, first + q, kmin, kmax, row);
        for (size_t b = 2 * (size_t)n; b < stride; ++b) row[b] = 0;
    }
}

static int gen_check(int n, int max_card, int kmin, int kmax) {
    if (n > 1024 || max_card > 256 || kmin < 0 || kmax < kmin) {
        bc_set_error("generator supports n_nodes <= 1024, domains <= 256, 0 <= kmin <= kmax");
        return BC_EINVAL;
    }
    return BC_OK;
}

extern "C" int bc_gen_range_queries(bc_model* m, uint64_t seed, uint64_t first, size_t n, int kmin, int kmax,
                                    void* desc_dev, void* stream) {
    if (!m || m->device < 0 || !desc_dev) { bc_set_error("bad arguments"); return BC_EINVAL; }
    int rc = gen_check(m->n, m->max_card, kmin, kmax);
    if (rc) return rc;
    if (n == 0) return BC_OK;
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    const int threads = 256;
    long long grid = (long long)((n + threads - 1) / threads);
    if (grid > (long long)m->sm_count * 8) grid = (long long)m->sm_count * 8;
    bc_gen_kernel<<<(int)grid, threads, m->n * sizeof(int32_t), static_cast<cudaStream_t>(stream)>>>(
        m->d_nodes, m->n, seed, first, n, kmin, kmax, static_cast<uint8_t*>(desc_dev),
        (size_t)bc_model_desc_stride(m, BC_DESC_RANGE_U8));
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch();
    return BC_OK;
}

extern "C" int bc_gen_range_queries_host(int n_nodes, const int32_t* card, uint64_t seed, uint64_t first, size_t n,
                                         int kmin, int kmax, void* desc_host) {
    if (!card || !desc_host || n_nodes <= 0) { bc_set_error("bad arguments"); return BC_EINVAL; }
    int mc = 0;
    for (int v = 0; v < n_nodes; ++v) mc = card[v] > mc ? card[v] : mc;
    int rc = gen_check(n_nodes, mc, kmin, kmax);
    if (rc) return rc;
    const size_t stride = (size_t)bc_round_up(2LL * n_nodes, 4);
    uint8_t* d = static_cast<uint8_t*>(desc_host);
    for (size_t q = 0; q < n; ++q) {
        uint8_t* row = d + q * stride;
        bc_gen_row(card, n_nodes, seed, first + q, kmin, kmax, row);
        for (size_t b = 2 * (size_t)n_nodes; b < stride; ++b) row[b] = 0;
    }
    return BC_OK;
}

extern "C" int bc_gen_sparse_queries_host(int n_nodes, const int32_t* card, uint64_t seed, uint64_t first, size_t n,
                                          int kmin, int kmax, uint32_t* row_off, uint32_t* entries, size_t* n_entries) {
    if (!card || !row_off || !entries || n_nodes <= 0) { bc_set_error("bad arguments"); return BC_EINVAL; }
    int mc = 0;
    for (int v = 0; v < n_nodes; ++v) mc = card[v] > mc ? card[v] : mc;
    int rc = gen_check(n_nodes, mc, kmin, kmax);
    if (rc) return rc;
    std::vector<uint8_t> row((size_t)bc_round_up(2LL * n_nodes, 4));
    size_t ne = 0;
    for (size_t q = 0; q < n; ++q) {
        bc_gen_row(card, n_nodes, seed, first + q, kmin, kmax, row.data());
        row_off[q] = (uint32_t)ne;
        for (int v = 0; v < n_nodes; ++v) {
            const int lo = row[2 * v], hi = row[2 * v + 1];
            if (lo > 0 || hi < card[v] - 1) entries[ne++] = (uint32_t)v | ((uint32_t)lo << 16) | ((uint32_t)hi << 24);
        }
    }
    row_off[n] = (uint32_t)ne;
    if (n_entries) *n_entries = ne;
    return BC_OK;
}

// ------------------------------------------------------------------------------------ FP32 peak
__global__ void __launch_bounds__(256) bc_ffma_kernel(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 123.456f) out[0] = s;  // keep the chain alive
}

extern "C" int bc_measure_fp32_peak(int device, double* tflops, double* sm_clock_mhz) {
    if (!tflops) { bc_set_error("tflops is NULL"); return BC_EINVAL; }
    BC_CUDA_CHECK(cudaSetDevice(device));
    int sms = 0, khz = 0;
    BC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    BC_CUDA_CHECK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
    float* d = nullptr;
    BC_CUDA_CHECK(cudaMalloc(&d, 4));
    cudaEvent_t e0, e1;
    BC_CUDA_CHECK(cudaEventCreate(&e0));
    BC_CUDA_CHECK(cudaEventCreate(&e1));
    const int grid = sms * 8, threads = 256, iters = 4096;
    double best = 0;
    for (int rep = 0; rep < 6; ++rep) {
        BC_CUDA_CHECK(cudaEventRecord(e0));
        bc_ffma_kernel<<<grid, threads>>>(d, iters, 0.999f, 0.001f);
        BC_CUDA_CHECK(cudaEventRecord(e1));
        BC_CUDA_CHECK(cudaEventSynchronize(e1));
        bc_count_launch();
        float ms = 0;
        BC_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 8 * 16 * (double)iters * grid * threads;
        const double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *tflops = best;
    if (sm_clock_mhz) *sm_clock_mhz = khz / 1000.0;
    return BC_OK;
}
