// K-spec runtime: obtain the per-model image and launch it.
//
// bc_model_specialize() looks for an ahead-of-time cubin ("<cache_dir>/spec_<hash>.cubin", written by
// bayescard_b200/aot.py with `ptxas -arch=sm_100a`) and otherwise hands the generated PTX to the
// driver's JIT through cudaLibraryLoadData -- no NVRTC, no compiler on the serving box.
#include <cstdlib>
#include <cstring>
#include <fstream>

#include "bc_internal.h"

void bc_spec_geometry(const bc_model& m, int* threads, int* min_blocks);

namespace {

std::string cache_path(const bc_model& m, const char* dir) {
    char name[64];
    snprintf(name, sizeof(name), "/spec_%016llx.cubin", (unsigned long long)bc_spec_hash_of(m));
    return std::string(dir) + name;
}

}  // namespace

int bc_spec_attach(bc_model* m, const void* image, size_t bytes) {
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaLibrary_t lib = nullptr;
    // cubin (ELF) or NUL-terminated PTX; the image is copied by the driver during the call
    char log[4096] = "";
    cudaJitOption opts[] = {cudaJitErrorLogBuffer, cudaJitErrorLogBufferSizeBytes};
    void* vals[] = {log, (void*)(uintptr_t)sizeof(log)};
    cudaError_t e = cudaLibraryLoadData(&lib, image, opts, vals, 2, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        bc_set_error("cudaLibraryLoadData failed: %s %.600s", cudaGetErrorString(e), log);
        cudaGetLastError();
        return BC_ECOMPILE;
    }
    // geometry travels with the image: {threads per CTA, queries per thread and trip, generator version, 0}
    uint32_t meta[4] = {128, 1, 0, 0};
    void* dptr = nullptr;
    size_t gbytes = 0;
    if (cudaLibraryGetGlobal(&dptr, &gbytes, lib, "bc_spec_meta") == cudaSuccess && gbytes >= sizeof(meta))
        BC_CUDA_CHECK(cudaMemcpy(meta, dptr, sizeof(meta), cudaMemcpyDeviceToHost));
    else
        cudaGetLastError();
    // an image may hold any subset of the entry points; formats without one use the generic kernel.  Generator versions
    // >= 5 emit no RANGE_U8 entry point (range rows are converted to BITS rows): it is only looked up in older images, so
    // that attaching a current image makes no failing API call (keeps compute-sanitizer's API-error report empty)
    cudaKernel_t kr = nullptr, kd = nullptr, kb = nullptr;
    if (cudaLibraryGetKernel(&kd, lib, "bc_spec_dense") != cudaSuccess) { kd = nullptr; cudaGetLastError(); }
    if (meta[2] < 5 && cudaLibraryGetKernel(&kr, lib, "bc_spec_range8") != cudaSuccess) { kr = nullptr; cudaGetLastError(); }
    if (cudaLibraryGetKernel(&kb, lib, "bc_spec_bits") != cudaSuccess) { kb = nullptr; cudaGetLastError(); }
    if (!kd && !kr && !kb) {
        bc_set_error("specialised image has none of bc_spec_bits / bc_spec_range8 / bc_spec_dense");
        cudaLibraryUnload(lib);
        return BC_ECUDA;
    }
    if (meta[0] == 0 || meta[0] > 1024 || meta[0] % 32) {
        bc_set_error("specialised image declares %u threads per CTA", meta[0]);
        cudaLibraryUnload(lib);
        return BC_ECUDA;
    }
    if (m->spec_lib) cudaLibraryUnload(m->spec_lib);
    m->spec_lib = lib;
    m->spec_range8 = kr;
    m->spec_dense = kd;
    m->spec_bits = kb;
    m->spec_threads = (int)meta[0];
    m->spec_qpt = meta[1] ? (int)meta[1] : 1;
    auto blocks_of = [&](cudaKernel_t k) {
        int nb = 0;
        if (!k || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void*)k, m->spec_threads, 0) != cudaSuccess || nb <= 0) {
            cudaGetLastError();
            nb = 1;
        }
        return nb;
    };
    m->spec_blocks_bits = blocks_of(kb);
    m->spec_blocks_dense = blocks_of(kd);
    m->spec_blocks_range8 = blocks_of(kr);
    return BC_OK;
}

int bc_spec_build(bc_model* m, const char* cache_dir) {
    if (m->arena.empty()) {
        bc_set_error("model too large for a specialised kernel");
        return BC_ELIMIT;
    }
    if (cache_dir && *cache_dir) {
        std::ifstream f(cache_path(*m, cache_dir), std::ios::binary);
        if (f) {
            std::string img((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
            if (!img.empty() && bc_spec_attach(m, img.data(), img.size()) == BC_OK) return BC_OK;
        }
    }
    const std::string ptx = bc_spec_generate(*m);  // std::string::c_str() is NUL terminated
    return bc_spec_attach(m, ptx.c_str(), ptx.size() + 1);
}

int bc_spec_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out,
                   cudaStream_t stream) {
    cudaKernel_t k = fmt == BC_DESC_DENSE_F32 ? m->spec_dense : fmt == BC_DESC_BITS ? m->spec_bits : m->spec_range8;
    if (!k) {
        bc_set_error("no specialised kernel for descriptor format %d", fmt);
        return BC_ECOMPILE;
    }
    const unsigned char* d = static_cast<const unsigned char*>(desc);
    unsigned long long stride = (unsigned long long)bc_model_desc_stride(m, fmt);
    unsigned long long n = nq;
    if (!m->d_spec_ctr) {
        bc_set_error("model has no work-counter ring (host-only model?)");
        return BC_EINVAL;
    }
    uint64_t* ctr = m->d_spec_ctr + 2 * (m->spec_ctr_next.fetch_add(1) % BC_SPEC_CTR_SLOTS);
    void* args[] = {(void*)&d, (void*)&stride, (void*)&fan_mask, (void*)&out, (void*)&n, (void*)&ctr};
    const int threads = m->spec_threads;
    const size_t per_cta = (size_t)threads * m->spec_qpt;
    const int resident = fmt == BC_DESC_DENSE_F32 ? m->spec_blocks_dense : fmt == BC_DESC_BITS ? m->spec_blocks_bits : m->spec_blocks_range8;
    // persistent grid: a whole number of CTAs per SM; smaller batches get one CTA per 'per_cta' queries
    long long grid = (long long)m->sm_count * resident;
    const long long needed = (long long)((nq + per_cta - 1) / per_cta);
    if (grid > needed) grid = needed;
    BC_CUDA_CHECK(cudaLaunchKernel((const void*)k, dim3((unsigned)grid), dim3(threads), args, 0, stream));
    bc_count_launch();
    return BC_OK;
}

// ------------------------------------------------------------------------------------ marginal and joint kernels
// One module per (model, target) or (model, a, b): "<cache_dir>/marg_<hash>.cubin" / "joint_<hash>.cubin" when present,
// otherwise the generated PTX through the driver JIT, exactly as for the spec module.  A slot is replaced as a whole under
// marg_mu.

// Loads an image with the entries bc_<kind>_bits / bc_<kind>_dense and reads its four-word global bc_<kind>_meta
// (threads per CTA first); the caller checks the rest of meta.  BC_ECUDA (image unloaded) without both entries or with a
// thread count a CTA cannot have.
static int module_load(bc_model* m, const void* image, const char* kind, const char* what, uint32_t meta[4], BcMargSlot* s) {
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaLibrary_t lib = nullptr;
    char log[4096] = "";
    cudaJitOption opts[] = {cudaJitErrorLogBuffer, cudaJitErrorLogBufferSizeBytes};
    void* vals[] = {log, (void*)(uintptr_t)sizeof(log)};
    cudaError_t e = cudaLibraryLoadData(&lib, image, opts, vals, 2, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        bc_set_error("cudaLibraryLoadData failed for %s: %s %.600s", what, cudaGetErrorString(e), log);
        cudaGetLastError();
        return BC_ECOMPILE;
    }
    const std::string k = kind;
    void* dptr = nullptr;
    size_t gbytes = 0;
    if (cudaLibraryGetGlobal(&dptr, &gbytes, lib, ("bc_" + k + "_meta").c_str()) == cudaSuccess && gbytes >= 4 * sizeof(uint32_t)) {
        e = cudaMemcpy(meta, dptr, 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            bc_set_error("reading the meta of %s: %s", what, cudaGetErrorString(e));
            cudaLibraryUnload(lib);
            return BC_ECUDA;
        }
    } else {
        cudaGetLastError();
    }
    if (cudaLibraryGetKernel(&s->bits, lib, ("bc_" + k + "_bits").c_str()) != cudaSuccess) { s->bits = nullptr; cudaGetLastError(); }
    if (cudaLibraryGetKernel(&s->dense, lib, ("bc_" + k + "_dense").c_str()) != cudaSuccess) { s->dense = nullptr; cudaGetLastError(); }
    if (!s->bits || !s->dense || meta[0] == 0 || meta[0] > 1024 || meta[0] % 32) {
        bc_set_error("image is not a module of %s (meta %u %u %u %u)", what, meta[0], meta[1], meta[2], meta[3]);
        cudaLibraryUnload(lib);
        return BC_ECUDA;
    }
    s->lib = lib;
    s->threads = (int)meta[0];
    auto blocks_of = [&](cudaKernel_t kk) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void*)kk, s->threads, 0) != cudaSuccess || nb <= 0) {
            cudaGetLastError();
            nb = 1;
        }
        return nb;
    };
    s->blocks_bits = blocks_of(s->bits);
    s->blocks_dense = blocks_of(s->dense);
    return BC_OK;
}

static int marg_attach(bc_model* m, int target, const void* image) {
    char what[64];
    snprintf(what, sizeof(what), "the marginal of node %d", target);
    // {threads per CTA, results per query, marginal generator version, target}
    uint32_t meta[4] = {0, 0, 0, 0};
    BcMargSlot s;
    int rc = module_load(m, image, "marg", what, meta, &s);
    if (rc != BC_OK) return rc;
    if (meta[1] != (uint32_t)m->nodes[target].card || meta[2] != BC_MARGINAL_VERSION || meta[3] != (uint32_t)target) {
        bc_set_error("image is not a marginal module of node %d (meta %u %u %u %u)", target, meta[0], meta[1], meta[2], meta[3]);
        cudaLibraryUnload(s.lib);
        return BC_ECUDA;
    }
    std::lock_guard<std::mutex> lock(m->marg_mu);
    if (m->marg.empty()) m->marg.resize(m->n);
    if (m->marg[target].lib) cudaLibraryUnload(m->marg[target].lib);
    m->marg[target] = s;
    return BC_OK;
}

static bool read_file(const std::string& path, std::string* img) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return false;
    img->assign((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    return !img->empty();
}

int bc_marg_build(bc_model* m, int target, const char* cache_dir) {
    if (m->arena.empty()) {
        bc_set_error("model too large for a specialised kernel");
        return BC_ELIMIT;
    }
    if (cache_dir && *cache_dir) {
        char name[64];
        snprintf(name, sizeof(name), "/marg_%016llx.cubin", (unsigned long long)bc_marginal_hash_of(*m, target));
        std::string img;
        if (read_file(std::string(cache_dir) + name, &img) && marg_attach(m, target, img.data()) == BC_OK) return BC_OK;
    }
    const std::string ptx = bc_marginal_generate(*m, target);
    return marg_attach(m, target, ptx.c_str());
}

bool bc_marg_attached(bc_model* m, int target) {
    std::lock_guard<std::mutex> lock(m->marg_mu);
    return !m->marg.empty() && m->marg[target].lib != nullptr;
}

// One launch of a marginal or joint slot: persistent grid of resident CTAs, a fresh work counter of the ring.
static int slot_launch(bc_model* m, const BcMargSlot& s, cudaKernel_t k, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask,
                       float* out, cudaStream_t stream) {
    const unsigned char* d = static_cast<const unsigned char*>(desc);
    unsigned long long stride = (unsigned long long)bc_model_desc_stride(m, fmt);
    unsigned long long n = nq;
    uint64_t* ctr = m->d_spec_ctr + 2 * (m->spec_ctr_next.fetch_add(1) % BC_SPEC_CTR_SLOTS);
    void* args[] = {(void*)&d, (void*)&stride, (void*)&fan_mask, (void*)&out, (void*)&n, (void*)&ctr};
    const int resident = fmt == BC_DESC_DENSE_F32 ? s.blocks_dense : s.blocks_bits;
    long long grid = (long long)m->sm_count * resident;
    const long long needed = (long long)((nq + s.threads - 1) / s.threads);
    if (grid > needed) grid = needed;
    BC_CUDA_CHECK(cudaLaunchKernel((const void*)k, dim3((unsigned)grid), dim3(s.threads), args, 0, stream));
    bc_count_launch();
    return BC_OK;
}

int bc_marg_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, int target, float* out,
                   cudaStream_t stream) {
    BcMargSlot s;
    {
        std::lock_guard<std::mutex> lock(m->marg_mu);
        if (!m->marg.empty()) s = m->marg[target];
    }
    cudaKernel_t k = fmt == BC_DESC_DENSE_F32 ? s.dense : fmt == BC_DESC_BITS ? s.bits : nullptr;
    if (!s.lib || !k) {
        bc_set_error("no specialised marginal kernel of node %d for descriptor format %d (call bc_model_specialize_marginal)",
                     target, fmt);
        return BC_ECOMPILE;
    }
    return slot_launch(m, s, k, desc, nq, fmt, fan_mask, out, stream);
}

static int joint_attach(bc_model* m, int a, int b, const void* image) {
    char what[64];
    snprintf(what, sizeof(what), "the joint marginal of nodes %d, %d", a, b);
    // {threads per CTA, a, b, joint generator version}
    uint32_t meta[4] = {0, 0, 0, 0};
    BcMargSlot s;
    int rc = module_load(m, image, "joint", what, meta, &s);
    if (rc != BC_OK) return rc;
    if (meta[1] != (uint32_t)a || meta[2] != (uint32_t)b || meta[3] != BC_JOINT_VERSION) {
        bc_set_error("image is not a joint marginal module of nodes %d, %d (meta %u %u %u %u)", a, b, meta[0], meta[1], meta[2], meta[3]);
        cudaLibraryUnload(s.lib);
        return BC_ECUDA;
    }
    std::lock_guard<std::mutex> lock(m->marg_mu);
    BcMargSlot& slot = m->joint[{a, b}];
    if (slot.lib) cudaLibraryUnload(slot.lib);
    slot = s;
    return BC_OK;
}

int bc_joint_build(bc_model* m, int a, int b, const char* cache_dir) {
    if (m->arena.empty()) {
        bc_set_error("model too large for a specialised kernel");
        return BC_ELIMIT;
    }
    if (cache_dir && *cache_dir) {
        char name[64];
        snprintf(name, sizeof(name), "/joint_%016llx.cubin", (unsigned long long)bc_joint_hash_of(*m, a, b));
        std::string img;
        if (read_file(std::string(cache_dir) + name, &img) && joint_attach(m, a, b, img.data()) == BC_OK) return BC_OK;
    }
    std::string ptx;
    const int rc = bc_joint_generate(*m, a, b, &ptx);
    if (rc != BC_OK) return rc;
    return joint_attach(m, a, b, ptx.c_str());
}

bool bc_joint_attached(bc_model* m, int a, int b) {
    std::lock_guard<std::mutex> lock(m->marg_mu);
    auto it = m->joint.find({a, b});
    return it != m->joint.end() && it->second.lib != nullptr;
}

int bc_joint_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, int a, int b, float* out,
                    cudaStream_t stream) {
    BcMargSlot s;
    {
        std::lock_guard<std::mutex> lock(m->marg_mu);
        auto it = m->joint.find({a, b});
        if (it != m->joint.end()) s = it->second;
    }
    cudaKernel_t k = fmt == BC_DESC_DENSE_F32 ? s.dense : fmt == BC_DESC_BITS ? s.bits : nullptr;
    if (!s.lib || !k) {
        bc_set_error("no joint marginal kernel of nodes %d, %d for descriptor format %d (call bc_model_specialize_joint)", a, b, fmt);
        return BC_ECOMPILE;
    }
    return slot_launch(m, s, k, desc, nq, fmt, fan_mask, out, stream);
}

void bc_marg_free(bc_model* m) {
    for (BcMargSlot& s : m->marg)
        if (s.lib) cudaLibraryUnload(s.lib);
    m->marg.clear();
    for (auto& kv : m->joint)
        if (kv.second.lib) cudaLibraryUnload(kv.second.lib);
    m->joint.clear();
}
