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

// ------------------------------------------------------------------------------------ marginal kernels
// One module per (model, target): "<cache_dir>/marg_<hash>.cubin" when present, otherwise the generated PTX through the
// driver JIT, exactly as for the spec module.  The slot of a target is replaced as a whole under marg_mu.
static int marg_attach(bc_model* m, int target, const void* image) {
    BC_CUDA_CHECK(cudaSetDevice(m->device));
    cudaLibrary_t lib = nullptr;
    char log[4096] = "";
    cudaJitOption opts[] = {cudaJitErrorLogBuffer, cudaJitErrorLogBufferSizeBytes};
    void* vals[] = {log, (void*)(uintptr_t)sizeof(log)};
    cudaError_t e = cudaLibraryLoadData(&lib, image, opts, vals, 2, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        bc_set_error("cudaLibraryLoadData failed for the marginal of node %d: %s %.600s", target, cudaGetErrorString(e), log);
        cudaGetLastError();
        return BC_ECOMPILE;
    }
    // {threads per CTA, results per query, marginal generator version, target}
    uint32_t meta[4] = {0, 0, 0, 0};
    void* dptr = nullptr;
    size_t gbytes = 0;
    if (cudaLibraryGetGlobal(&dptr, &gbytes, lib, "bc_marg_meta") == cudaSuccess && gbytes >= sizeof(meta))
        BC_CUDA_CHECK(cudaMemcpy(meta, dptr, sizeof(meta), cudaMemcpyDeviceToHost));
    else
        cudaGetLastError();
    BcMargSlot s;
    if (cudaLibraryGetKernel(&s.bits, lib, "bc_marg_bits") != cudaSuccess) { s.bits = nullptr; cudaGetLastError(); }
    if (cudaLibraryGetKernel(&s.dense, lib, "bc_marg_dense") != cudaSuccess) { s.dense = nullptr; cudaGetLastError(); }
    if (!s.bits || !s.dense || meta[0] == 0 || meta[0] > 1024 || meta[0] % 32 || meta[1] != (uint32_t)m->nodes[target].card ||
        meta[2] != BC_MARGINAL_VERSION || meta[3] != (uint32_t)target) {
        bc_set_error("image is not a marginal module of node %d (meta %u %u %u %u)", target, meta[0], meta[1], meta[2], meta[3]);
        cudaLibraryUnload(lib);
        return BC_ECUDA;
    }
    s.lib = lib;
    s.threads = (int)meta[0];
    auto blocks_of = [&](cudaKernel_t k) {
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void*)k, s.threads, 0) != cudaSuccess || nb <= 0) {
            cudaGetLastError();
            nb = 1;
        }
        return nb;
    };
    s.blocks_bits = blocks_of(s.bits);
    s.blocks_dense = blocks_of(s.dense);
    std::lock_guard<std::mutex> lock(m->marg_mu);
    if (m->marg.empty()) m->marg.resize(m->n);
    if (m->marg[target].lib) cudaLibraryUnload(m->marg[target].lib);
    m->marg[target] = s;
    return BC_OK;
}

int bc_marg_build(bc_model* m, int target, const char* cache_dir) {
    if (m->arena.empty()) {
        bc_set_error("model too large for a specialised kernel");
        return BC_ELIMIT;
    }
    if (cache_dir && *cache_dir) {
        char name[64];
        snprintf(name, sizeof(name), "/marg_%016llx.cubin", (unsigned long long)bc_marginal_hash_of(*m, target));
        std::ifstream f(std::string(cache_dir) + name, std::ios::binary);
        if (f) {
            std::string img((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
            if (!img.empty() && marg_attach(m, target, img.data()) == BC_OK) return BC_OK;
        }
    }
    const std::string ptx = bc_marginal_generate(*m, target);
    return marg_attach(m, target, ptx.c_str());
}

bool bc_marg_attached(bc_model* m, int target) {
    std::lock_guard<std::mutex> lock(m->marg_mu);
    return !m->marg.empty() && m->marg[target].lib != nullptr;
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

void bc_marg_free(bc_model* m) {
    for (BcMargSlot& s : m->marg)
        if (s.lib) cudaLibraryUnload(s.lib);
    m->marg.clear();
}
