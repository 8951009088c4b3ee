// Internal declarations shared by the translation units of libbayescard_b200.so.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <map>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/bayescard_b200.h"

#define BC_VERSION_STRING "bayescard_b200 0.1.0 (sm_100a)"
#define BC_CODEGEN_VERSION 10
#define BC_SPEC_CTR_SLOTS 256
#define BC_MARGINAL_VERSION 2   // marginal kernels (bc_marg_*): part of their cache name, independent of BC_CODEGEN_VERSION;
                                // 2: the kernels apply the fan-out mask
#define BC_JOINT_VERSION 1      // joint marginal kernels (bc_joint_*): part of their cache name
#define BC_JOINT_MAX_FFMA 32768 // FMA-pipe instructions per entry above which a pair gets no joint module (it expands)

// One record per node, copied to the device and (by K1) into shared memory.  32 bytes.
struct BcNodeRec {
    int32_t parent;      // topological index of the parent, -1 for the root
    int32_t card;        // number of states
    int32_t stride;      // row stride of T_v in floats
    int32_t lam_off;     // offset of this node's segment in a dense weight / lambda row (floats, multiple of 4)
    int64_t cpt_off;     // offset of T_v in the arena (floats)
    int32_t fan_off;     // offset of fanouts[v] in the fan arena (floats) or -1
    int32_t card_pa;     // card of the parent (1 for the root)
};

// Second per-node table (kept out of BcNodeRec so that record stays 32 bytes): BITS rows.
struct BcBitsRec {
    int32_t bit_off;     // first bit of this node's state mask in a BITS row
    int32_t card;
};

// Specialised marginal kernels of one target node, or joint marginal kernels of one pair of nodes (spec_jit.cu)
struct BcMargSlot {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t bits = nullptr, dense = nullptr;
    int threads = 0;
    int blocks_bits = 1, blocks_dense = 1;   // resident CTAs per SM
};

struct BcHostPipe;  // bc_api.cu
struct BcUmmaPlan;  // k2_umma.cu
struct BcK3Plan;    // k3_fused.cu

// State of the batched large-domain path (K2), built on first use.
struct BcK2Plan {
    std::vector<char> is_internal;     // node has children
    std::vector<double*> d_prefix;     // leaves: fp64 column prefix sums of T_v, (card+1) x card_pa
    BcUmmaPlan* umma = nullptr;        // tensor-core operands (transposed hi / lo CPTs, tensor maps)
    // Lambda workspace, kept between calls (grow only): calls on one model are serialised on ws_event, so a call
    // on another stream cannot overwrite the workspace of one that is still running
    float* d_ws = nullptr;
    size_t ws_bytes = 0;
    cudaEvent_t ws_event = nullptr;
};

struct bc_model {
    int device = -1;     // -1: host-only model (code generation / ahead-of-time build)
    int n = 0;
    std::vector<BcNodeRec> nodes;
    std::vector<float> arena;        // host copy (code generator input)
    std::vector<float> fan;
    std::vector<uint16_t> ent_node;  // node id of every entry of a lambda row
    std::vector<BcBitsRec> bits;     // BITS descriptor geometry
    int bits_words = 0;              // 32-bit words per BITS row (multiple of 4)
    int lam_total = 0;               // floats per lambda / dense row
    int max_card = 0;
    int mask_words = 1;
    int64_t flops_dense = 0;
    // device side
    float* d_arena = nullptr;
    size_t arena_floats_padded = 0;
    float* d_fan = nullptr;
    BcNodeRec* d_nodes = nullptr;
    BcBitsRec* d_bits = nullptr;
    uint32_t* d_bits_default = nullptr;  // BITS row of the unconstrained query (every state selected)
    float* d_dense_default = nullptr;    // DENSE_F32 row of the unconstrained query (1 on every state, 0 on row padding)
    uint16_t* d_ent_node = nullptr;
    int sm_count = 0;
    int smem_optin = 0;
    // specialised kernel
    cudaLibrary_t spec_lib = nullptr;
    cudaKernel_t spec_range8 = nullptr;
    cudaKernel_t spec_dense = nullptr;
    cudaKernel_t spec_bits = nullptr;
    int spec_threads = 0;            // threads per CTA (from the image's bc_spec_meta)
    int spec_qpt = 1;                // queries per thread per loop trip
    int spec_blocks_bits = 1, spec_blocks_dense = 1, spec_blocks_range8 = 1;  // resident CTAs per SM
    std::vector<uint32_t> bits_default;
    // work counters of the dynamically scheduled specialised kernels: a ring of {u64 next query, u32 CTAs done, pad}
    // slots (one per launch, so launches of one model on different streams never share a counter); each kernel
    // leaves its slot zeroed
    uint64_t* d_spec_ctr = nullptr;
    std::atomic<uint32_t> spec_ctr_next{0};
    // specialised marginal kernels, one slot per target node (empty until the first bc_model_specialize_marginal)
    std::vector<BcMargSlot> marg;
    std::map<std::pair<int, int>, BcMargSlot> joint;   // joint marginal kernels, keyed by the ordered pair (a, b)
    std::mutex marg_mu;                                // guards marg and joint
    BcK2Plan* k2 = nullptr;
    std::mutex k2_mu;                // guards the lazy construction of k2 (pipe_mu may already be held)
    BcK3Plan* k3 = nullptr;          // fused tensor-core tree kernel: edge schedule, TMEM columns, operand images
    std::mutex k3_mu;
    BcHostPipe* pipe = nullptr;
    std::mutex pipe_mu;
    // counts behind the CPTs (bc_model_set_counts / bc_model_update, bc_fit.cu): bc_fit_counts' layout, node v's counters
    // from cnt_off[v], its columns (one per parent state) from col_off[v]; both arrays end with the total
    unsigned long long* d_counts = nullptr;
    void* d_upd = nullptr;           // per-node table of the update kernels
    std::vector<int64_t> cnt_off, col_off;
    bool has_counts = false;
};

void bc_set_error(const char* fmt, ...);
void bc_count_launch(uint64_t n = 1);
// bc_api.cu: wait for the model's asynchronous host submissions; drop everything built from the CPT values (spec and
// marginal modules, K2 and K3 plans), which the next use rebuilds
int bc_pipe_quiesce_model(bc_model* m);
void bc_model_drop_cached(bc_model* m);

#define BC_CUDA_CHECK(expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            bc_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return BC_ECUDA;                                                                     \
        }                                                                                        \
    } while (0)

static inline int64_t bc_round_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// k1_generic.cu
int bc_k1_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask,
                 float* out, cudaStream_t stream, int32_t* out_exp = nullptr);
// bc_convert.cu
int bc_convert_launch(bc_model* m, const void* src, int src_fmt, void* dst, int dst_fmt, size_t nq, cudaStream_t stream);
int bc_expand_sparse_launch(bc_model* m, const uint32_t* row_off, const uint32_t* entries, size_t nq, void* dst_bits,
                            cudaStream_t stream);
int bc_expand_wsparse_launch(bc_model* m, const uint32_t* row_off, const uint32_t* words, size_t nq, float* dst_dense,
                             cudaStream_t stream);
#define BC_PACKED_BLOCK 128   // queries per blk_off entry of the PACKED wire format
void bc_packed_geometry(const bc_model* m, int* col_bits, int* state_bits);
// payload points at 32-bit word `word_base` of the bit stream (a slice of a larger batch keeps absolute entry indices)
int bc_expand_packed_launch(bc_model* m, const uint8_t* klen, const uint32_t* blk_off, const uint32_t* payload, unsigned long long word_base,
                            size_t nq, void* dst_bits, cudaStream_t stream);
// k2_batched.cu / k2_umma.cu
int bc_k2_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out, int use_umma,
                 cudaStream_t stream, int32_t* out_exp = nullptr);
void bc_k2_free(bc_model* m);
// one internal edge on the tensor cores; BC_ELIMIT = shape not served (caller falls back to FP32 SIMT)
int bc_k2_umma_edge(bc_model* m, const uint8_t* desc, size_t dstride, int fmt, size_t q0, int rows, int v, float* lam_v,
                    float* lam_v_lo, int ld_v, float* lam_pa, int ld_pa, int accumulate, cudaStream_t stream);
void bc_k2_umma_free(bc_model* m);
// k3_fused.cu: whole tree per 128-query tile on the tensor cores (BITS / DENSE_F32 rows); BC_ELIMIT = model not served
int bc_k3_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out, cudaStream_t stream,
                 int32_t* out_exp = nullptr);   // out_exp: scaled results (mantissa in out, exponent of two per query)
void bc_k3_free(bc_model* m);
// spec_codegen.cc
std::string bc_spec_generate(const bc_model& m);
uint64_t bc_spec_hash_of(const bc_model& m);
// spec_jit.cu
int bc_spec_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask,
                   float* out, cudaStream_t stream);
int bc_spec_attach(bc_model* m, const void* image, size_t bytes);
int bc_spec_build(bc_model* m, const char* cache_dir);
// marginal kernels: spec_codegen.cc (source, hash) and spec_jit.cu (attach, launch)
std::string bc_marginal_generate(const bc_model& m, int target);
uint64_t bc_marginal_hash_of(const bc_model& m, int target);
int bc_marg_build(bc_model* m, int target, const char* cache_dir);
bool bc_marg_attached(bc_model* m, int target);
int bc_marg_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, int target, float* out,
                   cudaStream_t stream);
void bc_marg_free(bc_model* m);   // unloads the marginal and the joint modules
// joint marginal kernels: spec_codegen.cc (source, hash; BC_ELIMIT above BC_JOINT_MAX_FFMA) and spec_jit.cu (attach, launch)
int bc_joint_generate(const bc_model& m, int a, int b, std::string* src);
uint64_t bc_joint_hash_of(const bc_model& m, int a, int b);
int bc_joint_build(bc_model* m, int a, int b, const char* cache_dir);
bool bc_joint_attached(bc_model* m, int a, int b);
int bc_joint_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, int a, int b, float* out,
                    cudaStream_t stream);
