// K3 -- fused whole-tree sum-product on the tensor cores: one CTA per SM carries tiles of 128 queries through EVERY
// edge of the tree without leaving the SM.
//
//     out[q] = sum_x prod_v w_v[x_v] * T_v[x_v, x_pa(v)]        (VariableEliminationJIT.query / .expectation,
//                                                                 reference Pgmpy/inference/ExactInference.py:112-287)
//
// evaluated leaf -> root as one small GEMM per edge v -> pa(v) (SURVEY.md section 0.5):
//
//     D[128 x N]  = U_v[128 x K] . T_v[K x N]        U_v = w_v (*) Lambda_v,  K = card(v), N = card(pa)
//     Lambda_pa  *= D
//
// What the schedule is built on (MEASURED, tools/microbench/umma_chain.cu, profiles/r2_microbench_umma_chain.txt):
//   * tcgen05.mma.kind::tf32 M128 x N x K8 instructions that accumulate into the SAME tensor-memory columns pipeline
//     at the floor rate (N / 2 clk each; 1 chain == 4 chains) -- there is no dependent-chain penalty;
//   * with the A operand in SHARED memory an instruction costs 32 + N / 4 clk (4 KB of A + 32 N bytes of B per instruction
//     over the 128 B/clk shared-memory port: N = 96 -> 56 clk), on top of the producers' and TMA's writes into the same
//     port; with A in TENSOR memory it runs at the floor for every N >= 32;
//   * tcgen05.ld moves ~190 B/clk/SM and neither slows the MMAs down nor is slowed by them.
// Hence (round 2): the operand U_v is written by the producer warps straight into a ring of TENSOR-MEMORY columns
// (tcgen05.st: hi and lo TF32 halves, 32 columns each per block of 32 child states) and read from there by the MMAs;
// shared memory only carries T_v^T (TMA) and the staged query weights.
//
// Roles (576 threads, one CTA per SM, all 512 tensor-memory columns):
//   * warps 0-3 / 4-7  TWO PRODUCER GROUPS (thread = query = TMEM lane) build alternate blocks: weights from the BITS tile
//     in shared memory or, for DENSE_F32 rows, from a shared-memory ring that the TMA warp fills with 2-D tensor-map loads
//     (128 queries x 32 floats, 128-byte swizzle) -- no global-memory latency in the loop; times the fan-out vector, times
//     Lambda_v (tcgen05.ld) for an internal node; split into TF32 hi (round to nearest) and lo = x - hi; tcgen05.st into the
//     A ring; one mbarrier arrive per warp;
//   * warps 8-11 / 14-17  TWO EPILOGUE GROUPS, each owning one half of the parent's columns: over a run of consecutive edges
//     into the same parent, Lambda_pa stays in REGISTERS (only D is read from tensor memory per edge -- TMEM reads are the
//     slow direction); at the end of a run it is written to tensor memory and published ("Lambda_v complete", one mbarrier
//     per internal edge) to the producers, or, for the root, folded into the tile's result on the spot;
//   * warp 12          MMA ISSUER (whole warp converged, elect.sync inside the asm, edge table in the kernel-parameter bank
//     so that every tcgen05 operand lives in uniform registers): error-compensated 3xTF32, A_lo.B_hi + A_hi.B_lo first, then
//     A_hi.B_hi (A_lo = 0 and skipped for unit-weight leaves); tcgen05.commit frees the A and B slots and hands the accumulator
//     to the epilogue warps;
//   * warp 13          TMA WARP: T_v^T blocks (hi and lo, pre-split and pre-swizzled once per model into an "operand image",
//     L2 resident) by ONE bulk copy per step, and the DENSE weight blocks; the step sequence is static, so both rings run
//     ahead across edges and tiles.
// Lambda_v of every live internal node sits in tensor memory (one fp32 column per state) from the end of the run that
// completes it; the columns are assigned on the host by first fit over the nodes' lifetimes in the edge schedule.
//
// Step sequence (K3Params::seq): the chain at the top of the tree -- edges that are each the only message into their parent --
// is cut off a tile's own pass and interleaved with the body of the CTA's NEXT tile (every hop of it waits for the complete
// result of the one before; alone it left the tensor pipe idle for 35-40 % of a tile).  Every role walks the same static
// (edge, tile) sequence; k3_kernel<FMT, true> additionally carries a power-of-two exponent per query through the epilogue
// (results beyond the fp32 range).  A CTA's timeline, measured with the clock stamps of BC_K3_TRACE_BUILD, and what bounds
// the kernel now are in DESIGN.md section 4.
//
// Algorithmic work per query = flops_dense(model) (every CPT entry once); HBM traffic = descriptor row + 4 B.
#include <cuda.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <memory>

#include "bc_internal.h"

struct K3Edge {            // 64 bytes, in the kernel parameter bank
    int32_t v, K, N, n_pad;
    int32_t lam_off;       // first float of column v in a DENSE row
    int32_t bit_off;       // first bit of column v in a BITS row
    int32_t fan_off;       // fanouts[v] in the fan arena, -1 if none
    int32_t col_v;         // TMEM column of Lambda_v, -1 for a leaf
    int32_t col_pa;        // TMEM column of Lambda_pa
    int32_t first;         // this edge is the first message into Lambda_pa
    int32_t nkb;           // blocks of 32 child states
    uint32_t idesc;        // tcgen05 instruction descriptor (M = 128, N = n_pad, TF32 x TF32 -> F32, K-major)
    uint64_t bimg_off;     // byte offset of the edge's operand images
    int32_t publish;       // >= 0: this edge is the LAST message into Lambda_pa, pa's own edge is `publish` (its producers may
                           // start); -2: ... and pa is the root (the tile's result follows); -1: more messages to come
    int32_t flags;         // kRunFirst / kRunLast: first / last edge of a RUN of consecutive edges into the same parent (the epilogue warps keep
                           // the parent's message in registers over a run); kRegs: the parent's domain fits the register accumulators
};
enum { kRunFirst = 1, kRunLast = 2, kRegs = 4 };
static_assert(sizeof(K3Edge) == 64, "K3Edge layout");

struct BcK3Plan {
    int failed = 0;
    std::vector<K3Edge> edges;
    std::vector<uint8_t> seq;      // step sequence of one pass (K3Params::seq)
    int n_tail = 0;
    uint8_t* d_bimg = nullptr;
    size_t bimg_bytes = 0;
    int npad_max = 16;
    int tmem_cols = 512;
    int a_col = 0, a_stages = 2;   // A ring: a_stages x 64 columns (32 hi + 32 lo)
    int d_col = 0, n_dbuf = 2;
    int b_stages = 4, w_stages = 4;
    int root_col = 0;
    int ctas_per_sm = 1;
    size_t smem = 0;
    void* encode = nullptr;        // cuTensorMapEncodeTiled (DENSE_F32 rows are staged by 2-D TMA loads)
};

namespace {

constexpr int kTile = 128;     // queries per CTA tile = TMEM lanes = UMMA M
constexpr int kMaxEdges = 127; // trees of up to 128 columns
// Longest contraction an edge may have (states of its child column).  All k-steps of an edge (three TF32 products per 8 states)
// accumulate into ONE fp32 accumulator in tensor memory, and the error grows with the number of chained accumulations (as in
// K2, see UmmaCfg in k2_umma.cu): 229-256-state columns (96 chained MMAs) came out up to 1.6e-5 off the fp64 oracle on DENSE
// rows with fan-out columns, beyond the 1e-5 the kernels are held to.  Columns of <= 128 states (48 MMAs; the shipped models
// have <= 84) stay within it.
constexpr int kMaxK = 128;
constexpr int kBK = 32;        // child states per ring step: one 128-byte row of T_v^T / of the weight box (128-byte swizzle), 4 k-steps of 8
constexpr int kStagesW = 8;    // DENSE weight ring: at most this many slots of 16 KB (K3Params::w_stages are used; the loads come from HBM)
constexpr int kWBytes = kTile * kBK * 4;
constexpr int kGroups = 2;     // producer groups of four warps, alternate blocks
constexpr int kWarpEpi = 4 * kGroups, kWarpMma = kWarpEpi + 4, kWarpTma = kWarpMma + 1, kWarpEpiB = kWarpTma + 1;
constexpr int kThreads = 32 * (kWarpEpiB + 4);   // two epilogue groups of four warps (one warp per TMEM lane quarter: warp % 4)
constexpr int kAcc = 48;       // message columns an epilogue thread keeps in registers (each group owns one half of the parent's columns)
constexpr int kMaxStages = 8;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct K3Params {
    K3Edge edge[kMaxEdges];    // in the kernel parameter bank (8 KB of the 32 KB sm_100 allows): uniform loads, warp-uniform control flow
    int n_edges;
    // the step sequence of one pass: entry = edge index | 0x80 for a TAIL edge, which belongs to the PREVIOUS tile of this CTA
    // (the chain at the top of the tree is folded under the next tile's leaves; see k3_prepare)
    uint8_t seq[kMaxEdges + 1];
    int n_seq, n_tail;
    int prefetch;              // fetch the next tile's BITS rows / mask words one pass ahead (BC_K3_NO_PREFETCH=1 turns it off)
    const uint8_t* bimg;
    const uint8_t* desc;
    size_t dstride;
    const uint32_t* fan_mask;
    const float* fan;
    int fan_floats;            // multiple of 4 (shared-memory copy, zero padded)
    int fan_n;                 // floats in the fan arena
    const float* root_T;       // T_root in the arena
    int root_card, root_col, root_bit_off, root_lam_off, root_fan_off;
    float* out;
    int32_t* out_exp;          // scaled results (k3_kernel<FMT, true>): out[q] * 2^out_exp[q]
    size_t nq;
    long long n_tiles;
    int bits_words;
    int b_slot_bytes;          // 2 * npad_max * 128
    int a_col, a_stages, b_stages, w_stages;
    int d_col, d_stride, n_dbuf;
    int mask_words;            // fan-out mask words per query
    float debias_unit;         // optional correction of the accumulator's truncation (BC_K3_DEBIAS, 0 = off = default)
    long long* trace;          // BC_K3_TRACE: clock64 stamps of CTA 0's fifth tile, [role][edge][2] (nullptr = off)
};
constexpr int kTraceTile = 4;
constexpr int kCnt = 4 * kMaxEdges * 2;   // per-step stamps behind the per-edge stamps: [step of the tile][8]
constexpr int kTraceSteps = 64;
#ifndef BC_K3_TRACE_BUILD
#define BC_K3_TRACE_BUILD 0   // 1: compile the clock stamps in (they cost issue slots in every role); BC_K3_TRACE=1 then prints them
#endif
#if BC_K3_TRACE_BUILD
#define K3_STAMP(role, e, k)                                                                                   \
    do {                                                                                                       \
        if (P.trace != nullptr && blockIdx.x == 0 && tile_iter == kTraceTile && lane == 0)                     \
            P.trace[((role) * kMaxEdges + (e)) * 2 + (k)] = clock64();                                         \
    } while (0)
// per-step stamps go to SHARED memory (a global read-modify-write per stamp would perturb what it measures) and are copied out
// at the end of the kernel: slots 0-4 producer (start, inputs ready, Lambda loaded, A slot free, stored + arrived)
#define K3_STEP(slot)                                                                                                    \
    do {                                                                                                                 \
        if (P.trace != nullptr && blockIdx.x == 0 && tile_iter == kTraceTile && lane == 0 && step_in_tile < kTraceSteps)  \
            s_trace[step_in_tile * 8 + (slot)] = clock64();                                                              \
    } while (0)
#else
#define K3_STAMP(role, e, k) do { (void)tile_iter; } while (0)
#define K3_STEP(slot) do { (void)step_in_tile; } while (0)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// (with the default time limit a failed try_wait comes back after ~50 clk and the spin loops of the 18 warps are 21 % of all
//  issued instructions -- ncu, profiles/r2_ncu_29_k3_dense_imdb1.json; with a suspend-time hint ptxas emits NANOSLEEP.SYNCS and the
//  spinning stops.  Measured: no change in throughput for hints of 100 ns ... 20 us -- the spinning warps only took issue slots
//  nobody else wanted -- so this is about power, not speed)
#ifndef BC_K3_SPLIT_CVT
#define BC_K3_SPLIT_CVT 0
#endif
#ifndef BC_K3_SUSPEND_NS
#define BC_K3_SUSPEND_NS 500
#endif
constexpr unsigned kSuspendNs = BC_K3_SUSPEND_NS;
__device__ __forceinline__ void mbar_wait(uint32_t bar, unsigned parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity), "r"(kSuspendNs)
        : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, unsigned bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
}
// D[tmem] (+)= A[tmem: 128 lanes x 8 columns] . B[smem, K-major, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (SBO),
// layout type 4, version 1 (sm_100)].  Called by the WHOLE (converged) issuer warp; elect.sync inside picks the lane, so ptxas
// keeps every operand in uniform registers instead of wrapping each instruction in a divergence loop.
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_c, uint32_t tmem_a, uint32_t b_lo32, uint32_t desc_hi32, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p, q;\n.reg .b64 db;\nelect.sync _|q, 0xffffffff;\nsetp.ne.b32 p, %5, 0;\n"
        "mov.b64 db, {%2, %3};\n"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], db, %4, p;\n}\n" ::"r"(tmem_c),
        "r"(tmem_a), "r"(b_lo32), "r"(desc_hi32), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {   // whole warp, one elected lane
    asm volatile(
        "{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}\n" ::"r"(bar)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
                 "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
        "%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
    const uint32_t* r = reinterpret_cast<const uint32_t*>(v);
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
        "%30,%31,%32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
        "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// x = hi + lo, hi = x rounded to the nearest TF32 number (ties away from zero: two integer instructions); lo = x - hi is
// exact in fp32 and symmetric around zero, so the tensor core's truncation of its low bits is unbiased
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
#if BC_K3_SPLIT_CVT
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x));   // round to nearest, ties away: one instruction
    hi = __uint_as_float(h);
#else
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
#endif
    lo = x - hi;
}

// selection bits of states [c0, c0 + 16) of a column for this thread's query (bits past the domain cleared)
__device__ __forceinline__ uint32_t bits16(const uint32_t* my_bits, int bits_words, int bit_off, int card, int c0) {
    const int b0 = bit_off + c0, idx = b0 >> 5, sh = b0 & 31;
    const uint32_t w0 = my_bits[idx * kTile];
    const uint32_t w1 = my_bits[(idx + 1 < bits_words ? idx + 1 : idx) * kTile];
    const int valid = card - c0;
    return __funnelshift_r(w0, w1, sh) & (valid >= 16 ? 0xFFFFu : ((1u << valid) - 1u));
}

// ... of states [c0, c0 + 32)
__device__ __forceinline__ uint32_t bits32(const uint32_t* my_bits, int bits_words, int bit_off, int card, int c0) {
    const int b0 = bit_off + c0, idx = b0 >> 5, sh = b0 & 31;
    const uint32_t w0 = my_bits[idx * kTile];
    const uint32_t w1 = my_bits[(idx + 1 < bits_words ? idx + 1 : idx) * kTile];
    const int valid = card - c0;
    return __funnelshift_r(w0, w1, sh) & (valid >= 32 ? 0xFFFFFFFFu : ((1u << valid) - 1u));
}

// weights of 8 consecutive states [c0, c0 + 8) of a column for this thread's query (the root's dot product)
template <int FMT>
__device__ __forceinline__ void weights8(const uint32_t* my_bits, int bits_words, const float* drow, int lam_off, int bit_off, int card, int c0,
                                         float* w) {
    if (FMT == BC_DESC_BITS) {
        const uint32_t m = bits16(my_bits, bits_words, bit_off, card, c0);
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = ((m >> j) & 1u) ? 1.f : 0.f;
    } else {
        const float4 a = __ldg(reinterpret_cast<const float4*>(drow + lam_off + c0));
        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c0 + 4 < card) b = __ldg(reinterpret_cast<const float4*>(drow + lam_off + c0 + 4));
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (c0 + j >= card) w[j] = 0.f;   // row padding / the next column's weights never contribute
    }
}

// Every role walks the same static sequence of (edge, tile) steps: pass `iter` of a CTA runs the body edges of its tile number
// `iter` interleaved with the TAIL edges (K3Params::seq) of tile `iter - 1`; one extra pass drains the last tile's tail.
#define K3_PASS_HEAD                                                                  \
    const long long tile_cur = (long long)blockIdx.x + (long long)iter * gridDim.x;   \
    const bool cur_ok = tile_cur < P.n_tiles;                                         \
    if (!cur_ok && (iter == 0 || P.n_tail == 0)) break;
#define K3_STEP_HEAD                                                                  \
    const int e = P.seq[si] & 127;                                                    \
    const bool back = (P.seq[si] & 128) != 0;                                         \
    if (back ? iter == 0 : !cur_ok) continue;                                         \
    const long long tile = back ? tile_cur - (long long)gridDim.x : tile_cur;         \
    const uint32_t tile_iter = back ? iter - 1u : iter;                               \
    (void)tile; (void)tile_iter;

struct Ring {   // slot / parity cursor of a ring of `n` slots advanced once per step
    uint32_t s = 0, par = 0;
    __device__ __forceinline__ void next(uint32_t n) {
        if (++s == n) { s = 0; par ^= 1u; }
    }
};

template <int FMT, bool SCALED>
__global__ void __launch_bounds__(kThreads, 1) k3_kernel(const __grid_constant__ K3Params P, const __grid_constant__ CUtensorMap tm_w) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler (role dispatch without divergence)
    // carve-up: B ring | W ring (DENSE) | BITS rows of two tiles [word][query] | fan-out mask of two tiles | fan arena | table | barriers
    uint8_t* p = smem;
    const uint32_t b_ring = smem_u32(p);
    p += (size_t)P.b_stages * P.b_slot_bytes;
    const uint32_t w_ring = smem_u32(p);
    const uint8_t* w_ring_ptr = p;
    p += (FMT == BC_DESC_DENSE_F32 ? (size_t)P.w_stages * kWBytes : 0);
    uint32_t* s_bits = reinterpret_cast<uint32_t*>(p);
    const size_t bits_tile = (FMT == BC_DESC_BITS ? (size_t)P.bits_words * kTile : 0);
    p += 2 * bits_tile * 4;
    uint32_t* s_fm = reinterpret_cast<uint32_t*>(p);
    const size_t fm_tile = (size_t)P.mask_words * kTile;
    p += 2 * fm_tile * 4;
    float* s_fan = reinterpret_cast<float*>(p);
    p += (size_t)P.fan_floats * 4;
    float4* s_tab = reinterpret_cast<float4*>(p);   // nibble -> four 0/1 floats
    p += 256;
    float* s_part = reinterpret_cast<float*>(p);    // the second epilogue group's share of the root's dot product, two tiles
    p += 2 * kTile * 4;
    float* s_max = reinterpret_cast<float*>(p);     // SCALED: row maxima exchanged between the two epilogue groups [exchange parity][group][query]
    p += 4 * kTile * 4;
    uint64_t* bars = reinterpret_cast<uint64_t*>(p);
    const uint32_t a_full0 = smem_u32(bars), a_empty0 = a_full0 + 8 * kMaxStages, b_full0 = a_empty0 + 8 * kMaxStages,
                   b_empty0 = b_full0 + 8 * kMaxStages, w_full0 = b_empty0 + 8 * kMaxStages, w_empty0 = w_full0 + 8 * kStagesW,
                   d_full0 = w_empty0 + 8 * kStagesW, d_empty0 = d_full0 + 16, bits_free0 = d_empty0 + 16, lam_ready0 = bits_free0 + 32;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * kMaxStages + 2 * kStagesW + 8 + kMaxEdges + 1);
    long long* s_trace = reinterpret_cast<long long*>(bars + 4 * kMaxStages + 2 * kStagesW + 8 + kMaxEdges + 2);   // BC_K3_TRACE only

    {   // tables -> shared memory
        for (int i = tid; i < P.fan_floats; i += kThreads) s_fan[i] = i < P.fan_n ? P.fan[i] : 0.f;
        if (tid < 16) s_tab[tid] = make_float4(tid & 1 ? 1.f : 0.f, tid & 2 ? 1.f : 0.f, tid & 4 ? 1.f : 0.f, tid & 8 ? 1.f : 0.f);
    }
    if (tid == 0) {
        for (int s = 0; s < kMaxStages; ++s) {
            mbar_init(a_full0 + 8 * s, 4);
            mbar_init(a_empty0 + 8 * s, 1);
            mbar_init(b_full0 + 8 * s, 1);
            mbar_init(b_empty0 + 8 * s, 1);
        }
        for (int s = 0; s < kStagesW; ++s) {
            mbar_init(w_full0 + 8 * s, 1);
            mbar_init(w_empty0 + 8 * s, 4);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(d_full0 + 8 * b, 1);
            mbar_init(d_empty0 + 8 * b, 8);      // both epilogue groups
            mbar_init(bits_free0 + 8 * b, 8);
        }
        for (int e = 0; e < P.n_edges; ++e) mbar_init(lam_ready0 + 8 * e, 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot, 0);   // warp-uniform for the compiler: tcgen05 operands live in uniform registers

    if (warp == kWarpTma) {
        // ================= TMA warp: keeps the B ring (and the DENSE weight ring) full; the step sequence is static
        if (lane == 0) {
            Ring rb, rw;
            for (uint32_t iter = 0;; ++iter) {
                K3_PASS_HEAD
                for (int si = 0; si < P.n_seq; ++si) {
                    K3_STEP_HEAD
                    const K3Edge& E = P.edge[e];
                    const unsigned bytes = (unsigned)E.n_pad * 256u;   // hi + lo, 128 B per row each
                    for (int kb = 0; kb < E.nkb; ++kb) {
                        if (FMT == BC_DESC_DENSE_F32) {
                            mbar_wait(w_empty0 + 8 * rw.s, rw.par ^ 1u);
                            mbar_expect_tx(w_full0 + 8 * rw.s, kWBytes);
                            tma_load_2d(w_ring + rw.s * kWBytes, &tm_w, E.lam_off + kb * kBK, (int)(tile * kTile), w_full0 + 8 * rw.s);
                            rw.next(P.w_stages);
                        }
                        mbar_wait(b_empty0 + 8 * rb.s, rb.par ^ 1u);
                        mbar_expect_tx(b_full0 + 8 * rb.s, bytes);
                        tma_bulk_g2s(b_ring + rb.s * P.b_slot_bytes, P.bimg + E.bimg_off + (size_t)kb * bytes, bytes, b_full0 + 8 * rb.s);
                        rb.next(P.b_stages);
                    }
                }
                if (!cur_ok) break;
            }
        }
    } else if (warp == kWarpMma) {
        // ================= MMA issuer warp: the whole warp runs the (uniform) loop, one elected lane issues.  (The issue
        // queue is deep and neither the commits nor the fence stall it -- tools/microbench/umma_issue.cu -- but this warp
        // shares its scheduler with three busy warps: every instruction of this loop costs the tensor pipe time.)
        Ring ra, rb;
        uint32_t ed = 0;   // step counter (D buffer = ed % n_dbuf)
        const uint32_t SA = (uint32_t)P.a_stages, SB = (uint32_t)P.b_stages, b_slot = (uint32_t)P.b_slot_bytes;
        const uint32_t desc_hi = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);   // SBO (8 rows of 128 B), version 1, 128-byte swizzle
        const uint32_t a_base = tmem + (uint32_t)P.a_col, b_base = (((b_ring & 0x3FFFFu) >> 4) | (1u << 16));
        for (uint32_t iter = 0;; ++iter) {
            K3_PASS_HEAD
            for (int si = 0; si < P.n_seq; ++si) {
                K3_STEP_HEAD
                const K3Edge& E = P.edge[e];
                const bool a_exact = FMT == BC_DESC_BITS && E.col_v < 0 && !(E.fan_off >= 0 && P.fan_mask != nullptr);
                const uint32_t db = P.n_dbuf == 2 ? (ed & 1u) : 0u, dpar = (P.n_dbuf == 2 ? (ed >> 1) : ed) & 1u;
                ++ed;   // (executed steps only)
                const uint32_t d = tmem + (uint32_t)(P.d_col + (int)db * P.d_stride);
                const uint32_t idesc = E.idesc, b_lo_off = (uint32_t)E.n_pad * 8u;   // n_pad * 128 B in 16-byte units
                const int K = E.K, nkb = E.nkb;
                mbar_wait(d_empty0 + 8 * db, dpar ^ 1u);   // the epilogue of the edge that used this accumulator is done
                K3_STAMP(0, e, 0);
                for (int kb = 0; kb < nkb; ++kb) {
                    const uint32_t a_hi = a_base + ra.s * 64u, a_lo = a_hi + 32u;
                    // low word of the B descriptors: start address >> 4 | LBO = 1
                    const uint32_t b_hi = b_base + ((rb.s * b_slot) >> 4), b_lo = b_hi + b_lo_off;
                    const int ks = min(4, (K - kb * kBK + 7) >> 3);   // k-steps of 8 states with anything in them
                    mbar_wait(b_full0 + 8 * rb.s, rb.par);
                    mbar_wait(a_full0 + 8 * ra.s, ra.par);
                    tc_fence_after();
                    // error-compensated product, the small terms first; a k-step is 8 TF32: 8 columns of A, 32 bytes (+2) of B
                    if (!a_exact) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (k < ks) {
                                umma_tf32_ts(d, a_lo + 8u * k, b_hi + 2u * k, desc_hi, idesc, kb != 0 || k != 0);
                                umma_tf32_ts(d, a_hi + 8u * k, b_lo + 2u * k, desc_hi, idesc, 1);
                            }
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (k < ks) umma_tf32_ts(d, a_hi + 8u * k, b_lo + 2u * k, desc_hi, idesc, kb != 0 || k != 0);
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k < ks) umma_tf32_ts(d, a_hi + 8u * k, b_hi + 2u * k, desc_hi, idesc, 1);
                    umma_commit(a_empty0 + 8 * ra.s);
                    umma_commit(b_empty0 + 8 * rb.s);
                    if (kb == nkb - 1) umma_commit(d_full0 + 8 * db);
                    ra.next(SA);
                    rb.next(SB);
                }
                K3_STAMP(0, e, 1);
            }
            if (!cur_ok) break;
        }
    } else if (warp < kWarpEpi) {
        // ================= producer warps: thread = query = TMEM lane; group g builds the blocks with (step & 1) == g
        const int g = warp >> 2, ql = tid & (kTile - 1);
        const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        const uint32_t sw = (uint32_t)ql & 7u;    // 128-byte swizzle: chunk j of row r lives at r * 128 + ((j ^ (r & 7)) << 4)
        Ring ra, rw;
        uint32_t it = 0;
        // A tile's BITS rows and fan-out mask words come from global memory, in front of the pass with their latency exposed (every
        // producer warp waits on the barrier behind them).  The mask word is fetched ONE PASS AHEAD into a register and only written
        // to shared memory at the start of its own pass.
        constexpr int kPre = 2;   // uint4 per thread kept in registers
        // Measured on one box (tools/runs/_r2_run54.sh): the mask word ahead is +2.7 % on DENSE + fan-out rows; the BITS rows ahead
        // (8 more live registers in the producers, at the 96-register cap) are -3 % -- so only the mask word travels ahead.
        const bool pre_ok = P.prefetch && FMT != BC_DESC_BITS && P.mask_words <= 1;
        uint4 nb[kPre];
        uint32_t nfm = 0;
#pragma unroll
        for (int i = 0; i < kPre; ++i) nb[i] = make_uint4(0u, 0u, 0u, 0u);
        auto fetch = [&](long long tile_f) {   // global -> registers
            const size_t q = (size_t)tile_f * kTile + ql;
            const size_t qc = q < P.nq ? q : P.nq - 1;
            if (FMT == BC_DESC_BITS) {
                const uint32_t* grow = reinterpret_cast<const uint32_t*>(P.desc + qc * P.dstride);
#pragma unroll
                for (int i = 0; i < kPre; ++i) {
                    const int w4 = 4 * g + 4 * kGroups * i;
                    if (w4 < P.bits_words) nb[i] = __ldg(reinterpret_cast<const uint4*>(grow + w4));
                }
            }
            if (P.fan_mask != nullptr && g == 0) nfm = __ldg(P.fan_mask + qc * (size_t)P.mask_words);
        };
        for (uint32_t iter = 0;; ++iter) {
            K3_PASS_HEAD
            if (cur_ok) {
                // ---- this pass's tile: BITS rows and fan-out mask words -> shared memory (the two groups share the work)
                const size_t q = (size_t)tile_cur * kTile + ql;
                const size_t qc = q < P.nq ? q : P.nq - 1;
                const uint32_t buf = iter & 1u;
                uint32_t* bits_t = s_bits + buf * bits_tile;
                uint32_t* fm_t = s_fm + buf * fm_tile;
                if (pre_ok && iter == 0) fetch(tile_cur);
                if (iter >= 2) mbar_wait(bits_free0 + 8 * buf, ((iter >> 1) - 1u) & 1u);   // the epilogue warps are done with the tile that used this buffer
                if (pre_ok) {
                    if (FMT == BC_DESC_BITS) {
#pragma unroll
                        for (int i = 0; i < kPre; ++i) {
                            const int w4 = 4 * g + 4 * kGroups * i;
                            if (w4 < P.bits_words) {
                                bits_t[(w4 + 0) * kTile + ql] = nb[i].x;
                                bits_t[(w4 + 1) * kTile + ql] = nb[i].y;
                                bits_t[(w4 + 2) * kTile + ql] = nb[i].z;
                                bits_t[(w4 + 3) * kTile + ql] = nb[i].w;
                            }
                        }
                    }
                    if (P.fan_mask != nullptr && g == 0) fm_t[ql] = nfm;
                    if (tile_cur + (long long)gridDim.x < P.n_tiles) fetch(tile_cur + (long long)gridDim.x);   // the next pass's tile
                } else {
                    if (FMT == BC_DESC_BITS) {
                        const uint32_t* grow = reinterpret_cast<const uint32_t*>(P.desc + qc * P.dstride);
                        for (int w4 = 4 * g; w4 < P.bits_words; w4 += 4 * kGroups) {   // bits_words is a multiple of 4
                            const uint4 x = __ldg(reinterpret_cast<const uint4*>(grow + w4));
                            bits_t[(w4 + 0) * kTile + ql] = x.x;
                            bits_t[(w4 + 1) * kTile + ql] = x.y;
                            bits_t[(w4 + 2) * kTile + ql] = x.z;
                            bits_t[(w4 + 3) * kTile + ql] = x.w;
                        }
                    }
                    if (P.fan_mask != nullptr && g == 0)
                        for (int w = 0; w < P.mask_words; ++w) fm_t[w * kTile + ql] = __ldg(P.fan_mask + qc * (size_t)P.mask_words + w);
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(32 * kWarpEpi) : "memory");   // the eight producer warps
            int step_in_tile = 0;
            for (int si = 0; si < P.n_seq; ++si) {
                K3_STEP_HEAD
                const K3Edge& E = P.edge[e];
                const uint32_t* my_bits = s_bits + (tile_iter & 1u) * bits_tile + ql;
                const uint32_t* fm_t = s_fm + (tile_iter & 1u) * fm_tile;
                const bool leaf = E.col_v < 0;
                const bool a_exact = FMT == BC_DESC_BITS && leaf && !(E.fan_off >= 0 && P.fan_mask != nullptr);
                const bool fan_on = E.fan_off >= 0 && P.fan_mask != nullptr && ((fm_t[(E.v >> 5) * kTile + ql] >> (E.v & 31)) & 1u);
                const int K = E.K, nkb = E.nkb;
                if ((warp & 3) == 0) K3_STAMP(1 + g, e, 0);
                if (!leaf) {   // every message into Lambda_v has been multiplied in
                    mbar_wait(lam_ready0 + 8 * e, tile_iter & 1u);
                    tc_fence_after();
                }
                for (int kb = 0; kb < nkb; ++kb, ++it, ++step_in_tile, ra.next(P.a_stages), rw.next(P.w_stages)) {
                    if ((it % (uint32_t)kGroups) != (uint32_t)g) {
                        // Parity waits only tell ADJACENT phases apart: a group that writes a slot every other time it comes round
                        // (slots not a multiple of the groups) must still see every phase of the slot's barrier, or its own wait
                        // two phases later passes on the stale parity and it overwrites an operand the MMAs have not read yet.
                        if (P.a_stages % kGroups != 0) mbar_wait(a_empty0 + 8 * ra.s, ra.par ^ 1u);
                        continue;
                    }
                    const int c0 = kb * kBK;
                    if ((warp & 3) == 0) K3_STEP(0);
                    float u[kBK], lv[kBK];
                    if (!leaf) {   // Lambda_v first: the TMEM round trip (~250 clk under load) hides behind the wait for the weights
#pragma unroll
                        for (int c = 0; c < 4; ++c)   // (the node's columns are allocated in units of 8: never read past them)
                            if (c0 + 8 * c < K) tmem_ld8(tlane + (uint32_t)(E.col_v + c0 + 8 * c), lv + 8 * c);
                    }
                    if (FMT == BC_DESC_BITS) {
                        const uint32_t m = bits32(my_bits, P.bits_words, E.bit_off, K, c0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 t = s_tab[(m >> (4 * j)) & 15u];
                            u[4 * j] = t.x; u[4 * j + 1] = t.y; u[4 * j + 2] = t.z; u[4 * j + 3] = t.w;
                        }
                    } else {
                        mbar_wait(w_full0 + 8 * rw.s, rw.par);
                        const uint8_t* row = w_ring_ptr + rw.s * kWBytes + ql * 128;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 t = *reinterpret_cast<const float4*>(row + (((uint32_t)j ^ sw) << 4));
                            u[4 * j] = t.x; u[4 * j + 1] = t.y; u[4 * j + 2] = t.z; u[4 * j + 3] = t.w;
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive(w_empty0 + 8 * rw.s);   // the slot may be refilled
                    }
                    if (fan_on) {
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            if (c0 + 4 * j < K) {
                                const float4 f = *reinterpret_cast<const float4*>(s_fan + E.fan_off + c0 + 4 * j);
                                u[4 * j] *= f.x; u[4 * j + 1] *= f.y; u[4 * j + 2] *= f.z; u[4 * j + 3] *= f.w;
                            }
                    }
                    if ((warp & 3) == 0) K3_STEP(1);
                    if (!leaf) {
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < kBK; ++j)
                            if (c0 + (j & ~7) < K) u[j] *= lv[j];
                    }
                    // States >= K of the last block: their rows of T_v^T are zeros in the operand image and whole k-steps past K are not
                    // issued, so any FINITE value there contributes 0 -- BITS rows (bits past the domain are cleared, the message's
                    // padding columns hold the zeros the epilogue wrote) need no masking at all.  In a DENSE row the floats past the
                    // domain are the column's own pad floats, then the NEXT columns' weights AND pad floats, all of them up to the end
                    // of the last issued 8-state k-step: the pad floats are caller-owned (could be NaN / Inf, and NaN * 0 is NaN), so
                    // states K .. round_up(K, 8) - 1 are zeroed.  Past that k-step nothing is read; past the row TMA fills zeros.
                    // (The first version's compare + select over all 32 states was 7.5 % of the instructions of this issue-bound
                    // kernel: ncu, profiles/r2_ncu_36_k3_bits_imdb1.json.)
                    if (FMT == BC_DESC_DENSE_F32 && (K & 7) != 0 && c0 + kBK > K) {
                        // one 8-state group, picked by a uniform switch
                        const int r = K - c0;   // first state past the domain
#define K3_MASK_GROUP(G)                                              \
    case G:                                                           \
        _Pragma("unroll") for (int j = 8 * G + 1; j < 8 * G + 8; ++j) \
            if (j >= r) u[j] = 0.f;                                   \
        break;
                        switch (r >> 3) {
                            K3_MASK_GROUP(0) K3_MASK_GROUP(1) K3_MASK_GROUP(2) K3_MASK_GROUP(3)
                            default: break;
                        }
#undef K3_MASK_GROUP
                    }
                    const uint32_t a_hi = tlane + (uint32_t)(P.a_col + (int)ra.s * 64);
                    if ((warp & 3) == 0) K3_STEP(2);
                    if (a_exact) {
                        // unit weights on a leaf: U is a 0/1 matrix, exact in TF32 -- no lo half
                        mbar_wait(a_empty0 + 8 * ra.s, ra.par ^ 1u);   // the MMAs that read this slot are done
                        if ((warp & 3) == 0) K3_STEP(3);
                        tc_fence_after();
                        tmem_st32(a_hi, u);
                    } else {
                        float l[kBK];
#pragma unroll
                        for (int j = 0; j < kBK; ++j) {
                            float h;
                            split_tf32(u[j], h, l[j]);
                            u[j] = h;
                        }
                        mbar_wait(a_empty0 + 8 * ra.s, ra.par ^ 1u);
                        if ((warp & 3) == 0) K3_STEP(3);
                        tc_fence_after();
                        tmem_st32(a_hi, u);
                        tmem_st32(a_hi + 32u, l);
                    }
                    tmem_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(a_full0 + 8 * ra.s);
                    if ((warp & 3) == 0) K3_STEP(4);
                }
                if ((warp & 3) == 0) K3_STAMP(1 + g, e, 1);
            }
            if (!cur_ok) break;
        }
    } else {
        // ================= epilogue warps, two groups of four (warps 8-11: the lower half of the parent's columns, warps 14-17: the
        // upper half).  Over a RUN of consecutive edges into the same parent the message Lambda_pa stays in REGISTERS: per edge
        // only D is read from tensor memory (TMEM reads run at ~190 B/clk/SM, a quarter of the write rate -- reading D and
        // Lambda_pa and writing Lambda_pa back cost 1 250 clk per N = 84 edge and paced the leaves); the accumulator buffer is
        // handed back to the MMA warp as soon as it has been read; at the end of a run the message goes to tensor memory for the
        // producers of pa's own edge -- or, for the root, straight into the tile's result.
        const int g = warp >= kWarpEpiB;
        const int ql = tid & (kTile - 1);
        const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t ed = 0;
        float acc[kAcc];
#pragma unroll
        for (int i = 0; i < kAcc; ++i) acc[i] = 0.f;
        // SCALED (results beyond the fp32 range, reference arithmetic: fp64, ExactInference.py:157-177): after every update the
        // message is renormalised to a row maximum in [1, 2) -- an exact power-of-two scale, agreed between the two epilogue
        // groups through shared memory -- and the exponent is added to the tile's exponent (this tile's, or the previous tile's for
        // a tail edge); the result leaves as mantissa and exponent.
        int ex_cur = 0, ex_prev = 0;
        uint32_t xc = 0;   // exchanges so far (parity = buffer)
        auto scale_of = [&](float m_local, bool both, int& e_out) -> float {   // 2^-e, e = exponent of the row maximum
            float M = m_local;
            if (both) {
                float* mine = s_max + ((xc & 1u) * 2u + (uint32_t)g) * kTile;
                float* theirs = s_max + ((xc & 1u) * 2u + (uint32_t)(g ^ 1)) * kTile;
                mine[ql] = m_local;
                asm volatile("bar.sync 2, 256;" ::: "memory");
                M = fmaxf(M, theirs[ql]);
                ++xc;
            }
            const int eb = (int)((__float_as_uint(M) >> 23) & 0xFFu);
            int e_ = (eb == 0 || eb == 0xFF) ? 0 : eb - 127;   // zero / subnormal / non-finite rows are left alone
            if (e_ > 126) e_ = 126;
            e_out = e_;
            return __uint_as_float((uint32_t)(127 - e_) << 23);
        };
        for (uint32_t iter = 0;; ++iter) {
            K3_PASS_HEAD
            if (SCALED) { ex_prev = ex_cur; ex_cur = 0; }
            for (int si = 0; si < P.n_seq; ++si) {
                K3_STEP_HEAD
                const K3Edge& E = P.edge[e];
                const uint32_t db = P.n_dbuf == 2 ? (ed & 1u) : 0u, dpar = (P.n_dbuf == 2 ? (ed >> 1) : ed) & 1u;
                ++ed;   // (executed steps only)
                int& ex = back ? ex_prev : ex_cur;
                const uint32_t dcol = tlane + (uint32_t)(P.d_col + (int)db * P.d_stride), pcol = tlane + (uint32_t)E.col_pa;
                const bool first = E.first, run_first = (E.flags & kRunFirst) != 0, run_last = (E.flags & kRunLast) != 0;
                const bool regs = (E.flags & kRegs) != 0, root = E.publish == -2;
                // this group's columns [lo, hi) of the parent's n8 (both multiples of 8; the split is a function of card(pa) only)
                const int n8 = (E.N + 7) & ~7, half = ((n8 >> 1) + 15) & ~15, mid = half < n8 ? half : n8;
                const int lo = g ? mid : 0, hi = g ? n8 : mid;
                // optional correction of the truncating accumulator (off by default, see DESIGN.md)
                const bool a_exact = FMT == BC_DESC_BITS && E.col_v < 0 && !(E.fan_off >= 0 && P.fan_mask != nullptr);
                const int n_mma = ((int)E.K + 7) / 8 * (a_exact ? 2 : 3);
                const float debias = 1.f + (float)(n_mma - 1) * P.debias_unit;
                mbar_wait(d_full0 + 8 * db, dpar);
                tc_fence_after();
                if (warp == kWarpEpi) K3_STAMP(3, e, 0);
                if (regs) {
                    if (run_first) {   // acc = D (first message into pa) or acc = Lambda_pa (an earlier run's product, from tensor memory)
                        const uint32_t src = first ? dcol : pcol;
#pragma unroll
                        for (int r = 0; r < kAcc / 16; ++r) {
                            const int j = lo + 16 * r;
                            if (j + 16 <= hi) tmem_ld16(src + (uint32_t)j, acc + 16 * r);
                            else if (j < hi) tmem_ld8(src + (uint32_t)j, acc + 16 * r);
                        }
                        if (first) {
                            tmem_ld_wait();
                            if (P.debias_unit != 0.f) {
#pragma unroll
                                for (int i = 0; i < kAcc; ++i) acc[i] *= debias;
                            }
                        }
                    }
                    if (!(run_first && first)) {   // a TMEM read round trip costs ~150 clk under load whatever its size: 24 columns per wait
#pragma unroll
                        for (int r = 0; r < kAcc / 24; ++r) {
                            const int j = lo + 24 * r;
                            if (j < hi) {
                                float dv[24];
#pragma unroll
                                for (int c = 0; c < 3; ++c) {
                                    if (j + 8 * c < hi) tmem_ld8(dcol + (uint32_t)(j + 8 * c), dv + 8 * c);
                                    else {
#pragma unroll
                                        for (int i = 0; i < 8; ++i) dv[8 * c + i] = 1.f;
                                    }
                                }
                                tmem_ld_wait();
                                if (P.debias_unit != 0.f) {
#pragma unroll
                                    for (int i = 0; i < 24; ++i) dv[i] *= debias;
                                }
#pragma unroll
                                for (int i = 0; i < 24; ++i) acc[24 * r + i] *= dv[i];
                            }
                        }
                    }
                    if (SCALED) {
                        float mloc = 0.f;
#pragma unroll
                        for (int r = 0; r < kAcc / 8; ++r)
                            if (lo + 8 * r < hi) {
#pragma unroll
                                for (int i = 0; i < 8; ++i) mloc = fmaxf(mloc, acc[8 * r + i]);
                            }
                        int e_;
                        const float sc = scale_of(mloc, mid < n8, e_);
                        if (e_ != 0) {
#pragma unroll
                            for (int i = 0; i < kAcc; ++i) acc[i] *= sc;
                        }
                        ex += e_;
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(d_empty0 + 8 * db);   // the accumulator has been read: the MMAs of the edge after next may start
                    if (run_last && !root) {   // the message goes to tensor memory
#pragma unroll
                        for (int r = 0; r < kAcc / 16; ++r) {
                            const int j = lo + 16 * r;
                            if (j + 16 <= hi) tmem_st16(pcol + (uint32_t)j, acc + 16 * r);
                            else if (j < hi) tmem_st8(pcol + (uint32_t)j, acc + 16 * r);
                        }
                        tmem_st_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0 && E.publish >= 0) mbar_arrive(lam_ready0 + 8 * E.publish);   // Lambda_pa is complete: pa's own edge may be built
                    }
                } else {
                    // Lambda_pa (*)= D in tensor memory without touching the register accumulator: a parent domain beyond 2 x kAcc
                    // states, or a TAIL edge (the only message into its parent, interleaved with another tile's run).  The root's
                    // only message is not copied at all: the result is read off the accumulator below.
                    if (!(first && root)) {
                        for (int j = lo; j < hi; j += 16) {
                            float dv[16];
                            tmem_ld8(dcol + (uint32_t)j, dv);
                            if (j + 8 < hi) tmem_ld8(dcol + (uint32_t)(j + 8), dv + 8);
                            tmem_ld_wait();
                            if (!first) {
#pragma unroll
                                for (int h8 = 0; h8 < 2; ++h8)
                                    if (j + 8 * h8 < hi) {
                                        float lv[8];
                                        tmem_ld8(pcol + (uint32_t)(j + 8 * h8), lv);
                                        tmem_ld_wait();
#pragma unroll
                                        for (int i = 0; i < 8; ++i) dv[8 * h8 + i] *= lv[i];
                                    }
                            }
                            if (P.debias_unit != 0.f) {
#pragma unroll
                                for (int i = 0; i < 16; ++i) dv[i] *= debias;
                            }
                            tmem_st8(pcol + (uint32_t)j, dv);
                            if (j + 8 < hi) tmem_st8(pcol + (uint32_t)(j + 8), dv + 8);
                        }
                        tmem_st_wait();
                        if (SCALED) {   // second and third pass over the message's own columns: maximum, then the scale
                            float mloc = 0.f;
                            for (int j = lo; j < hi; j += 8) {
                                float lv[8];
                                tmem_ld8(pcol + (uint32_t)j, lv);
                                tmem_ld_wait();
#pragma unroll
                                for (int i = 0; i < 8; ++i) mloc = fmaxf(mloc, lv[i]);
                            }
                            int e_;
                            const float sc = scale_of(mloc, mid < n8, e_);
                            // (every thread has its own exponent; the tcgen05 loads and stores are warp-wide instructions, so the
                            //  pass is unconditional: a thread with nothing to scale multiplies by 1)
                            for (int j = lo; j < hi; j += 8) {
                                float lv[8];
                                tmem_ld8(pcol + (uint32_t)j, lv);
                                tmem_ld_wait();
#pragma unroll
                                for (int i = 0; i < 8; ++i) lv[i] *= sc;
                                tmem_st8(pcol + (uint32_t)j, lv);
                            }
                            tmem_st_wait();
                            ex += e_;
                        }
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            mbar_arrive(d_empty0 + 8 * db);
                            if (E.publish >= 0) mbar_arrive(lam_ready0 + 8 * E.publish);
                        }
                    }
                }
                if (warp == kWarpEpi) K3_STAMP(3, e, 1);
                if (root) {
                    // ---- the tile's result: sum_c w_0[c] * Lambda_0[c] * T_0[c], each group over its own columns
                    const size_t q = (size_t)tile * kTile + ql;
                    const size_t qc = q < P.nq ? q : P.nq - 1;
                    const uint32_t buf = tile_iter & 1u;
                    const uint32_t* my_bits = s_bits + buf * bits_tile + ql;
                    const float* drow = reinterpret_cast<const float*>(P.desc + qc * P.dstride);
                    const bool fan_root = P.root_fan_off >= 0 && P.fan_mask != nullptr && (s_fm[buf * fm_tile + ql] & 1u);
                    float res = 0.f;
                    if (regs) {
#pragma unroll
                        for (int r = 0; r < kAcc / 8; ++r) {
                            const int c0 = lo + 8 * r;
                            if (c0 < hi && c0 < P.root_card) {
                                float w[8];
                                weights8<FMT>(my_bits, P.bits_words, drow, P.root_lam_off, P.root_bit_off, P.root_card, c0, w);
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    if (c0 + j < P.root_card) {
                                        float x = acc[8 * r + j] * w[j];
                                        if (fan_root) x *= s_fan[P.root_fan_off + c0 + j];
                                        res = fmaf(x, __ldg(P.root_T + c0 + j), res);
                                    }
                            }
                        }
                    } else {
                        // from tensor memory: the root's columns, or straight from the accumulator when this edge is the root's only message
                        const uint32_t src = first ? dcol : tlane + (uint32_t)P.root_col;
                        for (int c0 = lo; c0 < hi && c0 < P.root_card; c0 += 8) {
                            float lv[8], w[8];
                            tmem_ld8(src + (uint32_t)c0, lv);
                            weights8<FMT>(my_bits, P.bits_words, drow, P.root_lam_off, P.root_bit_off, P.root_card, c0, w);
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 8; ++j)
                                if (c0 + j < P.root_card) {
                                    float x = lv[j] * w[j] * (first ? debias : 1.f);
                                    if (fan_root) x *= s_fan[P.root_fan_off + c0 + j];
                                    res = fmaf(x, __ldg(P.root_T + c0 + j), res);
                                }
                        }
                        if (first) {   // the accumulator has been read
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(d_empty0 + 8 * db);
                        }
                    }
                    if (mid < n8) {   // the upper half's share travels through shared memory (two tiles deep: the groups drift by at most one)
                        if (g) s_part[buf * kTile + ql] = res;
                        asm volatile("bar.sync 2, 256;" ::: "memory");
                        if (!g) res += s_part[buf * kTile + ql];
                    }
                    if (!g && q < P.nq) {
                        P.out[q] = res;
                        if (SCALED) P.out_exp[q] = ex;
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bits_free0 + 8 * buf);   // this tile's BITS rows / mask words are no longer read
                }
            }
            if (!cur_ok) break;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
    }
    if (BC_K3_TRACE_BUILD && P.trace != nullptr && blockIdx.x == 0)
        for (int i = tid; i < kTraceSteps * 8; i += kThreads) P.trace[kCnt + i] = s_trace[i];
}

uint32_t host_tf32_hi(float x) {
    uint32_t b;
    std::memcpy(&b, &x, 4);
    return (b + 0x1000u) & 0xFFFFE000u;
}

int k3_prepare(bc_model* m) {
    if (m->k3) {
        if (m->k3->failed) bc_set_error("fused tensor-core kernel (K3) does not serve this model");
        return m->k3->failed ? BC_ELIMIT : BC_OK;
    }
    // the plan is built locally and published to m->k3 only when it is complete: a structural "does not serve" verdict is
    // published (failed = 1, so it is not recomputed); a CUDA error while uploading the operand image publishes nothing, so
    // that the next call retries instead of launching with a NULL image
    std::unique_ptr<BcK3Plan> plan(new BcK3Plan());
    BcK3Plan* k = plan.get();
    auto fail = [&](const char* why) {
        k->failed = 1;
        m->k3 = plan.release();
        bc_set_error("fused tensor-core kernel (K3) does not serve this model: %s", why);
        return BC_ELIMIT;
    };
    const int n = m->n;
    if (n < 2) return fail("single-node model");
    if (n - 1 > kMaxEdges) return fail("more than 128 columns (the edge table travels in the kernel parameter bank)");
    if (m->arena.empty()) return fail("no host copy of the CPT arena");
    // ---- edge schedule: depth-first post order (children before parents, a node's edge right after its last child's),
    //      heaviest subtree first: a Lambda then only lives while its own subtree is being folded, so the live set is
    //      bounded by the depth of the tree instead of its width (the reverse topological order kept 5+ messages of a
    //      20-column synthetic tree alive at once and did not fit tensor memory)
    std::vector<std::vector<int>> kids(n);
    std::vector<long long> weight(n, 0);
    for (int v = n - 1; v >= 1; --v) {
        weight[v] += (long long)m->nodes[v].card * m->nodes[v].card_pa;
        weight[m->nodes[v].parent] += weight[v];
        kids[m->nodes[v].parent].push_back(v);
    }
    std::vector<int> sched;   // sched[e] = child node of edge e
    {
        std::vector<std::pair<int, size_t>> stack{{0, 0}};
        // siblings: internal subtrees first, heaviest first (their messages leave tensor memory early); then the LEAVES in
        // ascending domain size -- the epilogue of an edge costs card(pa) columns whatever card(v) is, so small leaves at the
        // end would queue their epilogues up right where the parent's own edge is waiting for them
        for (int v = 0; v < n; ++v)
            std::stable_sort(kids[v].begin(), kids[v].end(), [&](int a, int b) {
                const bool ia = !kids[a].empty(), ib = !kids[b].empty();
                if (ia != ib) return ia;
                return ia ? weight[a] > weight[b] : m->nodes[a].card < m->nodes[b].card;
            });
        while (!stack.empty()) {
            auto& [v, i] = stack.back();
            if (i < kids[v].size()) {
                const int c = kids[v][i++];
                stack.push_back({c, 0});
            } else {
                if (v != 0) sched.push_back(v);
                stack.pop_back();
            }
        }
    }
    const int n_edges = (int)sched.size();
    std::vector<int> first_child_edge(n, -1), own_edge(n, -1);
    for (int e = 0; e < n_edges; ++e) {
        const int v = sched[e];
        own_edge[v] = e;
        const int pa = m->nodes[v].parent;
        if (first_child_edge[pa] < 0) first_child_edge[pa] = e;
    }
    int npad_max = 16;
    for (int v : sched) {
        const int np = (int)bc_round_up(m->nodes[v].card_pa, 16);
        if (np > 256) return fail("a parent domain exceeds 256 states");
        if (np > npad_max) npad_max = np;
    }
    // ---- TMEM columns (one CTA per SM owns all 512): [A ring: a_stages x 64][accumulators: n_dbuf x npad_max][Lambda of
    //      every internal node by first fit over lifetimes [edge of its first child, its own edge] (the root lives to the
    //      end), in units of 8 columns].  Lifetimes may be reused back to back although the roles run at different places
    //      of the step sequence: a node's columns are first WRITTEN by the epilogue of its first child's edge, which follows
    //      that edge's MMAs, which follow every block the producers built before -- including all READS of the previous
    //      occupant during its own edge.  Two accumulator buffers let the MMAs of the next edge run under this edge's epilogue.
    std::vector<int> col(n, -1);
    std::vector<int> order;   // internal nodes by start of lifetime
    for (int v = 0; v < n; ++v)
        if (first_child_edge[v] >= 0) order.push_back(v);
    std::sort(order.begin(), order.end(), [&](int a, int b) { return first_child_edge[a] < first_child_edge[b]; });
    // Runs: maximal sequences of consecutive edges into the same parent; the epilogue warps keep the parent's message in
    // registers over a run (domains of up to 2 x kAcc states).  The ROOT's message then never visits tensor memory unless its
    // runs are interrupted (two internal children) or its domain is too large for the registers.
    auto pa_of = [&](int e) { return (int)m->nodes[sched[e]].parent; };
    std::vector<int> n_msgs(n, 0);
    for (int e = 0; e < n_edges; ++e) ++n_msgs[pa_of(e)];
    // TAIL: the chain at the top of the tree -- the maximal suffix of the schedule made of edges that are the ONLY message into
    // their parent.  Each of them waits for the complete result of the one before (drain, epilogue, producers, MMAs: ~2 500 clk
    // per hop with the tensor pipe idle: 35-40 % of a tile on the IMDB models).  They are taken out of the tile's own pass and
    // interleaved with the body of the CTA's NEXT tile; their epilogue never touches the register accumulator (the body's run
    // is alive in it), the nodes they read and write keep their tensor-memory columns for the whole pass.
    int n_tail = 0;
    if (!std::getenv("BC_K3_NO_SKEW"))
        while (n_tail < n_edges - 1 && n_msgs[pa_of(n_edges - 1 - n_tail)] == 1) ++n_tail;
    const int n_body = n_edges - n_tail;
    std::vector<char> pinned(n, 0);   // nodes whose columns live across passes
    for (int e = n_body; e < n_edges; ++e) pinned[sched[e]] = pinned[pa_of(e)] = 1;
    int root_runs = 0;
    for (int e = 0; e < n_edges; ++e)
        if (pa_of(e) == 0 && (e == 0 || pa_of(e - 1) != 0)) ++root_runs;
    const bool root_only_msg = n_msgs[0] == 1;   // read straight off the accumulator
    const bool root_in_regs = root_only_msg || (bc_round_up(m->nodes[0].card, 16) <= 2 * kAcc && root_runs == 1);
    auto assign = [&](int a_stages, int n_dbuf) -> int {   // columns used, or -1 (col[] is only written when every node found a place)
        std::vector<int> place(n, -1);
        const int units_total = 512 / 8;
        std::vector<int> busy_until(units_total, -1);   // last edge index that uses the unit
        const int fixed_units = (a_stages * 64 + n_dbuf * npad_max) / 8;
        if (fixed_units > units_total) return -1;
        for (int u = 0; u < fixed_units; ++u) busy_until[u] = 1 << 30;
        int units_used = fixed_units;
        for (int v : order) {
            if (v == 0 && root_in_regs) continue;
            const int need = (int)bc_round_up(m->nodes[v].card, 8) / 8;
            const int start = pinned[v] ? 0 : first_child_edge[v];
            const int end = (own_edge[v] < 0 || pinned[v]) ? (1 << 30) : own_edge[v];   // (the root: to the end)
            int at = -1;
            for (int u0 = 0; u0 + need <= units_total && at < 0; ++u0) {
                bool ok = true;
                for (int u = u0; u < u0 + need; ++u)
                    if (busy_until[u] >= start) { ok = false; break; }
                if (ok) at = u0;
            }
            if (at < 0) return -1;
            for (int u = at; u < at + need; ++u) busy_until[u] = end;
            place[v] = at * 8;
            if (at + need > units_used) units_used = at + need;
        }
        col = place;
        return units_used * 8;
    };
    // preference: a deep A ring and two accumulators; give up ring depth first, the second accumulator last
    static const int kTry[][2] = {{3, 2}, {2, 2}, {3, 1}, {2, 1}};
    int a_stages = 0, n_dbuf = 0;
    for (const auto& t : kTry)
        if (assign(t[0], t[1]) > 0) { a_stages = t[0]; n_dbuf = t[1]; break; }
    if (const char* e = std::getenv("BC_K3_PLAN")) {   // experiments: "<a_stages>,<n_dbuf>"
        int wa = 0, wd = 0;
        if (std::sscanf(e, "%d,%d", &wa, &wd) == 2 && wa >= 2 && wa <= kMaxStages && (wd == 1 || wd == 2) && assign(wa, wd) > 0) {
            a_stages = wa;
            n_dbuf = wd;
        } else if (a_stages) {
            assign(a_stages, n_dbuf);
        }
    }
    if (!a_stages) return fail("live messages exceed the 512 columns of tensor memory");
    k->tmem_cols = 512;
    k->npad_max = npad_max;
    k->a_col = 0;
    k->a_stages = a_stages;
    k->d_col = a_stages * 64;
    k->n_dbuf = n_dbuf;
    k->root_col = col[0];
    // ---- operand images: per edge and block of 32 child states, T_v^T hi then lo, 128-byte swizzled rows
    size_t total = 0;
    k->edges.resize(n_edges);
    std::vector<int> last_child_edge(n, -1);
    for (int e = 0; e < n_edges; ++e) last_child_edge[m->nodes[sched[e]].parent] = e;
    for (int e = 0; e < n_edges; ++e) {
        const int v = sched[e];
        const BcNodeRec& nd = m->nodes[v];
        K3Edge& E = k->edges[e];
        std::memset(&E, 0, sizeof(E));
        E.v = v;
        E.K = nd.card;
        E.N = nd.card_pa;
        E.n_pad = (int)bc_round_up(nd.card_pa, 16);
        E.lam_off = nd.lam_off;
        E.bit_off = m->bits[v].bit_off;
        E.fan_off = nd.fan_off;
        E.col_v = col[v];
        E.col_pa = col[nd.parent];
        E.first = first_child_edge[nd.parent] == e;
        E.nkb = (nd.card + kBK - 1) / kBK;
        E.idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(E.n_pad >> 3) << 17) | ((uint32_t)(kTile >> 4) << 24);
        E.publish = last_child_edge[nd.parent] != e ? -1 : (nd.parent == 0 ? -2 : own_edge[nd.parent]);
        E.flags = ((e == 0 || pa_of(e - 1) != nd.parent) ? kRunFirst : 0) | ((e == n_edges - 1 || pa_of(e + 1) != nd.parent) ? kRunLast : 0) |
                  ((E.n_pad <= 2 * kAcc && e < n_body) ? kRegs : 0);
        E.bimg_off = total;
        total += (size_t)E.nkb * E.n_pad * 256;
    }
    {   // step sequence of one pass: the body in order, the previous tile's tail edges spread over it by estimated tensor time
        // (one hop of the chain needs the result of the one before: leave ~2 500 clk of body work between them)
        auto cost = [&](const K3Edge& E) { return (long long)((E.K + 7) / 8) * 3 * std::max(E.n_pad / 2, 40); };
        long long cum = 0;
        int t = 0;
        long long gap = 2500;
        if (const char* e = std::getenv("BC_K3_GAP")) gap = std::max(1, std::atoi(e));
        // the first tail edge READS the message of the node below the chain while the body's runs into that node REWRITE it for
        // the next tile: it must come before the body edge that ends the first of those runs (then its producers have read
        // the old message before that edge's MMAs, hence before its epilogue's write)
        int limit0 = n_body;
        if (n_tail > 0) {
            const int hub = sched[n_body];
            // (register accumulators: the message is written at the end of a run; a wider parent is updated in tensor memory
            //  by every edge into it, so the tail edge must come before the first of them)
            for (int e = 0; e < n_body; ++e)
                if (pa_of(e) == hub && ((k->edges[e].flags & kRunLast) || !(k->edges[e].flags & kRegs))) { limit0 = e; break; }
        }
        for (int e = 0; e < n_body; ++e) {
            if (t == 0 && n_tail > 0 && e == limit0) k->seq.push_back((uint8_t)(128 | (n_body + t++)));
            k->seq.push_back((uint8_t)e);
            cum += cost(k->edges[e]);
            while (t < n_tail && cum >= gap / 2 + (long long)t * gap) k->seq.push_back((uint8_t)(128 | (n_body + t++)));
        }
        while (t < n_tail) k->seq.push_back((uint8_t)(128 | (n_body + t++)));
        k->n_tail = n_tail;
    }
    std::vector<uint8_t> img(total, 0);
    for (const K3Edge& E : k->edges) {
        const BcNodeRec& nd = m->nodes[E.v];
        const float* T = m->arena.data() + nd.cpt_off;
        for (int kb = 0; kb < E.nkb; ++kb) {
            uint8_t* hi = img.data() + E.bimg_off + (size_t)kb * E.n_pad * 256;
            uint8_t* lo = hi + (size_t)E.n_pad * 128;
            for (int p = 0; p < E.N; ++p)
                for (int kk = 0; kk < kBK; ++kk) {
                    const int c = kb * kBK + kk;
                    if (c >= E.K) continue;
                    const float x = T[(size_t)c * nd.stride + p];
                    const uint32_t hb = host_tf32_hi(x);
                    float h;
                    std::memcpy(&h, &hb, 4);
                    const float l = x - h;
                    const uint32_t lb = host_tf32_hi(l);
                    const size_t off = (size_t)p * 128 + ((size_t)((kk >> 2) ^ (p & 7)) << 4) + (size_t)(kk & 3) * 4;   // 128-byte swizzle
                    std::memcpy(hi + off, &hb, 4);
                    std::memcpy(lo + off, &lb, 4);
                }
        }
    }
    k->bimg_bytes = total;
    // ---- shared memory: B ring (as deep as fits, at most 4), DENSE weight ring, BITS rows and fan-out mask words of two tiles
    const size_t fan_floats = (size_t)bc_round_up((int64_t)m->fan.size(), 4);
    int w_stages = 4;
    if (const char* e = std::getenv("BC_K3_WSTAGES")) w_stages = std::max(2, std::min(kStagesW, std::atoi(e)));
    const size_t per_fmt = std::max((size_t)w_stages * kWBytes, (size_t)2 * m->bits_words * kTile * 4);
    const size_t fixed = per_fmt + (size_t)2 * m->mask_words * kTile * 4 + fan_floats * 4 + 256 /* nibble table */ + 2 * kTile * 4 /* root partial sums */ + 4 * kTile * 4 /* row maxima (scaled results) */ +
                         8 * (4 * kMaxStages + 2 * kStagesW + 8 + kMaxEdges + 2) /* barriers, TMEM slot */ + 8 * kTraceSteps * 8 /* trace */ +
                         1024 /* alignment */;
    const size_t smem_optin = m->device >= 0 ? (size_t)m->smem_optin : (size_t)227 * 1024;   // host-only model: the sm_100 value
    int b_stages = kMaxStages;
    if (const char* e = std::getenv("BC_K3_BSTAGES")) b_stages = std::max(2, std::min(kMaxStages, std::atoi(e)));
    while (b_stages > 1 && (size_t)b_stages * npad_max * 256 + fixed > smem_optin) --b_stages;
    if ((size_t)b_stages * npad_max * 256 + fixed > smem_optin || b_stages < 2) return fail("operand rings exceed shared memory");
    // (after the structural limits: a model that does not fit at all is declined for that reason)
    for (int v = 1; v < n; ++v)
        if (m->nodes[v].card > kMaxK)
            return fail("a non-root column of more than 128 states (one accumulator over its k-steps loses the 1e-5 accuracy)");
    k->b_stages = b_stages;
    k->w_stages = w_stages;
    k->smem = (size_t)b_stages * npad_max * 256 + fixed;
    k->ctas_per_sm = 1;
    if (m->device >= 0) {   // (a host-only model keeps the plan for inspection: bc_model_fused_plan)
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &k->encode, cudaEnableDefault, &qr) != cudaSuccess || !k->encode ||
            qr != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            return fail("the driver does not export cuTensorMapEncodeTiled");
        }
        BC_CUDA_CHECK(cudaMalloc(&k->d_bimg, total));
        const cudaError_t ce = cudaMemcpy(k->d_bimg, img.data(), total, cudaMemcpyHostToDevice);
        if (ce != cudaSuccess) {
            cudaFree(k->d_bimg);
            bc_set_error("upload of the K3 operand image failed: %s", cudaGetErrorString(ce));
            return BC_ECUDA;
        }
    }
    m->k3 = plan.release();
    return BC_OK;
}

template <int FMT, bool SCALED>
int k3_launch_fmt(bc_model* m, const K3Params& P, const CUtensorMap& tm_w, int grid, cudaStream_t st) {
    static bool attr_set[64] = {};
    int dev = 0;
    BC_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_set[dev]) {
        BC_CUDA_CHECK(cudaFuncSetAttribute(k3_kernel<FMT, SCALED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->smem_optin));
        if (dev >= 0 && dev < 64) attr_set[dev] = true;
    }
    k3_kernel<FMT, SCALED><<<grid, kThreads, m->k3->smem, st>>>(P, tm_w);
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch();
    return BC_OK;
}

}  // namespace

int bc_k3_launch(bc_model* m, const void* desc, size_t nq, int fmt, const uint32_t* fan_mask, float* out, cudaStream_t st, int32_t* out_exp) {
    if (nq == 0) return BC_OK;
    if (fmt != BC_DESC_BITS && fmt != BC_DESC_DENSE_F32) {
        bc_set_error("the fused kernel reads BITS or DENSE_F32 rows (convert range rows with bc_convert_desc)");
        return BC_EINVAL;
    }
    if (reinterpret_cast<uintptr_t>(desc) & 15u) {
        bc_set_error("descriptor rows are read with 16-byte loads: the buffer must be 16-byte aligned");
        return BC_EINVAL;
    }
    {
        std::lock_guard<std::mutex> g(m->k3_mu);
        int rc = k3_prepare(m);
        if (rc) return rc;
    }
    const BcK3Plan* k = m->k3;
    K3Params P{};
    P.n_edges = (int)k->edges.size();
    std::memcpy(P.edge, k->edges.data(), sizeof(K3Edge) * k->edges.size());
    P.n_seq = (int)k->seq.size();
    P.n_tail = k->n_tail;
    P.prefetch = std::getenv("BC_K3_NO_PREFETCH") ? 0 : 1;
    std::memcpy(P.seq, k->seq.data(), k->seq.size());
    P.bimg = k->d_bimg;
    P.desc = static_cast<const uint8_t*>(desc);
    P.dstride = (size_t)bc_model_desc_stride(m, fmt);
    P.fan_mask = fan_mask;
    P.fan = m->d_fan;
    P.fan_floats = (int)bc_round_up((int64_t)m->fan.size(), 4);
    P.fan_n = (int)m->fan.size();
    const BcNodeRec& r = m->nodes[0];
    P.root_T = m->d_arena + r.cpt_off;
    P.root_card = r.card;
    P.root_col = k->root_col;
    P.root_bit_off = m->bits[0].bit_off;
    P.root_lam_off = r.lam_off;
    P.root_fan_off = r.fan_off;
    P.out = out;
    P.out_exp = out_exp;
    P.nq = nq;
    P.n_tiles = (long long)((nq + kTile - 1) / kTile);
    P.bits_words = m->bits_words;
    P.b_slot_bytes = k->npad_max * 256;
    P.a_col = k->a_col;
    P.a_stages = k->a_stages;
    P.b_stages = k->b_stages;
    P.w_stages = k->w_stages;
    P.d_col = k->d_col;
    P.d_stride = k->npad_max;
    P.n_dbuf = k->n_dbuf;
    P.mask_words = m->mask_words;
    P.debias_unit = 0.f;
    if (const char* e = std::getenv("BC_K3_DEBIAS")) P.debias_unit = (float)std::atof(e);
    long long grid = (long long)m->sm_count * k->ctas_per_sm;
    if (grid > P.n_tiles) grid = P.n_tiles;
    struct TraceDump {   // BC_K3_TRACE=1 (debugging): synchronises and prints the clock stamps of one tile
        long long* d = nullptr;
        const BcK3Plan* k;
        int fmt;
        ~TraceDump() {
            if (!d) return;
            std::vector<long long> h(kCnt + kTraceSteps * 8);
            cudaDeviceSynchronize();
            cudaMemcpy(h.data(), d, h.size() * 8, cudaMemcpyDeviceToHost);
            cudaFree(d);
            const long long t0 = h[(1 * kMaxEdges + 0) * 2];
            std::fprintf(stderr, "K3 trace fmt %d (clk since the producers entered edge 0 of the tile; role: start..end)\n", fmt);
            for (size_t e = 0; e < k->edges.size(); ++e) {
                const K3Edge& E = k->edges[e];
                std::fprintf(stderr, "  e%zu K%d N%d %s:", e, E.K, E.N, E.col_v < 0 ? "leaf" : "int ");
                static const char* names[4] = {"mma", "prodA", "prodB", "epi"};
                for (int r = 0; r < 4; ++r)
                    std::fprintf(stderr, "  %s %lld..%lld", names[r], h[(r * kMaxEdges + e) * 2] - t0, h[(r * kMaxEdges + e) * 2 + 1] - t0);
                std::fprintf(stderr, "\n");
            }
            std::fprintf(stderr, "  step: producer start, +inputs, +Lambda, +slot free, +stored | mma: B full, A full, issued (clk, same origin)\n");
            int step = 0;
            for (size_t e = 0; e < k->edges.size(); ++e)
                for (int kb = 0; kb < k->edges[e].nkb && step < kTraceSteps; ++kb, ++step) {
                    const long long* c = h.data() + kCnt + step * 8;
                    std::fprintf(stderr, "  e%zu.%d g%d: %6lld +%4lld +%4lld +%4lld +%4lld | %6lld %6lld %6lld\n", e, kb, step & 1, c[0] - t0, c[1] - c[0],
                                 c[2] - c[1], c[3] - c[2], c[4] - c[3], c[5] - t0, c[6] - t0, c[7] - t0);
                }
        }
    } trace_dump;
    trace_dump.k = k;
    trace_dump.fmt = fmt;
    if (BC_K3_TRACE_BUILD && std::getenv("BC_K3_TRACE") && P.n_tiles > (long long)(kTraceTile + 1) * grid) {
        if (cudaMalloc(&trace_dump.d, (kCnt + kTraceSteps * 8) * 8) == cudaSuccess) cudaMemset(trace_dump.d, 0, (kCnt + kTraceSteps * 8) * 8);
        P.trace = trace_dump.d;
    }
    CUtensorMap tm_w;
    std::memset(&tm_w, 0, sizeof(tm_w));
    if (fmt == BC_DESC_DENSE_F32) {
        // DENSE_F32 rows as a 2-D tensor [nq rows x lam_total floats]; one box = 128 queries x 32 states, 128-byte swizzle (the
        // producers read their own row conflict free); rows past the batch and columns past the row read as zeros
        const cuuint64_t dims[2] = {(cuuint64_t)m->lam_total, (cuuint64_t)nq};
        const cuuint64_t strides[1] = {(cuuint64_t)m->lam_total * 4};
        const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kTile};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult cr = reinterpret_cast<EncodeTiledFn>(k->encode)(&tm_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(desc), dims, strides,
                                                                       box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) {
            bc_set_error("cuTensorMapEncodeTiled failed (%d) for %zu DENSE_F32 rows of %d floats", (int)cr, nq, m->lam_total);
            return BC_ECUDA;
        }
        return out_exp ? k3_launch_fmt<BC_DESC_DENSE_F32, true>(m, P, tm_w, (int)grid, st)
                       : k3_launch_fmt<BC_DESC_DENSE_F32, false>(m, P, tm_w, (int)grid, st);
    }
    return out_exp ? k3_launch_fmt<BC_DESC_BITS, true>(m, P, tm_w, (int)grid, st) : k3_launch_fmt<BC_DESC_BITS, false>(m, P, tm_w, (int)grid, st);
}

extern "C" int bc_model_fused_plan(bc_model* m, int32_t* info, int32_t* edges, size_t edges_capacity) {
    if (!m || !info) { bc_set_error("model/info is NULL"); return BC_EINVAL; }
    {
        std::lock_guard<std::mutex> g(m->k3_mu);
        int rc = k3_prepare(m);
        if (rc) return rc;
    }
    const BcK3Plan* k = m->k3;
    info[0] = (int32_t)k->edges.size();
    info[1] = k->tmem_cols;
    info[2] = k->ctas_per_sm;
    info[3] = (int32_t)k->smem;
    info[4] = k->d_col;
    info[5] = k->npad_max * k->n_dbuf;   // accumulator columns [d_col, d_col + this); the A ring is [0, d_col)
    info[6] = k->root_col;
    info[7] = (int32_t)(k->bimg_bytes >> 10);
    if (edges) {
        if (edges_capacity < k->edges.size()) { bc_set_error("edges buffer too small"); return BC_EINVAL; }
        for (size_t e = 0; e < k->edges.size(); ++e) {
            const K3Edge& E = k->edges[e];
            int32_t* o = edges + 8 * e;
            o[0] = E.v; o[1] = E.K; o[2] = E.N; o[3] = E.n_pad; o[4] = E.col_v; o[5] = E.col_pa; o[6] = E.first; o[7] = E.nkb;
        }
    }
    return BC_OK;
}

extern "C" int bc_model_fused_sequence(bc_model* m, uint8_t* sequence, uint8_t* flags, size_t capacity, int32_t* n_tail) {
    if (!m || !sequence || !flags || !n_tail) { bc_set_error("model/sequence/flags/n_tail is NULL"); return BC_EINVAL; }
    {
        std::lock_guard<std::mutex> g(m->k3_mu);
        int rc = k3_prepare(m);
        if (rc) return rc;
    }
    const BcK3Plan* k = m->k3;
    if (capacity < k->edges.size() || k->seq.size() != k->edges.size()) { bc_set_error("sequence buffer too small"); return BC_EINVAL; }
    for (size_t i = 0; i < k->edges.size(); ++i) {
        sequence[i] = k->seq[i];
        flags[i] = (uint8_t)k->edges[i].flags;
    }
    *n_tail = k->n_tail;
    return BC_OK;
}

void bc_k3_free(bc_model* m) {
    if (!m->k3) return;
    cudaFree(m->k3->d_bimg);
    delete m->k3;
    m->k3 = nullptr;
}
