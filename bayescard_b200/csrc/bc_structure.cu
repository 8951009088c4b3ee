// Structure learning: all-pairs co-occurrence counts of a discretised table on the tensor cores, pairwise mutual
// information, and the Chow-Liu tree (maximum spanning tree on mutual information, Prim on the host).
//
// Replaces pomegranate's BayesianNetwork.from_samples(algorithm='chow-liu', root=0) of the reference
// (Models/BN_single_model.py:141-202).  Chow-Liu needs the joint histogram of EVERY pair of columns.  With X the
// rows x S one-hot matrix of the table (S = sum of the cards, state s = (column, bin)), all of them together are the
// integer Gram matrix G = X^T X: G[s_a][s_b] counts the rows in which both states occur.  G is an int8 GEMM with s32
// accumulation (tcgen05.mma ... kind::i8, SASS UTCIMMA), exact as long as one accumulation stays below 2^31 rows.
//
// Shape of the work (S padded to a multiple of 256 = W windows of 256 states):
//   * one CTA owns a window pair (I, J), J >= I, and a slice of the rows: its two M128 x N256 s32 accumulators (all
//     512 TMEM columns) hold the 256 x 256 block G[I][J]; slices are sized so that the grid is about one wave;
//   * a pre-pass (pair_prep_kernel) reads the table once, writes a column-major copy and a per-row keep mask (0 for a
//     row holding any bin id outside its column's domain, and for the padding rows) and counts the skipped rows;
//   * producer warps build the one-hot operand tiles in shared memory: per stage 128 table rows = K, both operands
//     K-major, byte [state][row] with the 128-byte swizzle (one 8-state x 128-row atom = 1 KB).  Every 16-byte chunk
//     (one state x 16 rows) is made in registers by a byte compare of 16 staged bin ids against the state's bin, masked
//     by the keep mask, and stored with one 16-byte write.  A stage holds window I (32 KB) and window J (32 KB; on the
//     diagonal J = I and the B operand points into window I);
//   * one thread issues the MMAs (M128 x N256 x K32, four per stage and accumulator) and frees stages with
//     tcgen05.commit; on the diagonal the second accumulator's left half is below the diagonal and skipped (N128);
//   * after the slice the producer warps drain TMEM (tcgen05.ld) and add every needed entry into the global 64-bit
//     counters of the output layout below.
//
// Output layout (bc_pair_counts; mirrored by bayescard_b200/structure.py:pair_count_layout): per column i its marginal
// counts (card_i, at C_i = sum_{k<i} card_k), then for every pair i < j in row-major pair order the block
// card_i x card_j, row-major ([a][b] at S + P_i + card_i * (C_j - C_{i+1}) + a * card_j + b, P_i = sum_{k<i} card_k *
// (S - C_{k+1})).  G[s_a][s_b] goes to the marginal of s_a if s_a == s_b, to the pair block if col(s_a) < col(s_b),
// and is dropped otherwise (the lower triangle; two bins of one column never co-occur).
#include <algorithm>
#include <cmath>

#include "bc_internal.h"

namespace {

constexpr int kTileRows = 128;                    // K per stage: one 128-byte swizzle atom of int8
constexpr int kWin = 256;                         // states per window
constexpr int kWinBytes = kWin * kTileRows;       // 32 KB of one-hot per window and stage
constexpr int kStageBytes = 2 * kWinBytes;
constexpr int kStages = 3;
constexpr int kProdWarps = 8;                     // also the epilogue warps
constexpr int kThreads = 32 * (kProdWarps + 1);   // + the MMA warp
constexpr int kMaxItems = 2 * kWin;               // runs of <= 8 states of one column, per window pair
constexpr int kRun = 8;
constexpr size_t kSmem = (size_t)kStages * kStageBytes + kMaxItems * sizeof(int2) + 256 + 1024;
constexpr long long kMaxSliceRows = 1ll << 30;    // s32 accumulators: a slice stays far below 2^31 rows
constexpr int kMaxStates = 16384;                 // padded S: ~1 GB of 64-bit counters

struct PairArgs {
    const void* cm;                  // column-major copy [n_cols][ld] of the table (element type T)
    const uint8_t* keep;             // [ld] 1: the row is counted
    size_t ld;                       // rows padded to a multiple of 128
    int n_win, n_pairs, n_tiles, tiles_per_slice;
    const int2* items;               // per window: runs {col, s_local | n << 9 | bin0 << 13}
    const int* win_item_off;         // [n_win + 1]
    const int* st_col;               // [n_win * 256] column of a state, -1 for padding
    const int* st_bin;               // [n_win * 256]
    const int* col_card;             // [n_cols]
    const int* col_first;            // [n_cols] C_i
    const long long* row_base;       // [n_cols] S + P_i - card_i * C_{i+1}
    unsigned long long* counts;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint32_t bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, unsigned parity) {
    asm volatile(
        "{\n.reg .pred p;\nWAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// K-major operand, 128-byte swizzle: rows (states) of 128 B, 8-row atoms 1024 B apart (SBO), layout type 2, version 1
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_c),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// 0x01 in every byte of x that is zero, else 0x00 (no carries across bytes: (x & 0x7f) + 0x7f <= 0xfe)
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
    return (~(x | ((x & 0x7f7f7f7fu) + 0x7f7f7f7fu)) >> 7) & 0x01010101u;
}
__device__ __forceinline__ uint32_t zero_halves(uint32_t x) {
    return (~(x | ((x & 0x7fff7fffu) + 0x7fff7fffu)) >> 15) & 0x00010001u;
}

// 16 staged bin ids of one column (16 consecutive rows) -> the one-hot bytes of state `bin`, masked by `keep`
template <typename T>
struct Chunk;
template <>
struct Chunk<uint8_t> {
    uint4 d;
    __device__ __forceinline__ void load(const uint8_t* p) { d = __ldg(reinterpret_cast<const uint4*>(p)); }
    __device__ __forceinline__ uint4 onehot(uint32_t bin, uint4 keep) const {
        const uint32_t b = bin * 0x01010101u;
        return make_uint4(zero_bytes(d.x ^ b) & keep.x, zero_bytes(d.y ^ b) & keep.y, zero_bytes(d.z ^ b) & keep.z,
                          zero_bytes(d.w ^ b) & keep.w);
    }
};
template <>
struct Chunk<uint16_t> {
    uint4 d0, d1;
    __device__ __forceinline__ void load(const uint16_t* p) {
        d0 = __ldg(reinterpret_cast<const uint4*>(p));
        d1 = __ldg(reinterpret_cast<const uint4*>(p) + 1);
    }
    __device__ __forceinline__ uint4 onehot(uint32_t bin, uint4 keep) const {
        const uint32_t b = bin * 0x00010001u;
        // rows 2k, 2k+1 sit in the halves of word k; __byte_perm(lo, hi, 0x6420) packs four rows into four bytes
        return make_uint4(__byte_perm(zero_halves(d0.x ^ b), zero_halves(d0.y ^ b), 0x6420) & keep.x,
                          __byte_perm(zero_halves(d0.z ^ b), zero_halves(d0.w ^ b), 0x6420) & keep.y,
                          __byte_perm(zero_halves(d1.x ^ b), zero_halves(d1.y ^ b), 0x6420) & keep.z,
                          __byte_perm(zero_halves(d1.z ^ b), zero_halves(d1.w ^ b), 0x6420) & keep.w);
    }
};

template <typename T>
__global__ void __launch_bounds__(kThreads, 1) pair_count_kernel(const __grid_constant__ PairArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    int2* s_items = reinterpret_cast<int2*>(smem + kStages * kStageBytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_items + kMaxItems);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 1);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + kStages), acc_full = smem_u32(bars + 2 * kStages);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // block -> (row slice, window pair I <= J); consecutive blocks share a slice (its table rows stay in L2)
    const int slice = blockIdx.x / a.n_pairs;
    int p = blockIdx.x - slice * a.n_pairs, I = 0;
    while (p >= a.n_win - I) p -= a.n_win - I++;
    const int J = I + p;
    const bool diag = I == J;
    const int t0 = slice * a.tiles_per_slice;
    const int nt = min(a.tiles_per_slice, a.n_tiles - t0);
    const int ia = a.win_item_off[I], n_a = a.win_item_off[I + 1] - ia;
    const int ib = a.win_item_off[J], n_b = diag ? 0 : a.win_item_off[J + 1] - ib;
    for (int i = threadIdx.x; i < n_a + n_b; i += blockDim.x) {
        int2 it = i < n_a ? a.items[ia + i] : a.items[ib + i - n_a];
        if (i >= n_a) it.y += kWin;  // window J is the second half of the stage
        s_items[i] = it;
    }
    // padding states are never written by the producers: zero every stage once
    for (int i = threadIdx.x; i < kStages * kStageBytes / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(full0 + 8 * s, 32 * kProdWarps);
            mbar_init(empty0 + 8 * s, 1);
        }
        mbar_init(acc_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kProdWarps) {  // TMEM: two accumulators of 256 s32 columns x 128 lanes
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the zero fill, before the tensor core reads it
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;

    if (warp == kProdWarps) {
        if (lane == 0) {  // ---- MMA issuer.  D = S32, A = B = U8, both K-major, M = 128, N = 256 (128)
            constexpr uint32_t id256 = (2u << 4) | ((256u >> 3) << 17) | ((128u >> 4) << 24);
            constexpr uint32_t id128 = (2u << 4) | ((128u >> 3) << 17) | ((128u >> 4) << 24);
            constexpr uint64_t half = (128 * kTileRows) >> 4;  // 128 states further: 16 KB in descriptor units
            for (int k = 0; k < nt; ++k) {
                const int s = k % kStages;
                mbar_wait(full0 + 8 * s, (k / kStages) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t base = smem_u32(smem + s * kStageBytes);
                const uint64_t da = umma_desc(base), db = umma_desc(diag ? base : base + kWinBytes);
#pragma unroll
                for (int kk = 0; kk < kTileRows / 32; ++kk) {  // K = 32 bytes per MMA: +2 in the 16-byte address field
                    const uint64_t o = (uint64_t)(kk * 2);
                    const uint32_t acc = (k | kk) != 0;
                    umma_i8(tmem, da + o, db + o, id256, acc);
                    if (diag)  // states 128..255 of I against 128..255 of J = I: the rest is below the diagonal
                        umma_i8(tmem + 256 + 128, da + half + o, db + half + o, id128, acc);
                    else
                        umma_i8(tmem + 256, da + half + o, db + o, id256, acc);
                }
                umma_commit(empty0 + 8 * s);
            }
            umma_commit(acc_full);
        }
    } else {
        // ---- producers: thread -> (16-row group g, item slot); a run of states of one column shares its bin ids
        const int pt = threadIdx.x, g = pt & 7, slot = pt >> 3;
        const T* cm = static_cast<const T*>(a.cm);
        for (int k = 0; k < nt; ++k) {
            const int s = k % kStages;
            mbar_wait(empty0 + 8 * s, ((k / kStages) & 1) ^ 1);
            uint8_t* st = smem + s * kStageBytes;
            const size_t r0 = (size_t)(t0 + k) * kTileRows + g * 16;
            const uint4 keep = __ldg(reinterpret_cast<const uint4*>(a.keep + r0));
            for (int i = slot; i < n_a + n_b; i += 32 * kProdWarps / 8) {
                const int2 it = s_items[i];
                const int s0 = it.y & 511, n = (it.y >> 9) & 15;
                const uint32_t bin0 = (uint32_t)it.y >> 13;
                Chunk<T> c;
                c.load(cm + (size_t)it.x * a.ld + r0);
                for (int j = 0; j < n; ++j) {
                    const int sx = s0 + j;
                    const uint4 v = c.onehot(bin0 + j, keep);
                    *reinterpret_cast<uint4*>(st + (sx >> 3) * 1024 + (sx & 7) * 128 + ((g ^ (sx & 7)) << 4)) = v;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> tensor-core reads
            mbar_arrive(full0 + 8 * s);
        }
        // ---- epilogue: warp w reads TMEM lane quarter w % 4 (hardware rule), columns 128 * (w / 4) ..
        mbar_wait(acc_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int quarter = warp & 3, chalf = warp >> 2, m = quarter * 32 + lane;
        for (int h = 0; h < 2; ++h) {
            const int sa = I * kWin + h * 128 + m;
            const int ca = a.st_col[sa], ba = a.st_bin[sa];
            const long long base = ca >= 0 ? a.row_base[ca] : 0;
            const int card_a = ca >= 0 ? a.col_card[ca] : 0;
            for (int c0 = chalf * 128; c0 < chalf * 128 + 128; c0 += 32) {
                uint32_t v[32];
                tmem_ld32(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(h * 256 + c0), v);
                if (ca < 0) continue;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (!v[j]) continue;
                    const int sb = J * kWin + c0 + j;
                    if (sb == sa) {
                        atomicAdd(&a.counts[a.col_first[ca] + ba], (unsigned long long)v[j]);
                    } else {
                        const int cb = a.st_col[sb];
                        if (cb > ca)
                            atomicAdd(&a.counts[base + (long long)card_a * a.col_first[cb] + (long long)ba * a.col_card[cb] + a.st_bin[sb]],
                                      (unsigned long long)v[j]);
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kProdWarps) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
    }
}

// table (row-major, any row stride) -> column-major copy + keep mask; skipped rows counted into *skipped
template <typename T>
__global__ void __launch_bounds__(256) pair_prep_kernel(const T* __restrict__ table, size_t n_rows, size_t row_stride, int n_cols,
                                                        const int* __restrict__ card, size_t ld, T* __restrict__ cm,
                                                        uint8_t* __restrict__ keep, unsigned long long* skipped) {
    // ld is a multiple of 128 and the grid a multiple of 32 threads: a warp's lanes leave the loop together
    for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < ld; r += (size_t)gridDim.x * blockDim.x) {
        const bool real = r < n_rows;
        const T* row = table + (real ? r : 0) * row_stride;
        bool ok = real;
        for (int c = 0; c < n_cols; ++c) {
            const T v = real ? row[c] : T(0);
            ok = ok && (int)v < __ldg(card + c);
            cm[(size_t)c * ld + r] = v;
        }
        keep[r] = ok ? 1 : 0;
        const unsigned bad = __ballot_sync(0xffffffffu, real && !ok);
        if (bad && (threadIdx.x & 31) == 0) atomicAdd(skipped, (unsigned long long)__popc(bad));
    }
}


// MI[i][j] = sum_ab (n_ab / N) log(N n_ab / (n_a n_b)) over n_ab > 0, fp64; one warp per pair i < j, both halves written
__global__ void __launch_bounds__(256) pair_mi_kernel(const unsigned long long* __restrict__ counts, int n_cols,
                                                      const int* __restrict__ card, const int* __restrict__ first,
                                                      const long long* __restrict__ row_base, double N, double* __restrict__ mi) {
    const int i = blockIdx.y, j = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (j <= i || j >= n_cols) return;
    const int ci = card[i], cj = card[j];
    const unsigned long long* ma = counts + first[i];
    const unsigned long long* mb = counts + first[j];
    const unsigned long long* blk = counts + row_base[i] + (long long)ci * first[j];
    double sum = 0.0;
    for (int e = lane; e < ci * cj; e += 32) {
        const unsigned long long nab = blk[e];
        if (!nab) continue;
        const int x = e / cj, y = e - x * cj;
        const double f = (double)nab;
        sum += (f / N) * log((N * f) / ((double)ma[x] * (double)mb[y]));
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) mi[(size_t)i * n_cols + j] = mi[(size_t)j * n_cols + i] = sum;
}

// Host-side plan: state tables, runs of states per window, layout offsets.  Everything is checked here, before any
// device work.
struct Plan {
    int n_cols = 0, n_win = 0;
    long long S = 0, n_counters = 0;
    std::vector<int> st_col, st_bin, win_off, card, first;
    std::vector<int2> items;
    std::vector<long long> row_base;
};

int make_plan(const char* who, int n_cols, const int32_t* card, int elem_bytes, Plan& pl) {
    if (n_cols < 2 || !card || (elem_bytes != 1 && elem_bytes != 2)) {
        bc_set_error("%s: bad arguments (n_cols %d >= 2, card non-null, elem_bytes %d in {1, 2})", who, n_cols, elem_bytes);
        return BC_EINVAL;
    }
    const int max_card = elem_bytes == 1 ? 256 : 65536;
    long long S = 0;
    for (int c = 0; c < n_cols; ++c) {
        if (card[c] <= 0 || card[c] > max_card) {
            bc_set_error("%s: column %d: card %d outside 1..%d (the element type)", who, c, card[c], max_card);
            return BC_EINVAL;
        }
        S += card[c];
    }
    const long long S_pad = bc_round_up(S, kWin);
    if (S_pad > kMaxStates) {
        bc_set_error("%s: sum of the cards %lld (padded %lld) exceeds %d states (the 64-bit counters of all pairs would "
                     "exceed ~1 GB)", who, S, S_pad, kMaxStates);
        return BC_ELIMIT;
    }
    pl.n_cols = n_cols;
    pl.S = S;
    pl.n_win = (int)(S_pad / kWin);
    pl.card.assign(card, card + n_cols);
    pl.first.resize(n_cols);
    pl.row_base.resize(n_cols);
    pl.st_col.assign(S_pad, -1);
    pl.st_bin.assign(S_pad, 0);
    long long C = 0, P = 0;
    for (int c = 0; c < n_cols; ++c) {
        pl.first[c] = (int)C;
        for (int b = 0; b < card[c]; ++b) {
            pl.st_col[C + b] = c;
            pl.st_bin[C + b] = b;
        }
        C += card[c];
        pl.row_base[c] = S + P - (long long)card[c] * C;  // + card_c * C_j gives the block (c, j)
        P += (long long)card[c] * (S - C);
    }
    pl.n_counters = S + P;
    pl.win_off.assign(1, 0);
    for (int w = 0; w < pl.n_win; ++w) {
        for (int s = w * kWin; s < (w + 1) * kWin && pl.st_col[s] >= 0;) {
            int n = 1;
            while (n < kRun && s + n < (w + 1) * kWin && pl.st_col[s + n] == pl.st_col[s]) ++n;
            pl.items.push_back(make_int2(pl.st_col[s], (s - w * kWin) | (n << 9) | (pl.st_bin[s] << 13)));
            s += n;
        }
        pl.win_off.push_back((int)pl.items.size());
    }
    return BC_OK;
}

// One device buffer with all the plan's tables (uploaded with one copy) and the scratch of a counting pass.
struct DevPlan {
    uint8_t* buf = nullptr;
    PairArgs args{};
};

template <typename X>
static size_t put(std::vector<uint8_t>& host, const std::vector<X>& v) {
    const size_t off = bc_round_up((int64_t)host.size(), 16);
    host.resize(off + v.size() * sizeof(X));
    if (!v.empty()) memcpy(host.data() + off, v.data(), v.size() * sizeof(X));
    return off;
}

int upload_plan(const Plan& pl, size_t n_rows, int elem_bytes, DevPlan& dp, cudaStream_t st) {
    std::vector<uint8_t> host;
    const size_t o_items = put(host, pl.items), o_win = put(host, pl.win_off), o_col = put(host, pl.st_col),
                 o_bin = put(host, pl.st_bin), o_card = put(host, pl.card), o_first = put(host, pl.first),
                 o_base = put(host, pl.row_base);
    const size_t n_tiles = (n_rows + kTileRows - 1) / kTileRows, ld = n_tiles * kTileRows;
    const size_t o_keep = bc_round_up((int64_t)host.size(), 256), o_cm = o_keep + ld;
    const size_t bytes = o_cm + (size_t)pl.n_cols * ld * elem_bytes;
    BC_CUDA_CHECK(cudaMallocAsync(&dp.buf, bytes, st));
    // pageable source: the copy is staged by the runtime before the call returns
    BC_CUDA_CHECK(cudaMemcpyAsync(dp.buf, host.data(), host.size(), cudaMemcpyHostToDevice, st));
    PairArgs& a = dp.args;
    a.cm = dp.buf + o_cm;
    a.keep = dp.buf + o_keep;
    a.ld = ld;
    a.n_win = pl.n_win;
    a.n_pairs = pl.n_win * (pl.n_win + 1) / 2;
    a.n_tiles = (int)n_tiles;
    a.items = reinterpret_cast<const int2*>(dp.buf + o_items);
    a.win_item_off = reinterpret_cast<const int*>(dp.buf + o_win);
    a.st_col = reinterpret_cast<const int*>(dp.buf + o_col);
    a.st_bin = reinterpret_cast<const int*>(dp.buf + o_bin);
    a.col_card = reinterpret_cast<const int*>(dp.buf + o_card);
    a.col_first = reinterpret_cast<const int*>(dp.buf + o_first);
    a.row_base = reinterpret_cast<const long long*>(dp.buf + o_base);
    return BC_OK;
}

int check_table(const char* who, const void* table_dev, size_t n_rows, size_t row_stride, int n_cols) {
    if ((!table_dev && n_rows) || row_stride < (size_t)n_cols) {
        bc_set_error("%s: %s", who, !table_dev && n_rows ? "table is NULL with rows" : "row stride < n_cols");
        return BC_EINVAL;
    }
    if (n_rows > (size_t)INT32_MAX * kTileRows) {
        bc_set_error("%s: %zu rows: more than 2^31 tiles of 128 rows", who, n_rows);
        return BC_ELIMIT;
    }
    return BC_OK;
}

// counts_dev: n_counters + 1 counters (the last one: skipped rows), zeroed here
int count_pairs(int device, const Plan& pl, DevPlan& dp, const void* table_dev, int elem_bytes, size_t n_rows,
                size_t row_stride, unsigned long long* counts_dev, cudaStream_t st) {
    BC_CUDA_CHECK(cudaMemsetAsync(counts_dev, 0, sizeof(unsigned long long) * (pl.n_counters + 1), st));
    if (!n_rows) return BC_OK;
    int sm_count = 0;
    BC_CUDA_CHECK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    PairArgs& a = dp.args;
    a.counts = counts_dev;
    const long long prep_grid = std::min<long long>((long long)(a.ld / 256) + 1, (long long)sm_count * 8);
    if (elem_bytes == 1)
        pair_prep_kernel<uint8_t><<<(unsigned)prep_grid, 256, 0, st>>>(static_cast<const uint8_t*>(table_dev), n_rows, row_stride,
                                                                        pl.n_cols, a.col_card, a.ld, (uint8_t*)a.cm,
                                                                        (uint8_t*)a.keep, counts_dev + pl.n_counters);
    else
        pair_prep_kernel<uint16_t><<<(unsigned)prep_grid, 256, 0, st>>>(static_cast<const uint16_t*>(table_dev), n_rows, row_stride,
                                                                         pl.n_cols, a.col_card, a.ld, (uint16_t*)a.cm,
                                                                         (uint8_t*)a.keep, counts_dev + pl.n_counters);
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch();
    // row slices: about one wave of one-CTA-per-SM blocks, every slice below 2^30 rows (s32 accumulators)
    long long n_slices = std::max(1, sm_count / a.n_pairs);
    n_slices = std::min<long long>(n_slices, a.n_tiles);
    long long per = (a.n_tiles + n_slices - 1) / n_slices;
    per = std::min<long long>(per, kMaxSliceRows / kTileRows);
    n_slices = (a.n_tiles + per - 1) / per;
    a.tiles_per_slice = (int)per;
    static bool attr_set[64] = {};
    if (device < 0 || device >= 64 || !attr_set[device]) {
        BC_CUDA_CHECK(cudaFuncSetAttribute(pair_count_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
        BC_CUDA_CHECK(cudaFuncSetAttribute(pair_count_kernel<uint16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmem));
        if (device >= 0 && device < 64) attr_set[device] = true;
    }
    const long long grid = n_slices * a.n_pairs;
    if (grid > INT32_MAX) {
        bc_set_error("bc_pair_counts: %lld blocks", grid);
        return BC_ELIMIT;
    }
    if (elem_bytes == 1)
        pair_count_kernel<uint8_t><<<(unsigned)grid, kThreads, kSmem, st>>>(a);
    else
        pair_count_kernel<uint16_t><<<(unsigned)grid, kThreads, kSmem, st>>>(a);
    BC_CUDA_CHECK(cudaGetLastError());
    bc_count_launch();
    return BC_OK;
}

int read_skipped(const unsigned long long* counter_dev, uint64_t* out, cudaStream_t st) {
    BC_CUDA_CHECK(cudaMemcpyAsync(out, counter_dev, sizeof(*out), cudaMemcpyDeviceToHost, st));
    BC_CUDA_CHECK(cudaStreamSynchronize(st));
    return BC_OK;
}

}  // namespace

extern "C" int bc_pair_counts(int device, int n_cols, const int32_t* card, const void* table_dev, int elem_bytes, size_t n_rows,
                              size_t row_stride_elems, unsigned long long* counts_dev, size_t n_counters,
                              uint32_t* bad_rows_host, void* stream) {
    Plan pl;
    int rc = make_plan("bc_pair_counts", n_cols, card, elem_bytes, pl);
    if (rc) return rc;
    if ((rc = check_table("bc_pair_counts", table_dev, n_rows, row_stride_elems, n_cols))) return rc;
    if (!counts_dev || (long long)n_counters != pl.n_counters) {
        bc_set_error("bc_pair_counts: counts buffer %s %zu counters, the layout needs %lld", counts_dev ? "holds" : "is NULL for",
                     n_counters, pl.n_counters);
        return BC_EINVAL;
    }
    BC_CUDA_CHECK(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DevPlan dp;
    if ((rc = upload_plan(pl, n_rows, elem_bytes, dp, st))) return rc;
    rc = count_pairs(device, pl, dp, table_dev, elem_bytes, n_rows, row_stride_elems, counts_dev, st);
    cudaFreeAsync(dp.buf, st);
    if (rc) return rc;
    if (bad_rows_host) {
        uint64_t bad = 0;
        if ((rc = read_skipped(counts_dev + n_counters, &bad, st))) return rc;
        *bad_rows_host = (uint32_t)std::min<uint64_t>(bad, 0xffffffffull);
    }
    return BC_OK;
}

// Prim on the MI matrix with pomegranate's tie rule (discrete_chow_liu_tree): the next edge is the (in-tree x, outside y)
// pair of largest MI, x scanned in the order the nodes joined the tree, y ascending, only a strictly larger MI replacing
// the best so far.  Kept O(n^2): best[y] is the first-joined x of largest MI, and among equal best[y] values the pair
// whose x joined first, then the smallest y, is the one the scan would meet first.
static void prim_tree(int n, const double* mi, int root, int32_t* parent) {
    std::vector<double> best(n, -INFINITY);
    std::vector<int> bx(n, -1), rank(n, -1);
    std::vector<char> in(n, 0);
    int last = root, joined = 0;
    in[root] = 1;
    rank[root] = joined++;
    parent[root] = -1;
    for (int step = 1; step < n; ++step) {
        for (int y = 0; y < n; ++y)
            if (!in[y] && (bx[y] < 0 || mi[(size_t)last * n + y] > best[y])) {
                best[y] = mi[(size_t)last * n + y];
                bx[y] = last;
            }
        int pick = -1;
        for (int y = 0; y < n; ++y) {
            if (in[y]) continue;
            if (pick < 0 || best[y] > best[pick] || (best[y] == best[pick] && rank[bx[y]] < rank[bx[pick]])) pick = y;
        }
        in[pick] = 1;
        rank[pick] = joined++;
        parent[pick] = bx[pick];
        last = pick;
    }
}

extern "C" int bc_chow_liu(int device, int n_cols, const int32_t* card, const void* table_dev, int elem_bytes, size_t n_rows,
                           size_t row_stride_elems, int root, unsigned long long* counts_dev, size_t n_counters,
                           int32_t* parent_host, double* mi_host, uint32_t* bad_rows_host, void* stream) {
    Plan pl;
    int rc = make_plan("bc_chow_liu", n_cols, card, elem_bytes, pl);
    if (rc) return rc;
    if ((rc = check_table("bc_chow_liu", table_dev, n_rows, row_stride_elems, n_cols))) return rc;
    if (root < 0 || root >= n_cols || !parent_host) {
        bc_set_error("bc_chow_liu: %s", !parent_host ? "parent output is NULL" : "root outside 0..n_cols-1");
        return BC_EINVAL;
    }
    if (counts_dev && (long long)n_counters != pl.n_counters) {
        bc_set_error("bc_chow_liu: counts buffer holds %zu counters, the layout needs %lld", n_counters, pl.n_counters);
        return BC_EINVAL;
    }
    BC_CUDA_CHECK(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    DevPlan dp;
    if ((rc = upload_plan(pl, n_rows, elem_bytes, dp, st))) return rc;
    unsigned long long* counts = counts_dev;
    double* d_mi = nullptr;
    std::vector<double> mi((size_t)n_cols * n_cols);
    uint64_t bad = 0;
    do {
        if (!counts && (rc = cudaMallocAsync(&counts, sizeof(unsigned long long) * (pl.n_counters + 1), st)) != cudaSuccess) {
            counts = nullptr;
            bc_set_error("bc_chow_liu: cudaMallocAsync of %lld counters failed", pl.n_counters + 1);
            rc = BC_ENOMEM;
            break;
        }
        if ((rc = count_pairs(device, pl, dp, table_dev, elem_bytes, n_rows, row_stride_elems, counts, st))) break;
        if ((rc = read_skipped(counts + pl.n_counters, &bad, st))) break;
        if (cudaMallocAsync(&d_mi, sizeof(double) * mi.size(), st) != cudaSuccess) {
            d_mi = nullptr;
            bc_set_error("bc_chow_liu: cudaMallocAsync of the %d x %d MI matrix failed", n_cols, n_cols);
            rc = BC_ENOMEM;
            break;
        }
        if (cudaMemsetAsync(d_mi, 0, sizeof(double) * mi.size(), st) != cudaSuccess) { rc = BC_ECUDA; break; }
        const PairArgs& a = dp.args;
        pair_mi_kernel<<<dim3((n_cols + 7) / 8, n_cols), 256, 0, st>>>(counts, n_cols, a.col_card, a.col_first, a.row_base,
                                                                     (double)(n_rows - bad), d_mi);
        bc_count_launch();
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(mi.data(), d_mi, sizeof(double) * mi.size(), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            bc_set_error("bc_chow_liu: %s", cudaGetErrorString(e));
            rc = BC_ECUDA;
        }
    } while (0);
    if (d_mi) cudaFreeAsync(d_mi, st);
    if (counts && counts != counts_dev) cudaFreeAsync(counts, st);
    cudaFreeAsync(dp.buf, st);
    if (rc) return rc;
    prim_tree(n_cols, mi.data(), root, parent_host);
    if (mi_host) std::copy(mi.begin(), mi.end(), mi_host);
    if (bad_rows_host) *bad_rows_host = (uint32_t)std::min<uint64_t>(bad, 0xffffffffull);
    return BC_OK;
}
