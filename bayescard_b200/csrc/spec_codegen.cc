// K-spec code generator: turns ONE learned tree into straight-line sm_100a PTX.
//
// The reference's docstring promises exactly this -- "Compiles a ppl program into a fixed linear
// algebra program to speed up the inference" (Pgmpy/inference/ExactInference.py:113-114) -- but
// re-plans every query in Python (copy.deepcopy per node, :100).  Here the plan is fixed at model
// load: one THREAD evaluates one query; every message vector lives in registers; every non-zero
// CPT entry T_v[c][p] is the 32-bit immediate of exactly one FMA-pipe instruction; there is no
// shared memory, no synchronisation and no data-dependent branch.
//
//   m_v[p]   = sum_c w_v[c] * lambda_v[c] * T_v[c][p]
//   lambda_v = prod_{children k} m_k                       (registers)
//   result   = sum_c w_0[c] * lambda_0[c] * T_0[c]
//
// Two entry points are generated (PTX, so that instruction selection is ours, not a C compiler's):
//
//   bc_spec_bits   w is a BITS row.  The state's bit becomes a PREDICATE (ptxas packs seven of them
//                  per R2P) and guards the FMAs of that state directly:
//                      @p fma.rn.f32 m_p, lambda_c, T, m_p        (leaf:  @p add.f32 m_p, m_p, T)
//                  so selecting costs ~1/7 ALU instruction per state instead of one select per
//                  state.  The first state of every node seeds the accumulators through one select
//                  + multiplies, which removes the zero-initialisation.  On B200 an ALU-pipe
//                  instruction costs two issue slots and an FMA-pipe one costs one (measured,
//                  profiles/r1_microbench_pipes.txt), hence the care.
//   bc_spec_dense  w is a DENSE_F32 row (fractional n_distinct weights): u = w * lambda, plain FMAs.
//
// Children are evaluated largest-subtree first so that the fewest message vectors are live at
// once (Sethi-Ullman order).  Exact zeros of the CPT (30 % of the shipped DMV / Census entries)
// emit no instruction; the number of FMAs actually emitted is reported in the header comment of
// the generated source (BC_SPEC_FFMA) and is what the roofline accounting uses.
//
// A second module per (model, target node t) answers GROUP BY t (bc_marginal_generate): out[q][b] for every state b of t.
// Every subtree off the root -> t path is evaluated upward as above; then a downward chain along the path carries
//   pi_0 = w_0 * lambda_0 * T_0,   pi_i[c] = w_i[c] * lambda_i[c] * sum_p T_i[c][p] * pi_{i-1}[p],   out = pi_k
// (lambda_i: product of the messages of a_i's children off the path), again one FMA per non-zero CPT entry.  Both passes
// apply the fan-out mask (p_fmask) as the spec module does: bit v multiplies w_v by fanouts[v].
//
// A third module per (model, ordered pair a, b) answers GROUP BY a, b (bc_joint_generate): out[q][i][j], the marginal's chain
// down to the two targets' lowest common ancestor, then a loop unrolled over the states of one target (gen_joint_body).
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>

#include "bc_internal.h"

namespace {

std::string fhex(float x) {
    uint32_t b;
    std::memcpy(&b, &x, 4);
    char s[16];
    snprintf(s, sizeof(s), "0f%08X", b);
    return s;
}
inline std::string I(long long x) { return std::to_string(x); }

// Experiment knobs (they are part of the image hash, so every variant has its own cache entry):
//   BC_SPEC_SYNC_EVERY=N   re-align the warps of a CTA with bar.sync every N generated instructions.  The code of
//                          a big tree is a straight line of 100-400 KB, larger than the SM's instruction cache;
//                          warps that drift apart each stream it from L2 on their own, warps kept within one
//                          cache-sized window of each other share the fetched lines.
//   BC_SPEC_DYNAMIC=0      back to the static split.  By DEFAULT the CTAs take their rounds of ntid queries from a global
//                          counter (p_ctr) instead of a fixed stride: SMs do not all run this fetch-bound code at the
//                          same speed (ncu: 510-679 k active cycles per SM on DMV), and with a static split the
//                          slowest SM sets the time.  Measured (profiles/r1_spec_dynamic.txt): DMV 3.00 -> 3.55e9 q/s
//                          (63 -> 75 % of the FP32 peak), Census 9.8 -> 10.8e9 (60 -> 66 %), IMDB unchanged.
//   BC_SPEC_THREADS / BC_SPEC_MIN_BLOCKS   override the CTA geometry chosen by bc_spec_geometry.
int env_int(const char* name, int dflt) {
    const char* e = std::getenv(name);
    if (!e || !*e) return dflt;
    const int v = std::atoi(e);
    return v >= 0 ? v : dflt;
}

struct Gen {
    const bc_model& m;
    const bool dense;
    std::vector<std::vector<int>> kids;
    std::string out;
    long long n_fma = 0;
    int nf = 0, np = 0, nr = 0;
    bool any_fan = false;
    std::vector<std::string> words;  // BITS row words / (dense: unused)
    std::vector<std::string> fmw;    // fan-out mask words

    Gen(const bc_model& mm, bool d) : m(mm), dense(d), kids(mm.n) {
        std::vector<long long> subtree(m.n, 0);
        for (int v = 1; v < m.n; ++v) kids[m.nodes[v].parent].push_back(v);
        for (int v = m.n - 1; v >= 0; --v) {
            subtree[v] += m.nodes[v].card;
            if (v > 0) subtree[m.nodes[v].parent] += subtree[v];
            if (m.nodes[v].fan_off >= 0) any_fan = true;
        }
        for (int v = 0; v < m.n; ++v)
            std::stable_sort(kids[v].begin(), kids[v].end(), [&](int a, int b) { return subtree[a] > subtree[b]; });
    }

    std::string F() { return "%f" + I(++nf); }
    std::string P() { return "%p" + I(++np); }
    std::string R() { return "%r" + I(++nr); }
    int sync_every = 0, since_sync = 0;
    void line(const std::string& s) {
        out += "    "; out += s; out += '\n';
        if (sync_every > 0 && ++since_sync >= sync_every && s[0] != '/') {
            out += "    bar.sync 0;\n";
            since_sync = 0;
        }
    }

    // The predicate "bit v of the query's fan-out mask is set" (a NULL mask loads words of 0: never set).
    std::string fan_pred(int v) {
        std::string t = R(), p = P();
        line("and.b32 " + t + ", " + fmw[v >> 5] + ", " + I(1LL << (v & 31)) + ";");
        line("setp.ne.u32 " + p + ", " + t + ", 0;");
        return p;
    }

    std::string bit_pred(int v, int c) {
        const int b = m.bits[v].bit_off + c;
        std::string t = R(), p = P();
        line("and.b32 " + t + ", " + words[b >> 5] + ", " + I(1LL << (b & 31)) + ";");
        line("setp.ne.u32 " + p + ", " + t + ", 0;");
        return p;
    }

    // Emits the message of node v; returns its registers, one per parent state (root: one).
    std::vector<std::string> message(int v) {
        const BcNodeRec& nd = m.nodes[v];
        const bool root = v == 0;
        const int card = nd.card, cols = root ? 1 : nd.card_pa;
        line("// ---- node " + I(v) + ": card " + I(card) + (root ? " (root)" : ", parent " + I(nd.parent)));
        std::vector<std::string> lam;
        for (int k : kids[v]) {
            std::vector<std::string> mk = message(k);
            if (lam.empty()) lam = mk;
            else
                for (int c = 0; c < card; ++c) line("mul.f32 " + lam[c] + ", " + lam[c] + ", " + mk[c] + ";");
        }
        const bool fan = nd.fan_off >= 0;
        const std::string pfb = fan ? fan_pred(v) : std::string();
        const float* T = m.arena.data() + nd.cpt_off;
        const int stride = root ? 1 : nd.stride;
        auto Tat = [&](int c, int p) { return root ? T[c] : T[(size_t)c * stride + p]; };
        // the seed row: the state with the most non-zero entries (fewest accumulators left to zero)
        int seed = 0, best = -1;
        for (int c = 0; c < card; ++c) {
            int nz = 0;
            for (int p = 0; p < cols; ++p) nz += Tat(c, p) != 0.f;
            if (nz > best) { best = nz; seed = c; }
        }
        std::vector<std::string> acc(cols);
        std::vector<int> order;
        order.push_back(seed);
        for (int c = 0; c < card; ++c)
            if (c != seed) order.push_back(c);
        // dense rows: the weights of this node are loaded four at a time, right before the first state of the group
        // is folded in (loading the whole node up front keeps up to card more registers live and spills on IMDB)
        std::vector<std::string> wreg(dense ? ((card + 3) / 4) * 4 : 0);
        auto need_weight = [&](int c) {
            const int j = c / 4;
            if (!wreg[4 * j].empty()) return;
            std::string a = F(), b = F(), c2 = F(), d = F();
            line("ld.global.nc.v4.f32 {" + a + ", " + b + ", " + c2 + ", " + d + "}, [%rrow+" + I(4LL * (nd.lam_off + 4 * j)) + "];");
            wreg[4 * j] = a; wreg[4 * j + 1] = b; wreg[4 * j + 2] = c2; wreg[4 * j + 3] = d;
        };
        for (int c : order) {
            bool any = false;
            for (int p = 0; p < cols; ++p) any |= Tat(c, p) != 0.f;
            if (!any && c != seed) continue;
            // lambda of this state, times the fan-out value when the query's fan bit is set
            std::string lc = lam.empty() ? std::string() : lam[c];
            if (fan) {
                const std::string fv = fhex(m.fan[nd.fan_off + c]);
                if (lc.empty()) {
                    lc = F();
                    line("selp.f32 " + lc + ", " + fv + ", 0f3F800000, " + pfb + ";");
                } else {
                    line("@" + pfb + " mul.f32 " + lc + ", " + lc + ", " + fv + ";");
                }
            }
            if (dense) {
                need_weight(c);
                std::string u = wreg[c];
                if (!lc.empty()) {
                    u = F();
                    line("mul.f32 " + u + ", " + wreg[c] + ", " + lc + ";");
                }
                for (int p = 0; p < cols; ++p) {
                    const float t = Tat(c, p);
                    if (c == seed) {
                        acc[p] = F();
                        if (t != 0.f) { line("mul.f32 " + acc[p] + ", " + u + ", " + fhex(t) + ";"); ++n_fma; }
                        else line("mov.f32 " + acc[p] + ", 0f00000000;");
                    } else if (t != 0.f) {
                        line("fma.rn.f32 " + acc[p] + ", " + u + ", " + fhex(t) + ", " + acc[p] + ";");
                        ++n_fma;
                    }
                }
                continue;
            }
            const std::string pc = bit_pred(v, c);
            if (c == seed) {
                std::string u = F();
                line("selp.f32 " + u + ", " + (lc.empty() ? std::string("0f3F800000") : lc) + ", 0f00000000, " + pc + ";");
                for (int p = 0; p < cols; ++p) {
                    const float t = Tat(c, p);
                    acc[p] = F();
                    if (t != 0.f) { line("mul.f32 " + acc[p] + ", " + u + ", " + fhex(t) + ";"); ++n_fma; }
                    else line("mov.f32 " + acc[p] + ", 0f00000000;");
                }
            } else {
                for (int p = 0; p < cols; ++p) {
                    const float t = Tat(c, p);
                    if (t == 0.f) continue;
                    ++n_fma;
                    if (lc.empty()) line("@" + pc + " add.f32 " + acc[p] + ", " + acc[p] + ", " + fhex(t) + ";");
                    else line("@" + pc + " fma.rn.f32 " + acc[p] + ", " + lc + ", " + fhex(t) + ", " + acc[p] + ";");
                }
            }
        }
        return acc;
    }

    // One step of the downward pass of a marginal along the path root = a_0 -> ... -> a_k = target, at path node v = a_i
    // (`skip` = a_{i+1}, -1 at the target).  Folds the messages of v's children off the path into lambda, then emits
    //     pi_i[c] = w_v[c] * lambda[c] * sum_p T_v[c][p] * pi_{i-1}[p]        (root: w_0[c] * lambda[c] * T_0[c])
    // with one FMA-pipe instruction per non-zero T_v[c][p]; returns pi_i, one register per state of v.  A path node with a
    // fan-out vector multiplies each state by fanouts[v][c] under its mask bit (@p mul, or a selp between two immediates at a
    // root without lambda), so a query without that bit computes exactly what the kernel without fan-out does.
    // `skip2`: a second child left out (a joint marginal's lowest common ancestor, whose two children lead to the targets).
    std::vector<std::string> path_step(int v, int skip, const std::vector<std::string>& prev, int skip2 = -1) {
        const BcNodeRec& nd = m.nodes[v];
        const bool root = v == 0;
        const int card = nd.card, cols = root ? 1 : nd.card_pa;
        std::vector<std::string> lam;
        for (int k : kids[v]) {
            if (k == skip || k == skip2) continue;
            std::vector<std::string> mk = message(k);
            if (lam.empty()) lam = mk;
            else
                for (int c = 0; c < card; ++c) line("mul.f32 " + lam[c] + ", " + lam[c] + ", " + mk[c] + ";");
        }
        line("// ---- path node " + I(v) + ": card " + I(card) + (root ? " (root)" : ", parent " + I(nd.parent)) +
             (skip < 0 ? " (target)" : ", next " + I(skip)));
        const bool fan = nd.fan_off >= 0;
        const std::string pfb = fan ? fan_pred(v) : std::string();
        const float* T = m.arena.data() + nd.cpt_off;
        const int stride = root ? 1 : nd.stride;
        std::vector<std::string> wreg(dense ? ((card + 3) / 4) * 4 : 0);
        std::string zero;
        std::vector<std::string> pi(card);
        for (int c = 0; c < card; ++c) {
            std::string x;   // lambda[c] * (T_0[c] | sum_p T[c][p] pi[p]): a register, or the immediate T_0[c]
            if (root) {
                const float t = T[c];
                if (t != 0.f) {
                    ++n_fma;
                    if (lam.empty() && !fan) x = fhex(t);
                    else if (lam.empty()) {   // fp32 T_0[c] * fanouts[c], rounded once as the mul.f32 would round it
                        x = F();
                        line("selp.f32 " + x + ", " + fhex(t * m.fan[nd.fan_off + c]) + ", " + fhex(t) + ", " + pfb + ";");
                    } else {
                        x = F();
                        line("mul.f32 " + x + ", " + lam[c] + ", " + fhex(t) + ";");
                    }
                }
            } else {
                for (int p = 0; p < cols; ++p) {
                    const float t = T[(size_t)c * stride + p];
                    if (t == 0.f) continue;
                    ++n_fma;
                    if (x.empty()) { x = F(); line("mul.f32 " + x + ", " + prev[p] + ", " + fhex(t) + ";"); }
                    else line("fma.rn.f32 " + x + ", " + prev[p] + ", " + fhex(t) + ", " + x + ";");
                }
                if (!x.empty() && !lam.empty()) line("mul.f32 " + x + ", " + x + ", " + lam[c] + ";");
            }
            if (fan && !x.empty() && !(root && lam.empty()))
                line("@" + pfb + " mul.f32 " + x + ", " + x + ", " + fhex(m.fan[nd.fan_off + c]) + ";");
            if (x.empty()) {   // an all-zero CPT row: the state holds no mass
                if (zero.empty()) { zero = F(); line("mov.f32 " + zero + ", 0f00000000;"); }
                pi[c] = zero;
                continue;
            }
            pi[c] = F();
            if (dense) {
                const int j = c / 4;
                if (wreg[4 * j].empty()) {
                    std::string a = F(), b = F(), c2 = F(), d = F();
                    line("ld.global.nc.v4.f32 {" + a + ", " + b + ", " + c2 + ", " + d + "}, [%rrow+" + I(4LL * (nd.lam_off + 4 * j)) + "];");
                    wreg[4 * j] = a; wreg[4 * j + 1] = b; wreg[4 * j + 2] = c2; wreg[4 * j + 3] = d;
                }
                line("mul.f32 " + pi[c] + ", " + wreg[c] + ", " + x + ";");
            } else {
                line("selp.f32 " + pi[c] + ", " + x + ", 0f00000000, " + bit_pred(v, c) + ";");
            }
        }
        return pi;
    }

    // u_v[c] = w_v[c] * fanouts[v][c] (under the mask bit) * prod(messages of v's children other than `skip`): what a node
    // strictly below the lowest common ancestor of a joint marginal contributes to every term, one register per state.
    std::vector<std::string> path_weights(int v, int skip) {
        const BcNodeRec& nd = m.nodes[v];
        const int card = nd.card;
        std::vector<std::string> lam;
        for (int k : kids[v]) {
            if (k == skip) continue;
            std::vector<std::string> mk = message(k);
            if (lam.empty()) lam = mk;
            else
                for (int c = 0; c < card; ++c) line("mul.f32 " + lam[c] + ", " + lam[c] + ", " + mk[c] + ";");
        }
        line("// ---- joint path node " + I(v) + ": card " + I(card) + ", parent " + I(nd.parent) +
             (skip < 0 ? " (target)" : ", next " + I(skip)));
        const bool fan = nd.fan_off >= 0;
        const std::string pfb = fan ? fan_pred(v) : std::string();
        std::vector<std::string> wreg(dense ? ((card + 3) / 4) * 4 : 0), u(card);
        for (int c = 0; c < card; ++c) {
            std::string lc = lam.empty() ? std::string() : lam[c];
            if (fan) {
                const std::string fv = fhex(m.fan[nd.fan_off + c]);
                if (lc.empty()) {
                    lc = F();
                    line("selp.f32 " + lc + ", " + fv + ", 0f3F800000, " + pfb + ";");
                } else {
                    line("@" + pfb + " mul.f32 " + lc + ", " + lc + ", " + fv + ";");
                }
            }
            if (dense) {
                const int j = c / 4;
                if (wreg[4 * j].empty()) {
                    std::string a = F(), b = F(), c2 = F(), d = F();
                    line("ld.global.nc.v4.f32 {" + a + ", " + b + ", " + c2 + ", " + d + "}, [%rrow+" + I(4LL * (nd.lam_off + 4 * j)) + "];");
                    wreg[4 * j] = a; wreg[4 * j + 1] = b; wreg[4 * j + 2] = c2; wreg[4 * j + 3] = d;
                }
                u[c] = wreg[c];
                if (!lc.empty()) {
                    u[c] = F();
                    line("mul.f32 " + u[c] + ", " + wreg[c] + ", " + lc + ";");
                }
            } else {
                u[c] = F();
                line("selp.f32 " + u[c] + ", " + (lc.empty() ? std::string("0f3F800000") : lc) + ", 0f00000000, " + bit_pred(v, c) + ";");
            }
        }
        return u;
    }
};

// Wraps the straight-line body of `g` in the query loop of one entry point and stores `res`, res.size() consecutive floats
// per query (row q at out + 4 * res.size() * q).  With `body_row` > 0 the body stores its own results instead (res is
// empty): body_row floats per query at [%rtmp + 4 k], under %pvalid; the row address is set before the body.
std::string gen_entry(const bc_model& m, Gen& g, const char* name, bool dense, int threads, int min_blocks,
                      const std::vector<std::string>& res, long long body_row = 0) {
    const int sync_every = g.sync_every;
    const int words = m.bits_words;
    const bool dynamic = env_int("BC_SPEC_DYNAMIC", 1) != 0;
    std::string s;
    s += std::string(".visible .entry ") + name +
         "(\n    .param .u64 p_desc,\n    .param .u64 p_stride,\n    .param .u64 p_fmask,\n    .param .u64 p_out,\n"
         "    .param .u64 p_nq,\n    .param .u64 p_ctr\n)\n.maxntid " + I(threads) + ", 1, 1\n.minnctapersm " + I(min_blocks) + "\n{\n";
    s += "    .reg .pred %p<" + I(g.np + 1) + ">;\n    .reg .pred %pfm, %pdone;\n";
    s += "    .reg .f32 %f<" + I(g.nf + 1) + ">;\n    .reg .b32 %r<" + I(g.nr + 1) + ">;\n";
    s += "    .reg .b32 %t0, %t1, %t2, %t3, %t4;\n";
    s += "    .reg .b64 %rdesc, %rstride, %rfmask, %rout, %rnq, %rq, %rstep, %rtmp, %rrow, %rqb, %rqc;\n";
    s += "    .reg .b64 %rctr, %rnext, %rnt, %rtid;\n";
    s += "    .reg .pred %pvalid, %pt0, %plast;\n";
    if (dynamic) s += "    .shared .align 8 .b64 bc_slot[2];\n";
    auto e = [&](const std::string& x) { s += "    " + x + "\n"; };
    e("ld.param.u64 %rdesc, [p_desc];");
    e("ld.param.u64 %rstride, [p_stride];");
    e("ld.param.u64 %rfmask, [p_fmask];");
    e("ld.param.u64 %rout, [p_out];");
    e("ld.param.u64 %rnq, [p_nq];");
    e("cvta.to.global.u64 %rdesc, %rdesc;");
    e("cvta.to.global.u64 %rout, %rout;");
    e("setp.ne.u64 %pfm, %rfmask, 0;");
    e("@%pfm cvta.to.global.u64 %rfmask, %rfmask;");
    const bool clamp = dynamic || sync_every > 0;  // threads past the end recompute the last query and skip the store
    if (dynamic) {
        // Round k of a CTA = ntid consecutive queries starting at the value its thread 0 drew from the global
        // counter; the draw for round k+1 is issued at the start of round k-1 (its latency hides behind a whole
        // round) and handed over through a two-slot shared-memory mailbox, one bar.sync per round.
        e("ld.param.u64 %rctr, [p_ctr];");
        e("cvta.to.global.u64 %rctr, %rctr;");
        e("mov.u32 %t0, %tid.x;");
        e("mov.u32 %t2, %ntid.x;");
        e("cvt.u64.u32 %rtid, %t0;");
        e("cvt.u64.u32 %rnt, %t2;");
        e("setp.eq.u32 %pt0, %t0, 0;");
        e("mov.u32 %t4, bc_slot;");
        e("@%pt0 atom.global.add.u64 %rnext, [%rctr], %rnt;");
        e("@%pt0 st.shared.u64 [%t4], %rnext;");
        e("@%pt0 atom.global.add.u64 %rnext, [%rctr], %rnt;");
        s += "LOOP:\n";
        e("bar.sync 0;");
        e("ld.shared.u64 %rqb, [%t4];");
        e("setp.ge.u64 %pdone, %rqb, %rnq;");
        e("@%pdone bra DONE;");
        e("mov.u32 %t1, bc_slot;");
        e("sub.u32 %t3, %t4, %t1;");
        e("xor.b32 %t3, %t3, 8;");
        e("add.u32 %t4, %t1, %t3;");
        e("@%pt0 st.shared.u64 [%t4], %rnext;");
        e("@%pt0 atom.global.add.u64 %rnext, [%rctr], %rnt;");
        e("add.u64 %rq, %rqb, %rtid;");
    } else {
        // query index of round k:  ((k * warps_per_cta + warp) * n_cta + cta) * 32 + lane.
        // Consecutive warp slots belong to DIFFERENT CTAs, so the last, partial round is spread over all
        // CTAs (and SMs) instead of filling the first ones only.
        e("mov.u32 %t0, %tid.x;");
        e("mov.u32 %t1, %ctaid.x;");
        e("mov.u32 %t2, %ntid.x;");
        e("mov.u32 %t3, %nctaid.x;");
        e("shr.u32 %t4, %t0, 5;");
        e("mad.lo.u32 %t4, %t4, %t3, %t1;");
        e("and.b32 %t0, %t0, 31;");
        e("mul.wide.u32 %rq, %t4, 32;");
        e("cvt.u64.u32 %rtmp, %t0;");
        e("add.u64 %rq, %rq, %rtmp;");
        e("mul.wide.u32 %rstep, %t2, %t3;");
        if (sync_every > 0) e("mul.wide.u32 %rqb, %t1, 32;");  // first query of the CTA's first warp slot
        s += "LOOP:\n";
        if (sync_every > 0) {
            // bar.sync needs a CTA-uniform trip count: loop while the CTA's FIRST slot is in range
            e("setp.ge.u64 %pdone, %rqb, %rnq;");
            e("@%pdone bra DONE;");
        } else {
            e("setp.ge.u64 %pdone, %rq, %rnq;");
            e("@%pdone bra DONE;");
        }
    }
    if (clamp) {
        e("setp.lt.u64 %pvalid, %rq, %rnq;");
        e("sub.u64 %rqc, %rnq, 1;");
        e("min.u64 %rqc, %rqc, %rq;");
        e("mad.lo.u64 %rrow, %rqc, %rstride, %rdesc;");
    } else {
        e("mad.lo.u64 %rrow, %rq, %rstride, %rdesc;");
    }
    if (!dense)
        for (int w = 0; w < words; w += 4)
            e("ld.global.nc.v4.u32 {" + g.words[w] + ", " + g.words[w + 1] + ", " + g.words[w + 2] + ", " + g.words[w + 3] +
              "}, [%rrow+" + I(4LL * w) + "];");
    if (g.any_fan) {
        e(std::string("mad.lo.u64 %rtmp, ") + (clamp ? "%rqc" : "%rq") + ", " + I(4LL * m.mask_words) + ", %rfmask;");
        for (int w = 0; w < m.mask_words; ++w) {
            e("mov.u32 " + g.fmw[w] + ", 0;");
            e("@%pfm ld.global.nc.u32 " + g.fmw[w] + ", [%rtmp+" + I(4LL * w) + "];");
        }
    }
    if (body_row > 0) {
        if (!clamp) e("setp.lt.u64 %pvalid, %rq, %rnq;");
        e("mul.lo.u64 %rtmp, %rq, " + I(4LL * body_row) + ";");
        e("add.u64 %rtmp, %rtmp, %rout;");
    }
    s += g.out;
    if (!res.empty()) {
        if (res.size() == 1) e("shl.b64 %rtmp, %rq, 2;");
        else e("mul.lo.u64 %rtmp, %rq, " + I(4LL * (long long)res.size()) + ";");
        e("add.u64 %rtmp, %rtmp, %rout;");
        for (size_t b = 0; b < res.size(); ++b)
            e(std::string(clamp ? "@%pvalid " : "") + "st.global.f32 [%rtmp" + (b ? "+" + I(4LL * (long long)b) : "") + "], " + res[b] + ";");
    }
    if (!dynamic) {
        e("add.u64 %rq, %rq, %rstep;");
        if (sync_every > 0) e("add.u64 %rqb, %rqb, %rstep;");
    }
    e("bra LOOP;");
    if (dynamic) {
        // The last CTA to leave zeroes the counter for the next launch.  Thread 0 first consumes its outstanding
        // draw (the shift is 0 for any real counter value, but the address now depends on it), so no draw of any
        // CTA can land after the reset.
        s += "DONE:\n";
        e("@!%pt0 bra OUT;");
        e("shr.u64 %rtmp, %rnext, 63;");
        e("add.u64 %rctr, %rctr, %rtmp;");
        e("mov.u32 %t3, %nctaid.x;");
        e("sub.u32 %t3, %t3, 1;");
        e("atom.global.inc.u32 %t1, [%rctr+8], %t3;");
        e("setp.eq.u32 %plast, %t1, %t3;");
        e("mov.b64 %rtmp, 0;");
        e("@%plast st.global.u64 [%rctr], %rtmp;");
        s += "OUT:\n    ret;\n}\n\n";
        return s;
    }
    s += "DONE:\n    ret;\n}\n\n";
    return s;
}

std::string gen_kernel(const bc_model& m, bool dense, int threads, int min_blocks, long long* n_fma) {
    Gen g(m, dense);
    g.sync_every = env_int("BC_SPEC_SYNC_EVERY", 0);
    if (!dense)
        for (int w = 0; w < m.bits_words; ++w) g.words.push_back(g.R());
    for (int w = 0; w < m.mask_words; ++w) g.fmw.push_back(g.R());
    const std::string res = g.message(0)[0];
    if (n_fma) *n_fma = g.n_fma;
    return gen_entry(m, g, dense ? "bc_spec_dense" : "bc_spec_bits", dense, threads, min_blocks, {res});
}

// The marginal of `target`: the upward pass of every subtree off the root -> target path (Gen::message), then the downward
// chain of path_step, then card(target) stores per query.
std::string gen_marginal_kernel(const bc_model& m, int target, bool dense, int threads, int min_blocks, long long* n_fma) {
    Gen g(m, dense);
    g.sync_every = env_int("BC_SPEC_SYNC_EVERY", 0);
    if (!dense)
        for (int w = 0; w < m.bits_words; ++w) g.words.push_back(g.R());
    if (g.any_fan)   // (a model without fan-out vectors gets the same registers, and the same source, as without a mask)
        for (int w = 0; w < m.mask_words; ++w) g.fmw.push_back(g.R());
    std::vector<int> path;
    for (int v = target; v > 0; v = m.nodes[v].parent) path.push_back(v);
    path.push_back(0);
    std::reverse(path.begin(), path.end());
    std::vector<std::string> pi;
    for (size_t i = 0; i < path.size(); ++i) pi = g.path_step(path[i], i + 1 < path.size() ? path[i + 1] : -1, pi);
    if (n_fma) *n_fma = g.n_fma;
    return gen_entry(m, g, dense ? "bc_marg_dense" : "bc_marg_bits", dense, threads, min_blocks, pi);
}

// The joint marginal of (a, b) with loop node X (a or b; Y is the other), c their lowest common ancestor:
//   1. every subtree off the root -> X and root -> Y paths upward (Gen::message), the chain root -> c (path_step, c leaving out
//      both children towards X and Y): pi_c;
//   2. u_v = w_v * fan_v * (messages of v's off-path children) for every v strictly below c on the X - c - Y path;
//   3. for each state i of X, unrolled: X below c: row i of T_X times u_X[i], climbed to c (u folded in at each node), times
//      pi_c; X == c: pi_c[i] times column i of the first CPT towards Y.  Then down to Y as path_step does, with the stored u,
//      and the card(Y) results of this i are stored at once.
// A structural zero (no non-zero CPT entry reaches a state) emits nothing and is stored from a zero register.
struct JointBody {
    long long n_fma = 0, cost = 0, pipe = 0;   // CPT-carrying FMAs; FMA-pipe + store instructions; FMA-pipe instructions
    std::string path;
};

float cpt_at(const bc_model& m, int v, int s, int p) {
    const BcNodeRec& nd = m.nodes[v];
    return m.arena[nd.cpt_off + (v == 0 ? s : (int64_t)s * nd.stride + p)];
}

JointBody gen_joint_body(const bc_model& m, Gen& g, int a, int b, int X, bool dense) {
    g.sync_every = env_int("BC_SPEC_SYNC_EVERY", 0);
    if (!dense)
        for (int w = 0; w < m.bits_words; ++w) g.words.push_back(g.R());
    if (g.any_fan)
        for (int w = 0; w < m.mask_words; ++w) g.fmw.push_back(g.R());
    const int Y = X == a ? b : a;
    auto root_path = [&](int v) {
        std::vector<int> p;
        for (; v > 0; v = m.nodes[v].parent) p.push_back(v);
        p.push_back(0);
        std::reverse(p.begin(), p.end());
        return p;
    };
    const std::vector<int> px = root_path(X), py = root_path(Y);
    size_t d = 0;
    while (d + 1 < px.size() && d + 1 < py.size() && px[d + 1] == py[d + 1]) ++d;
    const int c = px[d];
    const std::vector<int> up(px.begin() + d + 1, px.end());     // c's child towards X ... X (empty: X == c)
    const std::vector<int> down(py.begin() + d + 1, py.end());   // c's child towards Y ... Y (empty: Y == c)
    // 1. off the paths
    std::vector<std::string> pi;
    for (size_t i = 0; i < d; ++i) pi = g.path_step(px[i], px[i + 1], pi);
    const int cx = up.empty() ? -1 : up[0], cy = down.empty() ? -1 : down[0];
    pi = g.path_step(c, cx >= 0 ? cx : cy, pi, cx >= 0 ? cy : -1);
    const int card_c = m.nodes[c].card;
    std::vector<char> pz(card_c);   // all-zero CPT rows of c: path_step's shared zero, no mass
    for (int s = 0; s < card_c; ++s) {
        bool any = false;
        for (int p = 0; p < (c == 0 ? 1 : m.nodes[c].card_pa); ++p) any |= cpt_at(m, c, s, p) != 0.f;
        pz[s] = !any;
    }
    // 2. per-node vectors
    std::vector<std::vector<std::string>> u(m.n);
    for (size_t k = 0; k < up.size(); ++k) u[up[k]] = g.path_weights(up[k], k + 1 < up.size() ? up[k + 1] : -1);
    for (size_t k = 0; k < down.size(); ++k) u[down[k]] = g.path_weights(down[k], k + 1 < down.size() ? down[k + 1] : -1);
    const std::string zero = g.F();
    g.line("mov.f32 " + zero + ", 0f00000000;");
    // fma into x (a fresh register on the first term)
    auto acc = [&](std::string& x, const std::string& r, float t) {
        ++g.n_fma;
        if (x.empty()) { x = g.F(); g.line("mul.f32 " + x + ", " + r + ", " + fhex(t) + ";"); }
        else g.line("fma.rn.f32 " + x + ", " + r + ", " + fhex(t) + ", " + x + ";");
    };
    auto scale = [&](const std::string& x, const std::string& y) { g.line("mul.f32 " + x + ", " + x + ", " + y + ";"); };
    // down[k0..]: r over the states of down[k0]'s parent -> over the states of Y
    auto descend = [&](std::vector<std::string> r, size_t k0) {
        for (size_t k = k0; k < down.size(); ++k) {
            const int v = down[k];
            std::vector<std::string> nr(m.nodes[v].card);
            for (int t = 0; t < m.nodes[v].card; ++t) {
                for (int s = 0; s < m.nodes[v].card_pa; ++s) {
                    const float T = cpt_at(m, v, t, s);
                    if (!r[s].empty() && T != 0.f) acc(nr[t], r[s], T);
                }
                if (!nr[t].empty()) scale(nr[t], u[v][t]);
            }
            r = nr;
        }
        return r;
    };
    // 3. the unrolled loop over the states of X
    const int cb = m.nodes[b].card;
    for (int i = 0; i < m.nodes[X].card; ++i) {
        g.line("// ---- state " + I(i) + " of node " + I(X));
        std::vector<std::string> r;
        if (!up.empty()) {
            std::vector<std::string> vec(m.nodes[X].card_pa);
            for (int p = 0; p < m.nodes[X].card_pa; ++p) {
                const float T = cpt_at(m, X, i, p);
                if (T != 0.f) acc(vec[p], u[X][i], T);
            }
            for (size_t k = up.size() - 1; k-- > 0;) {
                const int w = up[k];
                std::vector<std::string> xin(m.nodes[w].card), nv(m.nodes[w].card_pa);
                for (int s = 0; s < m.nodes[w].card; ++s)
                    if (!vec[s].empty()) {
                        xin[s] = g.F();
                        g.line("mul.f32 " + xin[s] + ", " + vec[s] + ", " + u[w][s] + ";");
                    }
                for (int p = 0; p < m.nodes[w].card_pa; ++p)
                    for (int s = 0; s < m.nodes[w].card; ++s) {
                        const float T = cpt_at(m, w, s, p);
                        if (!xin[s].empty() && T != 0.f) acc(nv[p], xin[s], T);
                    }
                vec = nv;
            }
            r.assign(card_c, std::string());
            for (int s = 0; s < card_c; ++s)
                if (!vec[s].empty() && !pz[s]) {
                    r[s] = g.F();
                    g.line("mul.f32 " + r[s] + ", " + vec[s] + ", " + pi[s] + ";");
                }
            r = descend(r, 0);
        } else {
            const int v = down[0];
            r.assign(m.nodes[v].card, std::string());
            if (!pz[i])
                for (int t = 0; t < m.nodes[v].card; ++t) {
                    const float T = cpt_at(m, v, t, i);
                    if (T == 0.f) continue;
                    acc(r[t], pi[i], T);
                    scale(r[t], u[v][t]);
                }
            r = descend(r, 1);
        }
        for (int j = 0; j < m.nodes[Y].card; ++j) {
            const long long idx = X == a ? (long long)i * cb + j : (long long)j * cb + i;
            g.line("@%pvalid st.global.f32 [%rtmp" + (idx ? "+" + I(4 * idx) : std::string()) + "], " + (r[j].empty() ? zero : r[j]) + ";");
        }
    }
    JointBody jb;
    jb.n_fma = g.n_fma;
    for (size_t pos = 0; pos < g.out.size();) {
        size_t e = g.out.find('\n', pos);
        if (e == std::string::npos) e = g.out.size();
        size_t k = g.out.find_first_not_of(' ', pos);
        if (k < e && g.out[k] == '@') k = g.out.find(' ', k) + 1;
        auto starts = [&](const char* op) { return g.out.compare(k, std::strlen(op), op) == 0; };
        if (k < e && (starts("mul.f32") || starts("fma.rn.f32") || starts("add.f32"))) ++jb.pipe;
        if (k < e && starts("st.global")) ++jb.cost;
        pos = e + 1;
    }
    jb.cost += jb.pipe;
    for (size_t k = 0; k < px.size(); ++k) jb.path += (k ? " -> " : "") + I(px[k]);
    jb.path += "  |  ";
    for (size_t k = d; k < py.size(); ++k) jb.path += (k > d ? " -> " : "") + I(py[k]);
    return jb;
}

}  // namespace

// Thread count / occupancy target of the generated kernels.  Register need grows with the widest
// (node, parent) pair of domains on a root-to-leaf path.  Measured on B200 (profiles/r1_spec_v2_sweep.txt):
// small trees like 256-thread CTAs with <= 85 registers; DMV-sized ones want all 255 registers and no
// spills; beyond that three resident CTAs with a few spilled values beat two without.
void bc_spec_geometry(const bc_model& m, int* threads, int* min_blocks) {
    int widest = 0;
    for (int v = 1; v < m.n; ++v) widest = std::max(widest, m.nodes[v].card + m.nodes[v].card_pa);
    if (widest <= 40) { *threads = 256; *min_blocks = 3; }
    else if (widest <= 110) { *threads = 128; *min_blocks = 2; }
    else { *threads = 128; *min_blocks = 3; }
    const int t = env_int("BC_SPEC_THREADS", 0), b = env_int("BC_SPEC_MIN_BLOCKS", 0);
    if (t >= 32 && t <= 1024 && t % 32 == 0) *threads = t;
    if (b >= 1 && b <= 16) *min_blocks = b;
}

std::string bc_spec_generate(const bc_model& m) {
    int threads, min_blocks;
    bc_spec_geometry(m, &threads, &min_blocks);
    long long f1 = 0, f2 = 0;
    std::string k1 = gen_kernel(m, false, threads, min_blocks, &f1);
    std::string k2 = gen_kernel(m, true, threads, min_blocks, &f2);
    std::string s;
    s += "//\n// Generated by bayescard_b200 spec_codegen (version " + I(BC_CODEGEN_VERSION) + ") -- do not edit.\n";
    s += "// nodes: " + I(m.n) + "  dense flop/query: " + I(m.flops_dense) + "  executed flop/query: " + I(2 * f1) + "\n";
    s += "// BC_SPEC_THREADS=" + I(threads) + " BC_SPEC_MIN_BLOCKS=" + I(min_blocks) + " BC_SPEC_FFMA=" + I(f1) + "\n//\n";
    s += ".version 8.7\n.target sm_100a\n.address_size 64\n\n";
    // geometry travels with the image: {threads per CTA, queries per thread and trip, codegen version, 0}
    s += ".visible .global .align 4 .u32 bc_spec_meta[4] = {" + I(threads) + ", 1, " + I(BC_CODEGEN_VERSION) + ", 0};\n\n";
    s += k1;
    s += k2;
    return s;
}

uint64_t bc_spec_hash_of(const bc_model& m) {
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](const void* p, size_t n) {
        const unsigned char* b = static_cast<const unsigned char*>(p);
        for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
    };
    const int ver = BC_CODEGEN_VERSION;
    mix(&ver, sizeof(ver));
    const int knobs[4] = {env_int("BC_SPEC_SYNC_EVERY", 0), env_int("BC_SPEC_THREADS", 0), env_int("BC_SPEC_MIN_BLOCKS", 0),
                          env_int("BC_SPEC_DYNAMIC", 1)};
    if (knobs[0] || knobs[1] || knobs[2] || knobs[3] != 1) mix(knobs, sizeof(knobs));
    mix(&m.n, sizeof(m.n));
    for (const BcNodeRec& r : m.nodes) mix(&r, sizeof(r));
    mix(m.arena.data(), m.arena.size() * sizeof(float));
    mix(m.fan.data(), m.fan.size() * sizeof(float));
    return h;
}

// Module of the marginal kernels of one target: bc_marg_bits / bc_marg_dense, the same loop, geometry and work counter as the
// bc_spec_* entries, out[q][b] for b < card(target).  The header's BC_SPEC_FFMA counts the FMA-pipe instructions that carry a
// CPT entry: one per non-zero entry of the whole tree, as in the spec module.
std::string bc_marginal_generate(const bc_model& m, int target) {
    int threads, min_blocks;
    bc_spec_geometry(m, &threads, &min_blocks);
    long long f1 = 0, f2 = 0;
    std::string k1 = gen_marginal_kernel(m, target, false, threads, min_blocks, &f1);
    std::string k2 = gen_marginal_kernel(m, target, true, threads, min_blocks, &f2);
    std::string path;
    for (int v = target; v >= 0; v = m.nodes[v].parent) path = I(v) + (path.empty() ? "" : " -> " + path);
    std::string s;
    s += "//\n// Generated by bayescard_b200 spec_codegen, marginal generator (version " + I(BC_MARGINAL_VERSION) + ", codegen version " +
         I(BC_CODEGEN_VERSION) + ") -- do not edit.\n";
    s += "// nodes: " + I(m.n) + "  target: " + I(target) + "  card: " + I(m.nodes[target].card) + "  path: " + path + "\n";
    s += "// BC_SPEC_THREADS=" + I(threads) + " BC_SPEC_MIN_BLOCKS=" + I(min_blocks) + " BC_SPEC_FFMA=" + I(f1) + "\n//\n";
    s += ".version 8.7\n.target sm_100a\n.address_size 64\n\n";
    // {threads per CTA, results per query (= card of the target), marginal generator version, target}
    s += ".visible .global .align 4 .u32 bc_marg_meta[4] = {" + I(threads) + ", " + I(m.nodes[target].card) + ", " +
         I(BC_MARGINAL_VERSION) + ", " + I(target) + "};\n\n";
    s += k1;
    s += k2;
    return s;
}

uint64_t bc_marginal_hash_of(const bc_model& m, int target) {
    uint64_t h = bc_spec_hash_of(m);
    auto mix = [&](const void* p, size_t n) {
        const unsigned char* b = static_cast<const unsigned char*>(p);
        for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 1099511628211ull; }
    };
    const int tag[2] = {BC_MARGINAL_VERSION, target};
    mix(tag, sizeof(tag));
    return h;
}

// Module of the joint marginal of the ordered pair (a, b): bc_joint_bits / bc_joint_dense, the loop, geometry and work counter
// of the bc_spec_* entries, out[q][i][j] (i < card(a), j < card(b)) stored by the body.  The loop node X is whichever of a, b
// gives the BITS entry fewer FMA-pipe plus store instructions (a on a tie); both entries use it.  The header's BC_SPEC_FFMA
// counts the FMA-pipe instructions that carry a CPT entry.  BC_ELIMIT when an entry would hold more than BC_JOINT_MAX_FFMA
// FMA-pipe instructions: the straight line grows with card(X) times the path's CPTs.
int bc_joint_generate(const bc_model& m, int a, int b, std::string* src) {
    int threads, min_blocks;
    bc_spec_geometry(m, &threads, &min_blocks);
    Gen ga(m, false), gb(m, false);
    const JointBody ja = gen_joint_body(m, ga, a, b, a, false), jb = gen_joint_body(m, gb, a, b, b, false);
    const bool pick_b = jb.cost < ja.cost;
    Gen& g1 = pick_b ? gb : ga;
    const JointBody& j1 = pick_b ? jb : ja;
    const int X = pick_b ? b : a;
    long long pipe = j1.pipe;
    Gen g2(m, true);
    if (pipe <= BC_JOINT_MAX_FFMA) pipe = std::max(pipe, gen_joint_body(m, g2, a, b, X, true).pipe);
    if (pipe > BC_JOINT_MAX_FFMA) {
        bc_set_error("joint marginal of nodes %d, %d: %lld FMA-pipe instructions per query, above the cap of %d (BC_JOINT_MAX_FFMA)",
                     a, b, pipe, BC_JOINT_MAX_FFMA);
        return BC_ELIMIT;
    }
    const long long row = (long long)m.nodes[a].card * m.nodes[b].card;
    std::string s;
    s += "//\n// Generated by bayescard_b200 spec_codegen, joint marginal generator (version " + I(BC_JOINT_VERSION) + ", codegen version " +
         I(BC_CODEGEN_VERSION) + ") -- do not edit.\n";
    s += "// nodes: " + I(m.n) + "  a: " + I(a) + " (card " + I(m.nodes[a].card) + ")  b: " + I(b) + " (card " + I(m.nodes[b].card) +
         ")  X: " + I(X) + "  paths: " + j1.path + "\n";
    s += "// BC_SPEC_THREADS=" + I(threads) + " BC_SPEC_MIN_BLOCKS=" + I(min_blocks) + " BC_SPEC_FFMA=" + I(j1.n_fma) +
         " FMA-pipe=" + I(j1.pipe) + "\n//\n";
    s += ".version 8.7\n.target sm_100a\n.address_size 64\n\n";
    // {threads per CTA, a, b, joint generator version}
    s += ".visible .global .align 4 .u32 bc_joint_meta[4] = {" + I(threads) + ", " + I(a) + ", " + I(b) + ", " + I(BC_JOINT_VERSION) + "};\n\n";
    s += gen_entry(m, g1, "bc_joint_bits", false, threads, min_blocks, {}, row);
    s += gen_entry(m, g2, "bc_joint_dense", true, threads, min_blocks, {}, row);
    src->swap(s);
    return BC_OK;
}

uint64_t bc_joint_hash_of(const bc_model& m, int a, int b) {
    uint64_t h = bc_spec_hash_of(m);
    auto mix = [&](const void* p, size_t n) {
        const unsigned char* c = static_cast<const unsigned char*>(p);
        for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; }
    };
    const int tag[3] = {BC_JOINT_VERSION, a, b};
    mix(tag, sizeof(tag));
    return h;
}
