// Jagged PCS on the device: commit of a round of chip tables and the evaluation proof
// (Hadamard sumcheck of the dense trace against the jagged "little polynomial", the branching-program
// evaluation sumcheck, then the stacked/BaseFold proof of pcs.cu).
// Reference behaviour: slop/crates/jagged/src/prover.rs:106-328, hadamard.rs:93-151, poly.rs:136-296,384-470,
// jagged_eval/{sumcheck_poly.rs,sumcheck_sum_as_poly.rs,eval_sumcheck_prover.rs}; the GPU twins it replaces:
// sp1-gpu/crates/{jagged_sumcheck,jagged_assist} + sys/lib/{jagged_sumcheck,jagged_assist}/*.cu.
// HOW (results identical): the dense buffers of all rounds form one virtual long vector (no restacking copy);
// each sumcheck round after the first runs as ONE fused kernel (fix the previous variable + accumulate the next
// round's sums) so the folded vectors are written once and read once; the branching-program sumcheck evaluates all
// (column, node) pairs of a round in one launch.
#include "sumcheck.cuh"
#include <algorithm>
#include <memory>
#include <vector>

#include "pcs.cuh"

namespace {

using kb::Ext;
using hf::E4;

// ---- host sponge (PaddingFreeSponge) for the table-shape hash; a few dozen words ----------------------------------
void host_hash(const std::vector<uint32_t>& w, uint32_t* out8) {
    uint32_t st[16] = {0};
    size_t i = 0;
    while (i < w.size()) {
        size_t k = std::min<size_t>(8, w.size() - i);
        for (size_t j = 0; j < k; j++) st[j] = w[i + j];
        host_poseidon2_permute(st);
        i += k;
    }
    for (int j = 0; j < 8; j++) out8[j] = st[j];
}
void host_compress(const uint32_t* l, const uint32_t* r, uint32_t* out8) {
    uint32_t st[16];
    for (int j = 0; j < 8; j++) { st[j] = l[j]; st[8 + j] = r[j]; }
    host_poseidon2_permute(st);
    for (int j = 0; j < 8; j++) out8[j] = st[j];
}

// jagged little polynomial: ext[i] = col_eq[c(i)] * row_eq[i - prefix[c(i)]] for i < prefix[ncols], else 0.
// c(i) = the last column with prefix[c] <= i (zero-height columns share a prefix value: the last one has the non-empty range).
// start[i >> JP_SHIFT] (built on the host from the same prefix sums) is a column at or before c(i), so the search is a short
// forward walk instead of a binary search per element.
constexpr int JP_SHIFT = 12;
__global__ void __launch_bounds__(256) jagged_poly_kernel(const uint64_t* __restrict__ prefix, uint32_t ncols, const uint32_t* __restrict__ start,
                                                          const uint32_t* __restrict__ col_eq, const uint32_t* __restrict__ row_eq, uint64_t N,
                                                          uint32_t* __restrict__ ext) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    Ext v = kb::ext_zero();
    if (i < prefix[ncols]) {
        uint32_t lo = start[i >> JP_SHIFT];
        while (lo + 1 < ncols && prefix[lo + 1] <= i) lo++;
        v = kb::ext_mul(kb::ext_load(col_eq + 4 * lo), kb::ext_load(row_eq + 4 * (i - prefix[lo])));
    }
    kb::ext_store(ext + 4 * i, v);
}

struct SegTable {  // the virtual long base vector = concatenation of the rounds' dense buffers, then zeros
    const uint32_t* ptr[8];
    uint64_t end[8];
    int n;
};
__device__ __forceinline__ uint32_t seg_load(const SegTable& t, uint64_t i) {
    uint64_t start = 0;
#pragma unroll 1
    for (int s = 0; s < t.n; s++) { if (i < t.end[s]) return __ldg(t.ptr[s] + (i - start)); start = t.end[s]; }
    return 0;
}

// round 0: sum_j ext[2j]*base[2j]  and  sum_j (ext[2j]+ext[2j+1]) * (base[2j]+base[2j+1])   (base in F)
__global__ void __launch_bounds__(256) hadamard_sum0_kernel(SegTable base, const uint32_t* __restrict__ ext, uint64_t npairs,
                                                            uint32_t* __restrict__ partial, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < npairs; j += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t b0 = seg_load(base, 2 * j), b1 = seg_load(base, 2 * j + 1);
        Ext e0 = kb::ext_load(ext + 8 * j), e1 = kb::ext_load(ext + 8 * j + 4);
        s0 = kb::ext_add(s0, kb::ext_mul_base(e0, b0));
        sh = kb::ext_add(sh, kb::ext_mul_base(kb::ext_add(e0, e1), kb::add(b0, b1)));
    }
    block_post_sums<2>({s0, sh}, partial, mail);
}

// fix the last variable of round 0 (base F -> EF) and accumulate round-1 sums
__global__ void __launch_bounds__(256) hadamard_fold0_kernel(SegTable base, const uint32_t* __restrict__ ext, uint64_t nout_pairs, Ext alpha,
                                                             uint32_t* __restrict__ base_out, uint32_t* __restrict__ ext_out,
                                                             uint32_t* __restrict__ partial, uint64_t nout, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nout_pairs; j += (uint64_t)gridDim.x * blockDim.x) {
        Ext nb[2], ne[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            uint64_t o = 2 * j + h;  // output index; inputs 2o, 2o+1
            if (o < nout) {
                uint32_t b0 = seg_load(base, 2 * o), b1 = seg_load(base, 2 * o + 1);
                Ext e0 = kb::ext_load(ext + 8 * o), e1 = kb::ext_load(ext + 8 * o + 4);
                nb[h] = kb::ext_add(kb::ext_from_base(b0), kb::ext_mul_base(alpha, kb::sub(b1, b0)));
                ne[h] = kb::ext_add(e0, kb::ext_mul(alpha, kb::ext_sub(e1, e0)));
                kb::ext_store(base_out + 4 * o, nb[h]);
                kb::ext_store(ext_out + 4 * o, ne[h]);
            } else { nb[h] = kb::ext_zero(); ne[h] = kb::ext_zero(); }
        }
        s0 = kb::ext_add(s0, kb::ext_mul(ne[0], nb[0]));
        sh = kb::ext_add(sh, kb::ext_mul(kb::ext_add(ne[0], ne[1]), kb::ext_add(nb[0], nb[1])));
    }
    block_post_sums<2>({s0, sh}, partial, mail);
}

// ---- round 0 without the materialised little polynomial ("factored" path) -------------------------------------------------------
// ext[i] = col_eq[c(i)] * row_eq[i - prefix[c]] is a product of two small tables (2^11 and 2^22 entries), so when every column
// start is even (all heights even: the reference pads heights to multiples of 32, crates/hypercube/src/util.rs:57) a pair (2j, 2j+1)
// lies in one column and
//   sum_j ext[2j] b[2j]                       = sum_c col_eq[c] * sum_{j in c} row_eq[r_j] b[2j]
//   sum_j (ext[2j]+ext[2j+1]) (b[2j]+b[2j+1]) = sum_c col_eq[c] * sum_{j in c} (row_eq[r_j]+row_eq[r_j+1]) (b[2j]+b[2j+1])
// with base-field b: the inner sums cost EF x F products only and the 2^log_m-entry EF polynomial (4.3 GB for a 2^22-cycle shard) is
// never written or read.  Every warp walks a contiguous span of pairs, lanes keep running sums for their current column and
// multiply by col_eq[c] only when the column changes.  The fold by alpha keeps the product form:
//   ext'[o] = col_eq[c(2o)] * row_eq'[(2o - prefix[c]) / 2],   row_eq'[k] = row_eq[2k] + alpha (row_eq[2k+1] - row_eq[2k]).
__device__ __forceinline__ uint32_t jp_column(const uint64_t* __restrict__ prefix, uint32_t ncols, uint32_t c, uint64_t i) {
    while (c + 1 < ncols && prefix[c + 1] <= i) c++;
    return c;
}
__global__ void __launch_bounds__(256) hadamard_sum0_fused_kernel(SegTable base, const uint64_t* __restrict__ prefix, uint32_t ncols,
                                                                  const uint32_t* __restrict__ start, const uint32_t* __restrict__ col_eq,
                                                                  const uint32_t* __restrict__ row_eq, uint64_t npairs_real, uint64_t span,
                                                                  uint32_t* __restrict__ partial, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero();
    Ext t0 = kb::ext_zero(), th = kb::ext_zero();
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t j_begin = warp * span, j_end = min(j_begin + span, npairs_real);
    uint32_t c = 0xffffffffu;
    for (uint64_t j = j_begin + lane; j < j_end; j += 32) {
        const uint64_t i = 2 * j;
        const uint32_t cn = jp_column(prefix, ncols, c == 0xffffffffu ? start[i >> JP_SHIFT] : c, i);
        if (cn != c) {
            if (c != 0xffffffffu) {
                const Ext ce = kb::ext_load(col_eq + 4 * c);
                s0 = kb::ext_add(s0, kb::ext_mul(ce, t0)); sh = kb::ext_add(sh, kb::ext_mul(ce, th));
                t0 = kb::ext_zero(); th = kb::ext_zero();
            }
            c = cn;
        }
        const uint32_t b0 = seg_load(base, i), b1 = seg_load(base, i + 1);
        const uint64_t r = i - prefix[c];
        const Ext e0 = kb::ext_load(row_eq + 4 * r), e1 = kb::ext_load(row_eq + 4 * r + 4);
        t0 = kb::ext_add(t0, kb::ext_mul_base(e0, b0));
        th = kb::ext_add(th, kb::ext_mul_base(kb::ext_add(e0, e1), kb::add(b0, b1)));
    }
    if (c != 0xffffffffu) {
        const Ext ce = kb::ext_load(col_eq + 4 * c);
        s0 = kb::ext_add(s0, kb::ext_mul(ce, t0)); sh = kb::ext_add(sh, kb::ext_mul(ce, th));
    }
    block_post_sums<2>({s0, sh}, partial, mail);
}
// fix the last variable of round 0 in product form and accumulate round-1 sums; roweq2 = row_eq folded by alpha (fix_last_kernel)
__global__ void __launch_bounds__(256) hadamard_fold0_fused_kernel(SegTable base, const uint64_t* __restrict__ prefix, uint32_t ncols,
                                                                   const uint32_t* __restrict__ start, const uint32_t* __restrict__ col_eq,
                                                                   const uint32_t* __restrict__ roweq2, uint64_t area, uint64_t nout_pairs, Ext alpha,
                                                                   uint32_t* __restrict__ base_out, uint32_t* __restrict__ ext_out,
                                                                   uint32_t* __restrict__ partial, uint64_t nout, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nout_pairs; j += (uint64_t)gridDim.x * blockDim.x) {
        Ext nb[2], ne[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint64_t o = 2 * j + h;  // output index; inputs 2o, 2o+1
            if (o < nout) {
                const uint64_t i = 2 * o;
                const uint32_t b0 = seg_load(base, i), b1 = seg_load(base, i + 1);
                nb[h] = kb::ext_add(kb::ext_from_base(b0), kb::ext_mul_base(alpha, kb::sub(b1, b0)));
                if (i < area) {
                    const uint32_t c = jp_column(prefix, ncols, start[i >> JP_SHIFT], i);
                    ne[h] = kb::ext_mul(kb::ext_load(col_eq + 4 * c), kb::ext_load(roweq2 + 4 * ((i - prefix[c]) >> 1)));
                } else ne[h] = kb::ext_zero();
                kb::ext_store(base_out + 4 * o, nb[h]);
                kb::ext_store(ext_out + 4 * o, ne[h]);
            } else { nb[h] = kb::ext_zero(); ne[h] = kb::ext_zero(); }
        }
        s0 = kb::ext_add(s0, kb::ext_mul(ne[0], nb[0]));
        sh = kb::ext_add(sh, kb::ext_mul(kb::ext_add(ne[0], ne[1]), kb::ext_add(nb[0], nb[1])));
    }
    block_post_sums<2>({s0, sh}, partial, mail);
}

// rounds >= 1: fix the last variable (EF -> EF) and accumulate the next round's sums
__global__ void __launch_bounds__(256) hadamard_fold_kernel(const uint32_t* __restrict__ base, const uint32_t* __restrict__ ext,
                                                            uint64_t nout_pairs, Ext alpha, uint32_t* __restrict__ base_out,
                                                            uint32_t* __restrict__ ext_out, uint32_t* __restrict__ partial, uint64_t nout, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < nout_pairs; j += (uint64_t)gridDim.x * blockDim.x) {
        Ext nb[2], ne[2];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            uint64_t o = 2 * j + h;
            if (o < nout) {
                Ext b0 = kb::ext_load(base + 8 * o), b1 = kb::ext_load(base + 8 * o + 4);
                Ext e0 = kb::ext_load(ext + 8 * o), e1 = kb::ext_load(ext + 8 * o + 4);
                nb[h] = kb::ext_add(b0, kb::ext_mul(alpha, kb::ext_sub(b1, b0)));
                ne[h] = kb::ext_add(e0, kb::ext_mul(alpha, kb::ext_sub(e1, e0)));
                kb::ext_store(base_out + 4 * o, nb[h]);
                kb::ext_store(ext_out + 4 * o, ne[h]);
                if (nout == 1) kb::ext_store(partial + 8, nb[h]);  // last round: the dense component evaluation rides along
            } else { nb[h] = kb::ext_zero(); ne[h] = kb::ext_zero(); }
        }
        s0 = kb::ext_add(s0, kb::ext_mul(ne[0], nb[0]));
        sh = kb::ext_add(sh, kb::ext_mul(kb::ext_add(ne[0], ne[1]), kb::ext_add(nb[0], nb[1])));
    }
    block_post_sums<2>({s0, sh}, partial, mail);
}

// ---- branching program (slop/crates/jagged/src/poly.rs:136-175, 384-470) ---------------------------------------
// state index = carry + 2 * comparison_so_far ; returns -1 on failure
__device__ __forceinline__ int bp_transition(int row_bit, int index_bit, int cur_bit, int next_bit, int state) {
    int carry = state & 1, cmp = state >> 1;
    int new_cmp = (index_bit == next_bit) ? cmp : next_bit;
    int s = row_bit + carry + cur_bit;
    if (index_bit != (s & 1)) return -1;
    return (s >> 1) + 2 * new_cmp;
}

// ---- prefix / suffix form of the same evaluation -----------------------------------------------------------------
// The evaluation is  e0^T M_0 M_1 ... M_hl init  with one 4x4 transfer matrix per layer, M_l = M(cur_l, next_l).  In sumcheck
// round r only ONE layer holds the free variable: layers above it still see the column's boolean prefix-sum bits (and, in
// the second half, next-coordinates that were bound earlier and never change again), layers below it see coordinates that
// were bound in earlier rounds.  So per column k:  value = P_k . M_layer(lambda) . T_k[layer + 1]  with
//   T_k[l] = M_l ... M_hl init   (suffix table, one pass per half: bp_suffix_kernel)
//   P_k    = e0^T M_0 ... M_{layer-1}   (prefix row vector, one vector-matrix product per round: bp_update_kernel)
// i.e. two small products per (column, node) and round instead of hl+1 (the reference keeps the same prefix/suffix states,
// sp1-gpu/crates/sys/lib/jagged_assist).  Every product is exact field arithmetic, so the round polynomials are unchanged.
struct BpMat { Ext ri[4], cc[4]; };
__device__ __forceinline__ void bp_layer_coeffs(const uint32_t* __restrict__ ri_eq, uint32_t layer, uint32_t hl, const Ext& cur, const Ext& nxt, BpMat& m) {
    if (layer < hl) {
        const uint32_t* e = ri_eq + (size_t)layer * 16;
        m.ri[0] = kb::ext_load(e); m.ri[1] = kb::ext_load(e + 4); m.ri[2] = kb::ext_load(e + 8); m.ri[3] = kb::ext_load(e + 12);
    } else { m.ri[0] = kb::ext_one(); m.ri[1] = m.ri[2] = m.ri[3] = kb::ext_zero(); }
    const Ext cn = kb::ext_mul(cur, nxt);
    m.cc[3] = cn; m.cc[2] = kb::ext_sub(cur, cn); m.cc[1] = kb::ext_sub(nxt, cn);
    m.cc[0] = kb::ext_sub(kb::ext_sub(kb::ext_one(), cur), m.cc[1]);
}
// out = M res   (column form)
__device__ __forceinline__ void bp_apply(const BpMat& m, const Ext res[4], Ext out[4]) {
#pragma unroll
    for (int st = 0; st < 4; st++) {
        Ext acc = kb::ext_zero();
#pragma unroll
        for (int a = 0; a < 4; a++) {
            Ext inner = kb::ext_zero();
            bool any = false;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                int o = bp_transition(a >> 1, a & 1, c >> 1, c & 1, st);
                if (o >= 0) { inner = kb::ext_add(inner, kb::ext_mul(m.cc[c], res[o])); any = true; }
            }
            if (any) acc = kb::ext_add(acc, kb::ext_mul(m.ri[a], inner));
        }
        out[st] = acc;
    }
}
// out = P M   (row form)
__device__ __forceinline__ void bp_apply_row(const BpMat& m, const Ext P[4], Ext out[4]) {
    Ext o4[4] = {kb::ext_zero(), kb::ext_zero(), kb::ext_zero(), kb::ext_zero()};
#pragma unroll
    for (int st = 0; st < 4; st++)
#pragma unroll
        for (int a = 0; a < 4; a++) {
            const Ext q = kb::ext_mul(P[st], m.ri[a]);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                int o = bp_transition(a >> 1, a & 1, c >> 1, c & 1, st);
                if (o >= 0) o4[o] = kb::ext_add(o4[o], kb::ext_mul(q, m.cc[c]));
            }
        }
#pragma unroll
    for (int i = 0; i < 4; i++) out[i] = o4[i];
}
__device__ __forceinline__ Ext bp_bit(const uint8_t* b, uint32_t pos) { return b[pos] ? kb::ext_one() : kb::ext_zero(); }

// T[(l * nk + k) * 4 + s], l = hl+1 .. 0.  second_half: next-coordinates are the bound values rho_by_pos[dim-1-l]
__global__ void __launch_bounds__(128) bp_suffix_kernel(const uint8_t* __restrict__ bits, uint32_t nk, uint32_t dim, int second_half,
                                                        const uint32_t* __restrict__ rho_by_pos, const uint32_t* __restrict__ ri_eq,
                                                        uint32_t* __restrict__ T) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nk) return;
    const uint32_t hl = dim / 2;
    const uint8_t* b = bits + (size_t)k * dim;
    Ext res[4] = {kb::ext_zero(), kb::ext_zero(), kb::ext_one(), kb::ext_zero()};
    for (int s = 0; s < 4; s++) kb::ext_store(T + (((size_t)(hl + 1) * nk + k) * 4 + s) * 4, res[s]);
    for (int layer = (int)hl; layer >= 0; layer--) {
        Ext cur = kb::ext_zero(), nxt = kb::ext_zero();
        if ((uint32_t)layer < hl) {
            cur = bp_bit(b, hl - 1 - layer);
            nxt = second_half ? kb::ext_load(rho_by_pos + 4 * (dim - 1 - layer)) : bp_bit(b, dim - 1 - layer);
        }
        BpMat m;
        bp_layer_coeffs(ri_eq, (uint32_t)layer, hl, cur, nxt, m);
        Ext nres[4];
        bp_apply(m, res, nres);
        for (int s = 0; s < 4; s++) { res[s] = nres[s]; kb::ext_store(T + (((size_t)layer * nk + k) * 4 + s) * 4, res[s]); }
    }
}
// round r: thread (k, node) -> zc[k] * inter[k] * eq(lambda, bit) * P_k . M_layer(lambda_node) . T_k[layer+1]
__global__ void __launch_bounds__(128) bp_round2_kernel(const uint8_t* __restrict__ bits, uint32_t nk, uint32_t dim, uint32_t round,
                                                        const uint32_t* __restrict__ rho_by_pos, const uint32_t* __restrict__ ri_eq,
                                                        const uint32_t* __restrict__ zc, const uint32_t* __restrict__ inter,
                                                        const uint32_t* __restrict__ P, const uint32_t* __restrict__ T, Ext half,
                                                        uint32_t* __restrict__ partial, Mail mail) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    Ext v = kb::ext_zero();
    const uint32_t k = t >> 1, node = t & 1;
    const uint32_t hl = dim / 2, split = dim - round - 1;
    if (k < nk) {
        const uint8_t* b = bits + (size_t)k * dim;
        const bool second = round >= hl;
        const uint32_t layer = second ? round - hl : round;
        const Ext lam = node ? half : kb::ext_zero();
        const Ext cur = second ? lam : bp_bit(b, hl - 1 - layer);
        const Ext nxt = second ? kb::ext_load(rho_by_pos + 4 * (dim - 1 - layer)) : lam;
        BpMat m;
        bp_layer_coeffs(ri_eq, layer, hl, cur, nxt, m);
        Ext res[4], w[4];
        for (int s = 0; s < 4; s++) res[s] = kb::ext_load(T + (((size_t)(layer + 1) * nk + k) * 4 + s) * 4);
        bp_apply(m, res, w);
        Ext val = kb::ext_zero();
        if (round == 0 || round == hl) val = w[0];  // P_k = e0^T at the start of either half (bp_update_kernel resets it after this round)
        else
            for (int s = 0; s < 4; s++) val = kb::ext_add(val, kb::ext_mul(kb::ext_load(P + ((size_t)k * 4 + s) * 4), w[s]));
        const Ext eqv = node ? half : (b[split] ? kb::ext_zero() : kb::ext_one());
        v = kb::ext_mul(kb::ext_mul(kb::ext_load(zc + 4 * k), val), kb::ext_mul(kb::ext_load(inter + 4 * k), eqv));
    }
    // per block: the sum at node 0 (y_0), then at node 1 (y_half)
    block_post_sums<2>({node ? kb::ext_zero() : v, node ? v : kb::ext_zero()}, partial, mail);
}
// after round r's challenge: bind position split = dim-1-r: rho_by_pos, inter[k] *= eq(alpha, bit), P_k <- P_k M_layer(bound)
// (at the switch to the second half P_k restarts at e0^T: the caller rebuilds T with the bound next-coordinates first)
__global__ void __launch_bounds__(128) bp_update_kernel(const uint8_t* __restrict__ bits, uint32_t nk, uint32_t dim, uint32_t round, Ext alpha,
                                                        uint32_t* __restrict__ rho_by_pos, const uint32_t* __restrict__ ri_eq,
                                                        uint32_t* __restrict__ inter, uint32_t* __restrict__ P) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t hl = dim / 2, split = dim - round - 1;
    if (k == 0) kb::ext_store(rho_by_pos + 4 * split, alpha);
    if (k >= nk) return;
    const uint8_t* b = bits + (size_t)k * dim;
    const Ext f = b[split] ? alpha : kb::ext_sub(kb::ext_one(), alpha);
    kb::ext_store(inter + 4 * k, kb::ext_mul(kb::ext_load(inter + 4 * k), f));
    const bool second = round >= hl;
    const uint32_t layer = second ? round - hl : round;
    Ext Pk[4], out[4];
    for (int s = 0; s < 4; s++) Pk[s] = kb::ext_load(P + ((size_t)k * 4 + s) * 4);
    if (round == hl) { Pk[0] = kb::ext_one(); Pk[1] = Pk[2] = Pk[3] = kb::ext_zero(); }
    const Ext cur = second ? alpha : bp_bit(b, hl - 1 - layer);
    // second half: the next-coordinate of this layer was bound in round `layer` (written before this kernel ran)
    const Ext nxt = second ? kb::ext_load(rho_by_pos + 4 * (dim - 1 - layer)) : alpha;
    BpMat m;
    bp_layer_coeffs(ri_eq, layer, hl, cur, nxt, m);
    bp_apply_row(m, Pk, out);
    for (int s = 0; s < 4; s++) kb::ext_store(P + ((size_t)k * 4 + s) * 4, out[s]);
}

// p(x) through (0, y0), (1, y1), (1/2, yh): coefficients c0, c1, c2
inline void interp_0_1_half(const E4& y0, const E4& y1, const E4& yh, E4 c[3]) {
    const uint32_t two = hf::to_monty(2), three = hf::to_monty(3), four = hf::to_monty(4);
    c[0] = y0;
    c[1] = yh * four - y0 * three - y1;
    c[2] = (y1 + y0) * two - yh * four;
}
inline E4 eval3(const E4 c[3], const E4& x) { return (c[2] * x + c[1]) * x + c[0]; }

sp1b200_err sum_partials(sp1b200_ctx* ctx, const uint32_t* d_partial, unsigned nblk, E4 (&out)[2]) {
    std::vector<uint32_t> h((size_t)nblk * 8);
    SP1_CUDA(cudaMemcpyAsync(h.data(), d_partial, h.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    SP1_CUDA(cudaStreamSynchronize(ctx->stream));
    out[0] = E4(); out[1] = E4();
    for (unsigned k = 0; k < nblk; k++) { out[0] = out[0] + E4::load(&h[8 * k]); out[1] = out[1] + E4::load(&h[8 * k + 4]); }
    return nullptr;
}

}  // namespace

extern "C" {

// Jagged commit of one round of chip tables (slop/crates/jagged/src/prover.rs:106-160).
// dense_any: the tables' real cells back to back, each table column-major [cols x rows] (tables with 0 rows
// contribute nothing), host or device; the library keeps its own zero-padded device copy.
sp1b200_err sp1b200_jagged_commit(sp1b200_ctx* ctx, const uint32_t* dense_any, uint32_t n_tables, const uint64_t* rows, const uint64_t* cols,
                                  int keep_codeword, uint32_t* h_commit8, sp1b200_jagged_round** out) { SP1_DEVICE_GUARD(ctx);
    const uint32_t ls = ctx->params.log_stacking_height, mlr = ctx->params.max_log_row_count;
    auto r = std::make_unique<sp1b200_jagged_round>();
    uint64_t area = 0;
    for (uint32_t t = 0; t < n_tables; t++) {
        if (rows[t] > ((uint64_t)1 << mlr)) return sp1b200_set_error("jagged_commit: table %u has %llu rows > 2^%u", t, (unsigned long long)rows[t], mlr);
        r->row_counts.push_back(rows[t]); r->col_counts.push_back(cols[t]); area += rows[t] * cols[t];
    }
    const uint64_t S = (uint64_t)1 << ls, R = (uint64_t)1 << mlr;
    const uint64_t padded = std::max(((area + S - 1) / S) * S, S);
    const uint64_t added = padded - area;
    r->area = area; r->padded_area = padded;
    SP1_CUDA(cudaMallocFromPoolAsync((void**)&r->d_dense, padded * 4, ctx->pool, ctx->stream));
    const int up_slot = sp1b200_upload_acquire(ctx, dense_any);  // dense_any may be an upload slot still being filled
    cudaError_t ce = area ? cudaMemcpyAsync(r->d_dense, dense_any, area * 4, cudaMemcpyDefault, ctx->stream) : cudaSuccess;
    sp1b200_upload_release(ctx, up_slot);                        // the slot is free once this copy has run
    if (ce == cudaSuccess && added) ce = cudaMemsetAsync(r->d_dense + area, 0, added * 4, ctx->stream);
    sp1b200_err e = ce == cudaSuccess ? sp1b200_stacked_commit(ctx, r->d_dense, padded / S, keep_codeword, r->original_commit, &r->stacked)
                                      : sp1b200_set_error("jagged_commit: copying the dense trace: %s", cudaGetErrorString(ce));
    if (e) { cudaFreeAsync(r->d_dense, ctx->stream); r->d_dense = nullptr; return e; }
    const uint64_t added_cols = std::max<uint64_t>((added + R - 1) / R, 1);
    r->row_counts.push_back(R); r->row_counts.push_back(added - (added_cols - 1) * R);
    r->col_counts.push_back(added_cols - 1); r->col_counts.push_back(1);
    r->padding_cols = added_cols;
    std::vector<uint32_t> meta{hf::to_monty(r->row_counts.size())};
    for (uint64_t x : r->row_counts) meta.push_back(hf::to_monty(x));
    for (uint64_t x : r->col_counts) meta.push_back(hf::to_monty(x));
    uint32_t hsh[8];
    host_hash(meta, hsh);
    host_compress(r->original_commit, hsh, r->commit);
    if (h_commit8) memcpy(h_commit8, r->commit, 32);
    *out = r.release();
    return nullptr;
}

void sp1b200_jagged_round_free(sp1b200_ctx* ctx, sp1b200_jagged_round* r) { SP1_DEVICE_GUARD(ctx);
    if (!r) return;
    sp1b200_commit_free(ctx, r->stacked);
    if (r->d_dense) cudaFreeAsync(r->d_dense, ctx->stream);
    delete r;
}

// Per-column evaluations of every table column of the round at z_row (zero-padded to 2^max_log_row_count rows):
// the claims zerocheck hands to the PCS (crates/hypercube/src/prover/shard.rs:736-767).  h_out: sum(cols) ext elements.
sp1b200_err sp1b200_jagged_column_claims(sp1b200_ctx* ctx, const sp1b200_jagged_round* r, const uint32_t* h_z_row, uint32_t* h_out) { SP1_DEVICE_GUARD(ctx);
    const uint32_t mlr = ctx->params.max_log_row_count;
    DevFree mem(ctx);
    uint32_t *d_z, *d_eq, *d_out;
    // the real tables (the two padding entries at the end excluded), back to back in d_dense
    std::vector<ColTable> tables;
    uint64_t off = 0;
    size_t nc = 0;
    for (size_t t = 0; t + 2 < r->row_counts.size(); t++) {
        tables.push_back(ColTable{r->d_dense + off, r->row_counts[t], (uint32_t)r->col_counts[t], (uint32_t)nc});
        off += r->row_counts[t] * r->col_counts[t];
        nc += r->col_counts[t];
    }
    if (!nc) return nullptr;
    SP1_TRY(mem.alloc((void**)&d_z, mlr * 16));
    SP1_TRY(mem.alloc((void**)&d_eq, ((size_t)16) << mlr));
    SP1_TRY(mem.alloc((void**)&d_out, nc * 16));
    SP1_CUDA(cudaMemcpyAsync(d_z, h_z_row, mlr * 16, cudaMemcpyHostToDevice, ctx->stream));
    SP1_LAUNCH(ctx, eq_table_kernel, blocks_for((uint64_t)1 << mlr), 256, 0, d_z, (int)mlr, d_eq);
    SP1_TRY(column_evals(ctx, mem, tables, d_eq, nc, d_out));
    SP1_CUDA(cudaMemcpyAsync(h_out, d_out, nc * 16, cudaMemcpyDeviceToHost, ctx->stream));
    SP1_CUDA(cudaStreamSynchronize(ctx->stream));
    return nullptr;
}

// JaggedProver::prove_trusted_evaluations (slop/crates/jagged/src/prover.rs:162-328).
// h_claims: for each round, the evaluations at z_row of that round's table columns (ext each), back to back.
// Proof words: stacked proof | sumcheck {n_polys, per poly {n_coeffs, coeffs}, claimed_sum, point, eval} |
// jagged_eval (same layout) | per round {n_tables, (rows, cols)...} | original commitments | expected_eval |
// max_log_row_count | log_m        (field order of JaggedPcsProof, slop/crates/jagged/src/verifier.rs:17-27)
sp1b200_err sp1b200_jagged_prove(sp1b200_ctx* ctx, sp1b200_jagged_round* const* rounds, uint32_t n_rounds, const uint32_t* h_z_row,
                                 const uint32_t* h_claims, const uint32_t* h_replay, uint32_t* h_chal, uint32_t* h_proof, uint64_t cap,
                                 uint64_t* h_words) { SP1_DEVICE_GUARD(ctx);
    if (!n_rounds || n_rounds > 8) return sp1b200_set_error("jagged_prove: 1..8 rounds supported");
    const uint32_t mlr = ctx->params.max_log_row_count, ls = ctx->params.log_stacking_height;
    cudaStream_t st = ctx->stream;
    DevFree mem(ctx);
    HostChallenger ch;
    SP1_TRY(ch.init(ctx, h_chal));
    PhaseTimer t_all(ctx, "jagged.total");

    // column heights over all rounds (dummy tables included) and prefix sums
    std::vector<uint64_t> heights;
    uint64_t total_cols = 0;
    for (uint32_t r = 0; r < n_rounds; r++)
        for (size_t t = 0; t < rounds[r]->row_counts.size(); t++)
            for (uint64_t c = 0; c < rounds[r]->col_counts[t]; c++) { heights.push_back(rounds[r]->row_counts[t]); total_cols++; }
    std::vector<uint64_t> prefix;
    { uint64_t s = 0; for (uint64_t hgt : heights) { prefix.push_back(s); s += hgt; } prefix.push_back(prefix.back() + heights.back()); }
    const uint32_t lm = hf::log2_ceil(prefix.back());
    if (lm < ls) return sp1b200_set_error("jagged_prove: internal: log_m < log_stacking_height");
    const uint64_t N = (uint64_t)1 << lm;
    const uint32_t ncv = hf::log2_ceil(total_cols);
    std::vector<E4> z_col(ncv), z_row(mlr);
    for (auto& x : z_col) ch.sample_ext(x.c);
    for (uint32_t i = 0; i < mlr; i++) z_row[i] = E4::load(h_z_row + 4 * i);

    // column claims with zeros for the padding columns; sumcheck claim = MLE(column_claims)(z_col)
    std::vector<E4> column_claims;
    {
        size_t k = 0;
        for (uint32_t r = 0; r < n_rounds; r++) {
            uint64_t real = 0;
            for (size_t t = 0; t + 2 < rounds[r]->col_counts.size(); t++) real += rounds[r]->col_counts[t];
            for (uint64_t c = 0; c < real; c++) column_claims.push_back(E4::load(h_claims + 4 * (k++)));
            for (uint64_t c = 0; c < rounds[r]->padding_cols; c++) column_claims.push_back(E4());
        }
    }
    std::vector<E4> col_eq_full = hf::partial_lagrange(z_col);
    E4 claim;
    for (size_t i = 0; i < column_claims.size(); i++) claim = claim + col_eq_full[i] * column_claims[i];

    // device tables: col_eq (over last log2_ceil(ncols) coords of z_col == all of z_col), row_eq, prefix sums
    uint32_t *d_coleq, *d_zrow, *d_roweq, *d_ext, *d_ext2, *d_b, *d_b2, *d_partial;
    uint64_t* d_prefix;
    SP1_TRY(mem.alloc((void**)&d_coleq, col_eq_full.size() * 16));
    SP1_CUDA(cudaMemcpyAsync(d_coleq, col_eq_full.data(), col_eq_full.size() * 16, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_zrow, mlr * 16));
    SP1_CUDA(cudaMemcpyAsync(d_zrow, h_z_row, mlr * 16, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_roweq, ((size_t)16) << mlr));
    SP1_LAUNCH(ctx, eq_table_kernel, blocks_for((uint64_t)1 << mlr), 256, 0, d_zrow, (int)mlr, d_roweq);
    SP1_TRY(mem.alloc((void**)&d_prefix, prefix.size() * 8));
    SP1_CUDA(cudaMemcpyAsync(d_prefix, prefix.data(), prefix.size() * 8, cudaMemcpyHostToDevice, st));
    // start[b] = last column with prefix <= b << JP_SHIFT (two-pointer walk over the blocks of the real area)
    std::vector<uint32_t> jp_start((size_t)((prefix.back() >> JP_SHIFT) + 1));
    {
        uint32_t c = 0;
        for (size_t b = 0; b < jp_start.size(); b++) {
            const uint64_t i0 = (uint64_t)b << JP_SHIFT;
            while (c + 1 < total_cols && prefix[c + 1] <= i0) c++;
            jp_start[b] = c;
        }
    }
    uint32_t* d_jp_start;
    SP1_TRY(mem.alloc((void**)&d_jp_start, jp_start.size() * 4));
    SP1_CUDA(cudaMemcpyAsync(d_jp_start, jp_start.data(), jp_start.size() * 4, cudaMemcpyHostToDevice, st));
    // factored round 0 (no materialised little polynomial) whenever every column starts at an even index
    bool factored = lm >= 2;
    for (uint64_t p : prefix) factored = factored && (p & 1) == 0;
    uint32_t* d_roweq2 = nullptr;
    if (factored) {
        SP1_TRY(mem.alloc((void**)&d_ext, (N / 4 + 1) * 16));          // only from round 2 on
        SP1_TRY(mem.alloc((void**)&d_roweq2, ((size_t)16) << (mlr - 1)));
    } else {
        SP1_TRY(mem.alloc((void**)&d_ext, N * 16));
    }
    SP1_TRY(mem.alloc((void**)&d_ext2, (N / 2) * 16));
    SP1_TRY(mem.alloc((void**)&d_b, (N / 2) * 16));
    SP1_TRY(mem.alloc((void**)&d_b2, (N / 4 + 1) * 16));
    const unsigned MAXB = 148 * 8;
    static_assert(148 * 8 * 8 + 16 <= SP1_MAIL_WORDS, "round partials must fit the mailbox payload");
    d_partial = sp1b200_mail_dev(ctx);  // the round kernels post their block partials straight into the mailbox
    {
        PhaseTimer t(ctx, "jagged.little_poly");
        if (!factored) SP1_LAUNCH(ctx, jagged_poly_kernel, blocks_for(N), 256, 0, d_prefix, (uint32_t)total_cols, d_jp_start, d_coleq, d_roweq, N, d_ext);
        t.stop();
    }
    SegTable seg{};
    seg.n = (int)n_rounds;
    { uint64_t e = 0; for (uint32_t r = 0; r < n_rounds; r++) { seg.ptr[r] = rounds[r]->d_dense; e += rounds[r]->padded_area; seg.end[r] = e; } }

    // ---- Hadamard sumcheck (lambda = 1, t = 1) ---------------------------------------------------------------------
    SumcheckProof sc;
    E4 round_claim = claim;
    PhaseTimer t_sc(ctx, "jagged.sumcheck");
    auto grid_for = [&](uint64_t n) { unsigned g = blocks_for(n); return g > MAXB ? MAXB : (g ? g : 1u); };
    uint32_t *cur_b = nullptr, *cur_e = d_ext, *nxt_b = d_b, *nxt_e = d_ext2;
    unsigned prev_g = 0;
    uint32_t prev_seq = 0;
    for (uint32_t rd = 0; rd < lm; rd++) {
        const uint64_t n = N >> rd;  // current length
        E4 s[2];  // the sum at 0, 4 x the sum at 1/2
        unsigned g;
        if (rd == 0) {
            g = grid_for(n / 2);
            const Mail mail = sp1b200_mail_next(ctx);
            if (factored) {
                // contiguous span of pairs per warp (multiple of 32), over the real area only (beyond it the polynomial is zero)
                const uint64_t pairs_real = prefix.back() / 2, warps = (uint64_t)g * 8;
                const uint64_t span = (((pairs_real + warps - 1) / warps) + 31) / 32 * 32;
                SP1_LAUNCH(ctx, hadamard_sum0_fused_kernel, g, 256, 0, seg, d_prefix, (uint32_t)total_cols, d_jp_start, d_coleq, d_roweq, pairs_real,
                           span ? span : 32, d_partial, mail);
            } else {
                SP1_LAUNCH(ctx, hadamard_sum0_kernel, g, 256, 0, seg, cur_e, n / 2, d_partial, mail);
            }
            SP1_TRY(mail_sums(ctx, mail.seq, g, s));
        } else {
            SP1_TRY(mail_sums(ctx, prev_seq, prev_g, s));  // accumulated by the previous fold launch
        }
        E4 c[3];
        interp_0_1_half(s[0], round_claim - s[0], s[1] * hf::inv(hf::to_monty(4)), c);
        const E4 alpha = sc.round(ch, c, 3);
        round_claim = eval3(c, alpha);
        // fix the variable; the same launch accumulates the next round's sums (unless this was the last round)
        const uint64_t nout = n / 2;
        const Ext da = to_ext(alpha);
        g = grid_for((nout + 1) / 2);
        const Mail mail = sp1b200_mail_next(ctx); prev_seq = mail.seq;
        if (rd == 0) {
            if (factored) {
                SP1_LAUNCH(ctx, fix_last_kernel, blocks_for((uint64_t)1 << (mlr - 1)), 256, 0, d_roweq, (uint64_t)1 << (mlr - 1), da, d_roweq2);
                SP1_LAUNCH(ctx, hadamard_fold0_fused_kernel, g, 256, 0, seg, d_prefix, (uint32_t)total_cols, d_jp_start, d_coleq, d_roweq2, prefix.back(),
                           (nout + 1) / 2, da, nxt_b, nxt_e, d_partial, nout, mail);
            } else {
                SP1_LAUNCH(ctx, hadamard_fold0_kernel, g, 256, 0, seg, cur_e, (nout + 1) / 2, da, nxt_b, nxt_e, d_partial, nout, mail);
            }
            cur_b = nxt_b; cur_e = nxt_e; nxt_b = d_b2; nxt_e = d_ext;  // d_ext is free again (materialised path) / sized for round 2 on
        } else {
            SP1_LAUNCH(ctx, hadamard_fold_kernel, g, 256, 0, cur_b, cur_e, (nout + 1) / 2, da, nxt_b, nxt_e, d_partial, nout, mail);
            std::swap(cur_b, nxt_b); std::swap(cur_e, nxt_e);
        }
        prev_g = g;
    }
    // component evaluations: base[0] (the dense trace at the sumcheck point), ext[0]
    // (posted by the last fold launch next to its, unused, partial sums: payload EF slot 2)
    if (lm < 2) return sp1b200_set_error("jagged_prove: fewer than two sumcheck variables (log_m = %u)", lm);
    SP1_TRY(sp1b200_mail_wait(ctx, prev_seq));
    const E4 base_eval = E4::load(sp1b200_mail_host(ctx) + 8);
    t_sc.stop();

    // ---- jagged evaluation (branching program) sumcheck --------------------------------------------------------------
    SumcheckProof je;
    E4 je_claimed, je_eval;
    {
        PhaseTimer t(ctx, "jagged.eval_sumcheck");
        const uint32_t dim = 2 * (lm + 1);
        // merged prefix sums (bits), condensed over equal consecutive entries; z_col eq values summed per group
        std::vector<uint8_t> bits;
        std::vector<E4> zc;
        uint32_t nk = 0;
        for (size_t c = 0; c + 1 < prefix.size(); c++) {
            std::vector<uint8_t> b(dim);
            for (uint32_t i = 0; i <= lm; i++) { b[i] = (prefix[c] >> (lm - i)) & 1; b[lm + 1 + i] = (prefix[c + 1] >> (lm - i)) & 1; }
            if (nk && std::equal(b.begin(), b.end(), bits.end() - dim)) zc.back() = zc.back() + col_eq_full[c];
            else { bits.insert(bits.end(), b.begin(), b.end()); zc.push_back(col_eq_full[c]); nk++; }
        }
        // per-layer eq((z_row_l, z_index_l), .) ; z_index = the sumcheck point (lm coords), num_vars = max(mlr, lm) -> lm+1 layers used
        const uint32_t hl = lm + 1;
        std::vector<uint32_t> ri((size_t)hl * 16);
        auto lsb = [](const std::vector<E4>& p, uint32_t i) { return p.size() <= i ? E4() : p[p.size() - 1 - i]; };
        if (mlr > hl) return sp1b200_set_error("jagged_prove: max_log_row_count %u exceeds log_m+1 = %u (unsupported shape)", mlr, hl);
        for (uint32_t l = 0; l < hl; l++) {
            E4 zr = lsb(z_row, l), zi = lsb(sc.point, l), one = E4::one();
            E4 p = zr * zi;
            E4 e11 = p, e10 = zr - p, e01 = zi - p, e00 = one - zr - e01;
            e00.store(&ri[l * 16]); e01.store(&ri[l * 16 + 4]); e10.store(&ri[l * 16 + 8]); e11.store(&ri[l * 16 + 12]);
        }
        uint8_t* d_bits; uint32_t *d_ri, *d_zc, *d_inter, *d_part;
        SP1_TRY(mem.alloc((void**)&d_bits, bits.size()));
        SP1_TRY(mem.alloc((void**)&d_ri, ri.size() * 4));
        SP1_TRY(mem.alloc((void**)&d_zc, (size_t)nk * 16));
        SP1_TRY(mem.alloc((void**)&d_inter, (size_t)nk * 16));
        const unsigned nblk = (2 * nk + 127) / 128;
        SP1_TRY(mem.alloc((void**)&d_part, (size_t)nblk * 32));
        SP1_CUDA(cudaMemcpyAsync(d_bits, bits.data(), bits.size(), cudaMemcpyHostToDevice, st));
        SP1_CUDA(cudaMemcpyAsync(d_ri, ri.data(), ri.size() * 4, cudaMemcpyHostToDevice, st));
        SP1_CUDA(cudaMemcpyAsync(d_zc, zc.data(), (size_t)nk * 16, cudaMemcpyHostToDevice, st));
        std::vector<E4> ones(nk, E4::one());
        SP1_CUDA(cudaMemcpyAsync(d_inter, ones.data(), (size_t)nk * 16, cudaMemcpyHostToDevice, st));
        const E4 half = E4::from_base(hf::inv(hf::to_monty(2)));
        const Ext dhalf = to_ext(half);
        // prefix / suffix states (see bp_suffix_kernel): T for the first half now, rebuilt once when the second half starts
        uint32_t *d_T, *d_P, *d_rho_pos;
        SP1_TRY(mem.alloc((void**)&d_T, (size_t)(hl + 2) * nk * 64));
        SP1_TRY(mem.alloc((void**)&d_P, (size_t)nk * 64));
        SP1_TRY(mem.alloc((void**)&d_rho_pos, (size_t)dim * 16));
        {
            std::vector<E4> p0((size_t)nk * 4);
            for (uint32_t k = 0; k < nk; k++) p0[4 * k] = E4::one();
            SP1_CUDA(cudaMemcpyAsync(d_P, p0.data(), p0.size() * 16, cudaMemcpyHostToDevice, st));
            SP1_CUDA(cudaMemsetAsync(d_rho_pos, 0, (size_t)dim * 16, st));
        }
        SP1_LAUNCH(ctx, bp_suffix_kernel, blocks_for(nk, 128), 128, 0, d_bits, nk, dim, 0, d_rho_pos, d_ri, d_T);
        // claimed sum = full evaluation at the boolean prefix sums (full_jagged_little_polynomial_evaluation, poly.rs:183-232):
        // the first-half suffix table reads exactly those bits, so column k evaluates to T_k[0][0]
        {
            std::vector<uint32_t> t0((size_t)nk * 16);
            SP1_CUDA(cudaMemcpyAsync(t0.data(), d_T, t0.size() * 4, cudaMemcpyDeviceToHost, st));
            SP1_CUDA(cudaStreamSynchronize(st));
            for (uint32_t k = 0; k < nk; k++) je_claimed = je_claimed + zc[k] * E4::load(&t0[16 * k]);
        }
        ch.observe_n(je_claimed.c, 4);
        E4 cl = je_claimed;
        const bool bp_mail = (size_t)nblk * 8 <= SP1_MAIL_WORDS;  // otherwise fall back to copy + synchronise
        for (uint32_t round = 0; round < dim; round++) {
            if (round == hl) SP1_LAUNCH(ctx, bp_suffix_kernel, blocks_for(nk, 128), 128, 0, d_bits, nk, dim, 1, d_rho_pos, d_ri, d_T);
            const Mail mail = sp1b200_mail_next(ctx);
            SP1_LAUNCH(ctx, bp_round2_kernel, nblk, 128, 0, d_bits, nk, dim, round, d_rho_pos, d_ri, d_zc, d_inter, d_P, d_T, dhalf,
                       bp_mail ? sp1b200_mail_dev(ctx) : d_part, bp_mail ? mail : Mail{nullptr, nullptr, 0});
            E4 y[2];  // values at 0 and 1/2
            if (bp_mail) SP1_TRY(mail_sums(ctx, mail.seq, nblk, y));
            else SP1_TRY(sum_partials(ctx, d_part, nblk, y));
            E4 c[3];
            interp_0_1_half(y[0], cl - y[0], y[1], c);
            const E4 alpha = je.round(ch, c, 3);
            cl = eval3(c, alpha);
            SP1_LAUNCH(ctx, bp_update_kernel, blocks_for(nk, 128), 128, 0, d_bits, nk, dim, round, to_ext(alpha), d_rho_pos, d_ri, d_inter, d_P);
        }
        je_eval = cl;
        t.stop();
    }

    // ---- dense PCS: prove_untrusted_evaluation(point, base_eval) ---------------------------------------------------
    ch.observe_n(base_eval.c, 4);
    uint32_t chal[34];
    ch.store(chal);
    std::vector<sp1b200_commit*> handles;
    for (uint32_t r = 0; r < n_rounds; r++) handles.push_back(rounds[r]->stacked);
    std::vector<uint32_t> pt(sc.point.size() * 4);
    for (size_t i = 0; i < sc.point.size(); i++) sc.point[i].store(&pt[4 * i]);
    // the stacked proof is written straight into the caller's buffer; the jagged sections are appended after it
    uint64_t nw = 0;
    SP1_TRY(sp1b200_stacked_prove(ctx, handles.data(), n_rounds, pt.data(), (uint32_t)sc.point.size(), h_replay, chal, h_proof, cap, &nw));
    std::vector<uint32_t> proof;
    auto put = [&](const uint32_t* p, size_t n) { proof.insert(proof.end(), p, p + n); };
    auto put1 = [&](uint32_t v) { proof.push_back(v); };
    sc.emit(proof, claim, round_claim);
    je.emit(proof, je_claimed, je_eval);
    for (uint32_t r = 0; r < n_rounds; r++) {
        put1((uint32_t)rounds[r]->row_counts.size());
        for (size_t t = 0; t < rounds[r]->row_counts.size(); t++) { put1((uint32_t)rounds[r]->row_counts[t]); put1((uint32_t)rounds[r]->col_counts[t]); }
    }
    for (uint32_t r = 0; r < n_rounds; r++) put(rounds[r]->original_commit, 8);
    put(base_eval.c, 4);
    put1(mlr);
    put1(lm);
    t_all.stop();
    memcpy(h_chal, chal, sizeof(chal));
    if (h_words) *h_words = nw + proof.size();
    if (nw + proof.size() > cap) return sp1b200_set_error("jagged_prove: proof needs %llu words, capacity %llu", (unsigned long long)(nw + proof.size()), (unsigned long long)cap);
    if (h_proof) memcpy(h_proof + nw, proof.data(), proof.size() * 4);
    return nullptr;
}

}  // extern "C"
