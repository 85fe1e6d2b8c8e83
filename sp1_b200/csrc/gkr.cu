// LogUp-GKR on the device.
// Reference behaviour: crates/hypercube/src/logup_gkr/{prover.rs:70-215, execution.rs:13-382, logup_poly.rs:71-552, cpu.rs:76-226};
// GPU twin it replaces: sp1-gpu/crates/logup_gkr + sys/lib/logup_gkr/{first_layer,execution,round,lookahead}.cu.
// HOW (results identical):
//  * the circuit is kept as ONE fraction sequence per (chip, interaction) and level, F_l[j] (numerator EF, denominator EF),
//    F_{l+1}[j] = F_l[2j] (+) F_l[2j+1]; the reference's four arrays of a layer are the parity classes of F_l
//    (numerator_0 = even entries, numerator_1 = odd entries), so no transposition or re-layout is needed between levels;
//  * every sumcheck round of a layer is one launch over ALL chips (work items are looked up in a small prefix table),
//    fused as "fix the previous variable + accumulate the next round's three sums";
//  * once a layer's row variables are exhausted the remaining (interaction) variables range over <= 2^v <= a few
//    thousand values, which the host transcript driver folds directly.
#include "sumcheck.cuh"
#include <algorithm>
#include <memory>
#include <vector>

#include "machine.cuh"

namespace {

using kb::Ext;
using hf::E4;

struct TermDev { uint32_t source, col, weight; };
struct VColDev { uint32_t term_start, n_terms, constant; };
struct InterDev { uint32_t is_send, arg_index, n_values, vcol_start; };

struct HostInteractions {  // parsed from the machine blob's interaction section
    std::vector<std::vector<InterDev>> per_chip;
    std::vector<VColDev> vcols;
    std::vector<TermDev> terms;
};

struct ChipJob {           // one chip inside a batched launch
    uint64_t work_start;   // prefix of work items
    uint64_t in_off, out_off;  // element offsets of the chip's arrays in the in / out arenas
    uint32_t rows_in;      // rows (or sequence length) of the input arrays
    uint32_t I;            // interactions of the chip
    uint32_t int_off;      // offset into eq_interaction
    uint32_t pad;
};
constexpr int MAX_JOBS = 96;  // 96 * 40 B + 16 B < 4 KB of kernel parameters
struct JobTable { ChipJob j[MAX_JOBS]; uint32_t n; uint64_t total; };

__device__ __forceinline__ int find_job(const JobTable& t, uint64_t w) {
    int lo = 0, hi = (int)t.n;  // j[lo].work_start <= w < j[hi].work_start (hi = n: total)
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (t.j[mid].work_start <= w) lo = mid; else hi = mid; }
    return lo;
}

__device__ __forceinline__ Ext ldE(const uint32_t* p, uint64_t i) { return kb::ext_load(p + 4 * i); }
__device__ __forceinline__ void stE(uint32_t* p, uint64_t i, const Ext& e) { kb::ext_store(p + 4 * i, e); }

// ---- level 0: per (chip, interaction k, row r) fraction from the trace (execution.rs:13-36, 114-252) -----------------------
// q = a / b for work indices that almost always fit 32 bits: the 64-bit division (~60 instructions) only when needed
__device__ __forceinline__ uint32_t div_small(uint64_t a, uint64_t b) {
    return ((a | b) >> 32) ? (uint32_t)(a / b) : (uint32_t)a / (uint32_t)b;
}

__global__ void __launch_bounds__(256) gkr_first_level_kernel(const uint32_t* __restrict__ main, const uint32_t* __restrict__ prep, uint64_t h,
                                                              const InterDev* __restrict__ inter, uint32_t I, const VColDev* __restrict__ vcols,
                                                              const TermDev* __restrict__ terms, Ext alpha, const uint32_t* __restrict__ betas,
                                                              uint32_t* __restrict__ num, uint32_t* __restrict__ den) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= h * I) return;
    const uint32_t k = div_small(t, h);
    const uint64_t r = t - (uint64_t)k * h;
    const InterDev in = inter[k];
    auto apply = [&](const VColDev& v) {
        uint32_t acc = v.constant;
        for (uint32_t q = 0; q < v.n_terms; q++) {
            const TermDev tm = terms[v.term_start + q];
            const uint32_t x = __ldg((tm.source == 4 ? main : prep) + (uint64_t)tm.col * h + r);
            acc = kb::add(acc, kb::mul(x, tm.weight));
        }
        return acc;
    };
    Ext d = kb::ext_add(alpha, kb::ext_mul_base(ldE(betas, 0), kb::from_canonical(in.arg_index)));
    for (uint32_t j = 0; j < in.n_values; j++) d = kb::ext_add(d, kb::ext_mul_base(ldE(betas, j + 1), apply(vcols[in.vcol_start + 1 + j])));
    uint32_t m = apply(vcols[in.vcol_start]);
    if (!in.is_send) m = kb::neg(m);
    stE(num, (uint64_t)k * h + r, kb::ext_from_base(m));
    stE(den, (uint64_t)k * h + r, d);
}

// ---- level l -> l+1: F'[j] = F[2j] (+) F[2j+1]  (missing odd entry = padding (0,1): identity) ------------------------------
__global__ void __launch_bounds__(256) gkr_level_kernel(JobTable jobs, const uint32_t* __restrict__ num, const uint32_t* __restrict__ den,
                                                        uint32_t* __restrict__ num_o, uint32_t* __restrict__ den_o) {
    uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= jobs.total) return;
    const ChipJob& c = jobs.j[find_job(jobs, w)];
    const uint64_t lw = w - c.work_start;
    const uint32_t len_o = (c.rows_in + 1) / 2;
    const uint32_t k = div_small(lw, len_o);
    const uint32_t j = (uint32_t)(lw - (uint64_t)k * len_o);
    const uint64_t base = c.in_off + (uint64_t)k * c.rows_in;
    Ext n0 = ldE(num, base + 2 * j), d0 = ldE(den, base + 2 * j);
    Ext n = n0, d = d0;
    if (2 * j + 1 < c.rows_in) {
        Ext n1 = ldE(num, base + 2 * j + 1), d1 = ldE(den, base + 2 * j + 1);
        n = kb::ext_add(kb::ext_mul(d1, n0), kb::ext_mul(d0, n1));
        d = kb::ext_mul(d0, d1);
    }
    stE(num_o, c.out_off + (uint64_t)k * len_o + j, n);
    stE(den_o, c.out_off + (uint64_t)k * len_o + j, d);
}

// the four layer arrays seen through a fraction sequence F (length len): row i -> (n0,d0) = F[2i], (n1,d1) = F[2i+1]
struct Row4 { Ext n0, d0, n1, d1; };
__device__ __forceinline__ Row4 row_from_seq(const uint32_t* num, const uint32_t* den, uint64_t base, uint32_t len, uint32_t i) {
    Row4 r;
    r.n0 = kb::ext_zero(); r.n1 = kb::ext_zero(); r.d0 = kb::ext_one(); r.d1 = kb::ext_one();
    if (2 * i < len) { r.n0 = ldE(num, base + 2 * i); r.d0 = ldE(den, base + 2 * i); }
    if (2 * i + 1 < len) { r.n1 = ldE(num, base + 2 * i + 1); r.d1 = ldE(den, base + 2 * i + 1); }
    return r;
}
// working layout of a chip (after the first fix): [4][I][rows] EF = n0 | d0 | n1 | d1
__device__ __forceinline__ Row4 row_from_work(const uint32_t* a, uint64_t base, uint32_t I, uint32_t rows, uint32_t k, uint32_t i) {
    Row4 r;
    r.n0 = kb::ext_zero(); r.n1 = kb::ext_zero(); r.d0 = kb::ext_one(); r.d1 = kb::ext_one();
    if (i < rows) {
        const uint64_t s = (uint64_t)I * rows, o = base + (uint64_t)k * rows + i;
        r.n0 = ldE(a, o); r.d0 = ldE(a, o + s); r.n1 = ldE(a, o + 2 * s); r.d1 = ldE(a, o + 3 * s);
    }
    return r;
}
__device__ __forceinline__ Row4 fix_rows(const Row4& x, const Row4& y, const Ext& a) {
    Row4 r;
    r.n0 = kb::ext_add(x.n0, kb::ext_mul(a, kb::ext_sub(y.n0, x.n0)));
    r.d0 = kb::ext_add(x.d0, kb::ext_mul(a, kb::ext_sub(y.d0, x.d0)));
    r.n1 = kb::ext_add(x.n1, kb::ext_mul(a, kb::ext_sub(y.n1, x.n1)));
    r.d1 = kb::ext_add(x.d1, kb::ext_mul(a, kb::ext_sub(y.d1, x.d1)));
    return r;
}
// contributions of the row pair (x = row 2i, y = row 2i+1) to (eval_0, eval_half, eq_sum)   logup_poly.rs:330-505
__device__ __forceinline__ void pair_sums(const Row4& x, const Row4& y, const Ext& e, const Ext& er0, const Ext& er1, const Ext& lambda,
                                          Ext& s0, Ext& sh, Ext& se) {
    Ext t0 = kb::ext_add(kb::ext_mul(lambda, kb::ext_add(kb::ext_mul(x.d0, x.n1), kb::ext_mul(x.d1, x.n0))), kb::ext_mul(x.d0, x.d1));
    Ext D0 = kb::ext_add(x.d0, y.d0), D1 = kb::ext_add(x.d1, y.d1), N0 = kb::ext_add(x.n0, y.n0), N1 = kb::ext_add(x.n1, y.n1);
    Ext th = kb::ext_add(kb::ext_mul(lambda, kb::ext_add(kb::ext_mul(D0, N1), kb::ext_mul(D1, N0))), kb::ext_mul(D0, D1));
    const Ext ee0 = kb::ext_mul(e, er0), ees = kb::ext_mul(e, kb::ext_add(er0, er1));  // shared by the three sums
    s0 = kb::ext_add(s0, kb::ext_mul(ee0, t0));
    sh = kb::ext_add(sh, kb::ext_mul(ees, th));
    se = kb::ext_add(se, ees);
}

// round 0 of a layer: sums straight from the fraction sequence. work item = (chip, k, row pair i)
__global__ void __launch_bounds__(256) gkr_sum_seq_kernel(JobTable jobs, const uint32_t* __restrict__ num, const uint32_t* __restrict__ den,
                                                          const uint32_t* __restrict__ eq_int, const uint32_t* __restrict__ eq_row, Ext lambda,
                                                          uint32_t* __restrict__ partial, Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero(), se = kb::ext_zero();
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < jobs.total; w += (uint64_t)gridDim.x * blockDim.x) {
        const ChipJob& c = jobs.j[find_job(jobs, w)];
        const uint64_t lw = w - c.work_start;
        const uint32_t rows = (c.rows_in + 1) / 2, pairs = (rows + 1) / 2;
        const uint32_t k = div_small(lw, pairs), i = (uint32_t)(lw - (uint64_t)k * pairs);
        const uint64_t base = c.in_off + (uint64_t)k * c.rows_in;
        Row4 x = row_from_seq(num, den, base, c.rows_in, 2 * i), y = row_from_seq(num, den, base, c.rows_in, 2 * i + 1);
        pair_sums(x, y, ldE(eq_int, c.int_off + k), ldE(eq_row, 2 * i), ldE(eq_row, 2 * i + 1), lambda, s0, sh, se);
    }
    block_post_sums<3>({s0, sh, se}, partial, mail);
}

// fix the last row variable (input = fraction sequence or working arrays), write the working arrays of the next round and
// accumulate that round's sums.  work item = (chip, k, NEW row pair i): new rows 2i, 2i+1 come from old rows 4i .. 4i+3.
template <bool FROM_SEQ>
__global__ void __launch_bounds__(256) gkr_fix_sum_kernel(JobTable jobs, const uint32_t* __restrict__ in_a, const uint32_t* __restrict__ in_b,
                                                          uint32_t* __restrict__ out, const uint32_t* __restrict__ eq_int,
                                                          const uint32_t* __restrict__ eq_row_new, Ext alpha, Ext lambda, uint32_t* __restrict__ partial,
                                                          Mail mail) {
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero(), se = kb::ext_zero();
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < jobs.total; w += (uint64_t)gridDim.x * blockDim.x) {
        const ChipJob& c = jobs.j[find_job(jobs, w)];
        const uint64_t lw = w - c.work_start;
        const uint32_t rows_old = FROM_SEQ ? (c.rows_in + 1) / 2 : c.rows_in;
        const uint32_t rows_new = (rows_old + 1) / 2, pairs = (rows_new + 1) / 2;
        const uint32_t k = div_small(lw, pairs), i = (uint32_t)(lw - (uint64_t)k * pairs);
        Row4 nr[2];
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
            const uint32_t o = 2 * i + hh;  // new row index; old rows 2o, 2o+1
            Row4 x, y;
            if (FROM_SEQ) {
                const uint64_t base = c.in_off + (uint64_t)k * c.rows_in;
                x = row_from_seq(in_a, in_b, base, c.rows_in, 2 * o); y = row_from_seq(in_a, in_b, base, c.rows_in, 2 * o + 1);
            } else {
                x = row_from_work(in_a, c.in_off, c.I, rows_old, k, 2 * o); y = row_from_work(in_a, c.in_off, c.I, rows_old, k, 2 * o + 1);
            }
            nr[hh] = fix_rows(x, y, alpha);
            if (o < rows_new) {
                const uint64_t s = (uint64_t)c.I * rows_new, q = c.out_off + (uint64_t)k * rows_new + o;
                stE(out, q, nr[hh].n0); stE(out, q + s, nr[hh].d0); stE(out, q + 2 * s, nr[hh].n1); stE(out, q + 3 * s, nr[hh].d1);
            } else {  // beyond the real rows: padding values for the sums below
                nr[hh].n0 = kb::ext_zero(); nr[hh].n1 = kb::ext_zero(); nr[hh].d0 = kb::ext_one(); nr[hh].d1 = kb::ext_one();
            }
        }
        pair_sums(nr[0], nr[1], ldE(eq_int, c.int_off + k), ldE(eq_row_new, 2 * i), ldE(eq_row_new, 2 * i + 1), lambda, s0, sh, se);
    }
    block_post_sums<3>({s0, sh, se}, partial, mail);
}

// ---- interaction variables (logup_poly.rs:118-176 + the generic round of sumcheck/src/prover.rs) -------------------------------
// After the last row variable every (chip, interaction) holds one row; the layer becomes four arrays over the padded
// interaction index (numerator 0 / denominator 1 beyond the machine's interactions), plus the eq table over that index.
// arr = [5][n] EF: n0 | n1 | d0 | d1 | eq.
__global__ void __launch_bounds__(256) gkr_flatten_kernel(JobTable jobs, const uint32_t* __restrict__ work, const uint32_t* __restrict__ eq_int,
                                                          uint32_t n, uint32_t* __restrict__ arr, uint32_t* __restrict__ payload, Mail mail) {
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        Ext n0 = kb::ext_zero(), n1 = kb::ext_zero(), d0 = kb::ext_one(), d1 = kb::ext_one();
        for (int q = 0; q < jobs.n; q++) {
            const ChipJob& c = jobs.j[q];
            if (t >= c.int_off && t < c.int_off + c.I) {
                const uint64_t o = c.in_off + (t - c.int_off), sI = c.I;  // one row per interaction: [4][I][1]
                n0 = ldE(work, o); d0 = ldE(work, o + sI); n1 = ldE(work, o + 2 * sI); d1 = ldE(work, o + 3 * sI);
            }
        }
        stE(arr, t, n0); stE(arr, (uint64_t)n + t, n1); stE(arr, 2ull * n + t, d0); stE(arr, 3ull * n + t, d1);
        stE(arr, 4ull * n + t, ldE(eq_int, t));
        if (n == 1) { stE(payload, 3, n0); stE(payload, 5, n1); stE(payload, 7, d0); stE(payload, 9, d1); }
    }
    if (mail.flag) sp1_mail_done(mail);
}
// One interaction round in one block: (optionally) bind the previous variable with alpha, store the halved arrays, and post
// (eval_0, eval_half, eq_sum) of the next variable.  When two entries remain they are posted too (payload EF slots 3..10:
// n0[0] n0[1] n1[0] n1[1] d0[0] d0[1] d1[0] d1[1]) so that the host can finish the layer without another launch.
__global__ void __launch_bounds__(256) gkr_inter_round_kernel(const uint32_t* __restrict__ in, uint32_t n_in, int fold, Ext alpha, Ext lambda,
                                                              uint32_t* __restrict__ out, uint32_t* __restrict__ payload, Mail mail) {
    const uint32_t n_cur = fold ? n_in / 2 : n_in;
    Ext s0 = kb::ext_zero(), sh = kb::ext_zero(), se = kb::ext_zero();
    for (uint32_t j = threadIdx.x; j < n_cur / 2; j += blockDim.x) {
        Ext v[5][2];
#pragma unroll
        for (int a = 0; a < 5; a++)
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const uint32_t x = 2 * j + hh;
                if (fold) {
                    const Ext lo = ldE(in, (uint64_t)a * n_in + 2 * x), hi = ldE(in, (uint64_t)a * n_in + 2 * x + 1);
                    v[a][hh] = kb::ext_add(lo, kb::ext_mul(alpha, kb::ext_sub(hi, lo)));
                    stE(out, (uint64_t)a * n_cur + x, v[a][hh]);
                } else v[a][hh] = ldE(in, (uint64_t)a * n_in + x);
            }
        const Ext &n0a = v[0][0], &n1a = v[1][0], &d0a = v[2][0], &d1a = v[3][0], &ea = v[4][0], &eb = v[4][1];
        s0 = kb::ext_add(s0, kb::ext_mul(ea, kb::ext_add(kb::ext_mul(lambda, kb::ext_add(kb::ext_mul(d0a, n1a), kb::ext_mul(d1a, n0a))), kb::ext_mul(d0a, d1a))));
        const Ext N0 = kb::ext_add(v[0][0], v[0][1]), N1 = kb::ext_add(v[1][0], v[1][1]), D0 = kb::ext_add(v[2][0], v[2][1]), D1 = kb::ext_add(v[3][0], v[3][1]);
        const Ext es = kb::ext_add(ea, eb);
        sh = kb::ext_add(sh, kb::ext_mul(es, kb::ext_add(kb::ext_mul(lambda, kb::ext_add(kb::ext_mul(D0, N1), kb::ext_mul(D1, N0))), kb::ext_mul(D0, D1))));
        se = kb::ext_add(se, es);
        if (n_cur == 2) {
#pragma unroll
            for (int a = 0; a < 4; a++) { stE(payload, 3 + 2 * a, v[a][0]); stE(payload, 4 + 2 * a, v[a][1]); }
        }
    }
    block_post_sums<3>({s0, sh, se}, payload, mail);
}

// every read is bounds-checked against the end of the blob and every column against the chip's widths: a blob exported for another
// chip set must become an error, not an out-of-bounds read on host or device
const uint32_t* parse_vcol(const uint32_t* b, const uint32_t* end, HostInteractions& H, uint32_t main_w, uint32_t prep_w) {
    if (end - b < 2) return nullptr;
    VColDev v; v.n_terms = *b++; v.constant = *b++; v.term_start = (uint32_t)H.terms.size();
    if ((uint64_t)v.n_terms * 3 > (uint64_t)(end - b)) return nullptr;
    for (uint32_t i = 0; i < v.n_terms; i++) {
        if ((b[0] != LEAF_MAIN && b[0] != LEAF_PREP) || b[1] >= (b[0] == LEAF_MAIN ? main_w : prep_w)) return nullptr;
        H.terms.push_back(TermDev{b[0], b[1], b[2]}); b += 3;
    }
    H.vcols.push_back(v);
    return b;
}

}  // namespace

// parses the interaction section that follows the AIR records in the machine blob (called by sp1b200_machine_create);
// widths[2k], widths[2k+1] = main / preprocessed width of chip k.  Returns nullptr (with the error set) on a malformed section.
void* sp1b200_parse_interactions(const uint32_t* b, const uint32_t* end, size_t n_chips, const uint32_t* widths) {
    auto H = std::make_unique<HostInteractions>();
    H->per_chip.resize(n_chips);
    if (b >= end) return H.release();  // machine without interactions (zerocheck-only tests)
    size_t k = 0;
    for (auto& chip : H->per_chip) {
        const uint32_t mw = widths[2 * k], pw = widths[2 * k + 1];
        if (end - b < 1) { sp1b200_set_error("machine_create: truncated interaction section (chip %zu)", k); return nullptr; }
        uint32_t n = *b++;
        for (uint32_t i = 0; i < n; i++) {
            if (end - b < 3) { sp1b200_set_error("machine_create: truncated interaction section (chip %zu)", k); return nullptr; }
            InterDev in; in.is_send = *b++; in.arg_index = *b++; in.n_values = *b++; in.vcol_start = (uint32_t)H->vcols.size();
            if (in.n_values > 255) { sp1b200_set_error("machine_create: chip %zu interaction %u has %u values", k, i, in.n_values); return nullptr; }
            for (uint32_t v = 0; v <= in.n_values; v++) {   // multiplicity, then the values
                b = parse_vcol(b, end, *H, mw, pw);
                if (!b) { sp1b200_set_error("machine_create: chip %zu interaction %u: malformed or out-of-range virtual column", k, i); return nullptr; }
            }
            chip.push_back(in);
        }
        k++;
    }
    return H.release();
}
void sp1b200_free_interactions(void* p) { delete static_cast<HostInteractions*>(p); }

#include "gkr_driver.inc"
