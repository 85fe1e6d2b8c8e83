// Zerocheck on the device: AIR constraint bytecode interpreter + per-round sum / fix kernels + the multi-chip
// sumcheck driver.  Reference behaviour: crates/hypercube/src/prover/shard.rs:474-646,
// crates/hypercube/src/prover/zerocheck/{sum_as_poly.rs:49-440, fix_last_variable.rs:8-62}, slop/crates/sumcheck/src/prover.rs:13-96;
// GPU twin it replaces: sp1-gpu/crates/zerocheck/src/prover.rs + sys/lib/zerocheck/{sequential,gkr_sweep,geq_corrections,pad_adj}.cu.
// Input contract for the constraints = the reference GPU prover's bytecode (sys/include/zerocheck/sequential.cuh:13-49):
// DagInstr / LeafRef / BcOp, asserts as (register, alpha index) pairs.
// HOW (B200): every chip's bytecode is re-scheduled at upload (zc_lower.hpp) so that its live set fits a SHARED-MEMORY
// register file; one launch per round covers ALL chips (block -> (chip, row chunk), evaluation node on grid.y), a second tiny
// launch reduces the per-block partial sums, and one 5 KB copy + one sync per round feeds the host transcript.  The linear
// opening-batching term  sum_j gamma^j col_j  is evaluated once per row pair (at 0 and 1) instead of at every node.
// The eq table is built once and halved per round; trace columns stay column-major (base field in round 0, EF afterwards);
// geq / padded-row corrections and the 5-node interpolation run on the host from nine EF partial sums per chip.
#include "sumcheck.cuh"
#include <algorithm>
#include <memory>
#include <vector>

#include "machine.cuh"
#include "zc_lower.hpp"

namespace {

using kb::Ext;
using hf::E4;

constexpr int ZC_BLOCK = 128;
constexpr int ZC_LOCAL_REGS = 128;    // second tier: register file in local memory
constexpr int ZC_GLOBAL_REGS = 1024;  // last tier: register file in a global-memory workspace (the reference's largest tier,
                                      // sys/lib/zerocheck/sequential.cu:298-335, keeps K regs[1024] in per-thread local memory)
constexpr unsigned ZC_GLOBAL_MAXB = 148 * 2;  // blocks of a global-tier job: bounds the workspace (blocks x regs x 3 nodes x 128 x 16 B)
constexpr size_t ZC_MAX_PIECES = 16;

template <class K> struct Ops;
template <> struct Ops<uint32_t> {
    static __device__ __forceinline__ uint32_t zero() { return 0; }
    static __device__ __forceinline__ uint32_t from_base(uint32_t x) { return x; }
    static __device__ __forceinline__ uint32_t add(uint32_t a, uint32_t b) { return kb::add(a, b); }
    static __device__ __forceinline__ uint32_t sub(uint32_t a, uint32_t b) { return kb::sub(a, b); }
    static __device__ __forceinline__ uint32_t mul(uint32_t a, uint32_t b) { return kb::mul(a, b); }
    static __device__ __forceinline__ uint32_t load(const uint32_t* p, uint64_t i) { return __ldg(p + i); }
    static __device__ __forceinline__ Ext scale(const Ext& e, uint32_t k) { return kb::ext_mul_base(e, k); }
};
template <> struct Ops<Ext> {
    static __device__ __forceinline__ Ext zero() { return kb::ext_zero(); }
    static __device__ __forceinline__ Ext from_base(uint32_t x) { return kb::ext_from_base(x); }
    static __device__ __forceinline__ Ext add(const Ext& a, const Ext& b) { return kb::ext_add(a, b); }
    static __device__ __forceinline__ Ext sub(const Ext& a, const Ext& b) { return kb::ext_sub(a, b); }
    static __device__ __forceinline__ Ext mul(const Ext& a, const Ext& b) { return kb::ext_mul(a, b); }
    static __device__ __forceinline__ Ext load(const Ext* p, uint64_t i) { return kb::ext_load(reinterpret_cast<const uint32_t*>(p + i)); }
    static __device__ __forceinline__ Ext scale(const Ext& e, const Ext& k) { return kb::ext_mul(e, k); }
};

// one chip in one round
struct ZcJob {
    const void* main; const void* prep; const uint32_t* alpha_pows; uint64_t h;
    uint32_t blk_start, nblk, chip, columns;   // columns != 0: this job also evaluates the opening-batching term
    uint32_t zc_begin, zc_end;                 // the piece of the chip's instruction stream this job interprets
    const void* batch;                         // EF rounds: the chip's pre-batched column B[r] = sum_j gamma^(j+1) col_j[r] (nullptr in round 0)
};
static_assert(sizeof(ZcJob) == 64, "ZcJob layout");
struct ZcFixJob {
    const void* main; const void* prep; uint32_t* out; uint64_t h;
    uint32_t main_w, prep_w, blk_start, pad;
};

// register file: every register holds the value at ALL THREE evaluation nodes (the program is decoded once per row pair and
// the three evaluations run in lockstep: one instruction fetch, three independent products in flight, one pass over the
// columns).  RF_SMEM: shared memory [reg][node][thread]; RF_LOCAL: a local array (<= 128 registers); RF_GLOBAL: the same
// [reg][node][thread] layout in a per-block slice of a global workspace (coalesced, sized by the program's real pressure, L1/L2
// resident for the hot registers) for programs of up to 1024 live registers.
enum { RF_SMEM = 0, RF_LOCAL = 1, RF_GLOBAL = 2 };
template <class K, int RF> struct RegFile;
template <class K> struct RegFile<K, RF_SMEM> {
    K* base;
    __device__ __forceinline__ RegFile(unsigned char* smem, void*, uint32_t) : base(reinterpret_cast<K*>(smem) + threadIdx.x) {}
    __device__ __forceinline__ K get(uint32_t r, int n) const { return base[(r * 3 + n) * ZC_BLOCK]; }
    __device__ __forceinline__ void set(uint32_t r, int n, const K& v) { base[(r * 3 + n) * ZC_BLOCK] = v; }
};
template <class K> struct RegFile<K, RF_LOCAL> {
    K regs[ZC_LOCAL_REGS * 3];
    __device__ __forceinline__ RegFile(unsigned char*, void*, uint32_t) {}
    __device__ __forceinline__ K get(uint32_t r, int n) const { return regs[r * 3 + n]; }
    __device__ __forceinline__ void set(uint32_t r, int n, const K& v) { regs[r * 3 + n] = v; }
};
template <class K> struct RegFile<K, RF_GLOBAL> {
    K* base;
    __device__ __forceinline__ RegFile(unsigned char*, void* ws, uint32_t ws_regs)
        : base(static_cast<K*>(ws) + (size_t)blockIdx.x * ws_regs * 3 * ZC_BLOCK + threadIdx.x) {}
    __device__ __forceinline__ K get(uint32_t r, int n) const { return base[(size_t)(r * 3 + n) * ZC_BLOCK]; }
    __device__ __forceinline__ void set(uint32_t r, int n, const K& v) { base[(size_t)(r * 3 + n) * ZC_BLOCK] = v; }
};

// column values at the nodes t = 0, 2, 4 of row pair i:  z, z + 2d, z + 4d  with d = o - z (o = 0 past the last real row)
template <class K, int N0>
__device__ __forceinline__ void load_nodes(const K* __restrict__ base, uint32_t col, uint64_t h, uint64_t i, K (&v)[3]) {
    using O = Ops<K>;
    const K* c = base + (uint64_t)col * h;
    const K z = O::load(c, 2 * i);
    const K o = (2 * i + 1 < h) ? O::load(c, 2 * i + 1) : O::zero();
    const K d = O::sub(o, z);
    const K d2 = O::add(d, d);
    if (N0 == 0) v[0] = z;
    v[1] = O::add(z, d2);
    v[2] = O::add(v[1], d2);
}

// partial[(blockIdx.x * 3 + node) * 3 + {0,1,2}] =
//   0: sum_rows E[i] * [constraints](node)     1 (node 0 only): sum_rows E[i] * sum_j g_j col_j(0)     2 (node 0 only): same at 1
// FIRST (round 0): the constraints vanish on the boolean rows, so node 0 is skipped (N0 = 1).
template <class K, int RF, bool FIRST>
__global__ void __launch_bounds__(ZC_BLOCK) zc_sum_kernel(const ZcJob* __restrict__ jobs, int n_jobs, const ChipProg* __restrict__ chips,
                                                          const uint32_t* __restrict__ pv, const uint32_t* __restrict__ gkr_pows,
                                                          const uint32_t* __restrict__ E, uint32_t* __restrict__ partial,
                                                          void* __restrict__ ws, uint32_t ws_regs) {
    using O = Ops<K>;
    constexpr int N0 = FIRST ? 1 : 0;
    extern __shared__ __align__(16) unsigned char zc_smem[];
    __shared__ uint32_t red[5][4][ZC_BLOCK / 32];
    const ZcJob job = jobs[find_job(jobs, n_jobs, blockIdx.x)];
    const ChipProg& prog = chips[job.chip];
    const K* main = static_cast<const K*>(job.main);
    const K* prep = static_cast<const K*>(job.prep);
    const uint64_t h = job.h;
    const uint64_t terms = (h + 1) / 2;
    RegFile<K, RF> rf(zc_smem, ws, ws_regs);
    Ext acc[5];  // constraints at nodes 0,1,2 ; opening-batching term at 0 and at 1
#pragma unroll
    for (int a = 0; a < 5; a++) acc[a] = kb::ext_zero();
    const ZcInstr* __restrict__ zc = prog.zc + job.zc_begin;
    const uint32_t n_zc = job.zc_end - job.zc_begin;
    for (uint64_t i = (uint64_t)(blockIdx.x - job.blk_start) * ZC_BLOCK + threadIdx.x; i < terms; i += (uint64_t)job.nblk * ZC_BLOCK) {
        const Ext e = kb::ext_load(E + 4 * i);
        Ext row[3] = {kb::ext_zero(), kb::ext_zero(), kb::ext_zero()};
        ZcInstr in = n_zc ? zc[0] : ZcInstr{};
        for (uint32_t pc = 0; pc < n_zc; pc++) {
            const ZcInstr nxt = zc[pc + 1 < n_zc ? pc + 1 : pc];  // prefetch: the stream is block-uniform and L1 resident
            switch (in.op) {
                case ZC_LOAD_MAIN: case ZC_LOAD_PREP: {
                    K v[3];
                    load_nodes<K, N0>(in.op == ZC_LOAD_MAIN ? main : prep, (uint32_t)in.a | ((uint32_t)in.b << 16), h, i, v);
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, v[n]);
                    break;
                }
                case ZC_CONST: { const K c = O::from_base(prog.consts[in.a]);
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, c);
                    break; }
                case ZC_PUBLIC: { const K c = O::from_base(pv[prog.publics[in.a]]);
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, c);
                    break; }
                case ZC_ADD: {
                    K r[3];
#pragma unroll
                    for (int n = N0; n < 3; n++) r[n] = O::add(rf.get(in.a, n), rf.get(in.b, n));
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, r[n]);
                    break; }
                case ZC_SUB: {
                    K r[3];
#pragma unroll
                    for (int n = N0; n < 3; n++) r[n] = O::sub(rf.get(in.a, n), rf.get(in.b, n));
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, r[n]);
                    break; }
                case ZC_MUL: {
                    K r[3];
#pragma unroll
                    for (int n = N0; n < 3; n++) r[n] = O::mul(rf.get(in.a, n), rf.get(in.b, n));
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, r[n]);
                    break; }
                case ZC_NEG: {
                    K r[3];
#pragma unroll
                    for (int n = N0; n < 3; n++) r[n] = O::sub(O::zero(), rf.get(in.a, n));
#pragma unroll
                    for (int n = N0; n < 3; n++) rf.set(in.out, n, r[n]);
                    break; }
                case ZC_ASSERT: {
                    const Ext al = kb::ext_load(job.alpha_pows + 4 * in.b);
#pragma unroll
                    for (int n = N0; n < 3; n++) row[n] = kb::ext_add(row[n], O::scale(al, rf.get(in.a, n)));
                    break; }
                default: __trap();
            }
            in = nxt;
        }
#pragma unroll
        for (int n = N0; n < 3; n++) acc[n] = kb::ext_add(acc[n], kb::ext_mul(row[n], e));
        if (!job.columns) continue;
        // the opening-batching term is linear in the row variable: evaluate it at 0 and 1 only
        Ext s0 = kb::ext_zero(), s1 = kb::ext_zero();
        const bool has_o = 2 * i + 1 < h;
        if (job.batch) {
            // EF rounds: the term is linear in the columns too, so it is carried as ONE pre-batched column per chip that is folded
            // with the others (zc_batch0_kernel builds it after round 0): two loads instead of 2 x width extension products
            const uint32_t* B = static_cast<const uint32_t*>(job.batch);
            acc[3] = kb::ext_add(acc[3], kb::ext_mul(kb::ext_load(B + 8 * i), e));
            if (has_o) acc[4] = kb::ext_add(acc[4], kb::ext_mul(kb::ext_load(B + 8 * i + 4), e));
            continue;
        }
        for (uint32_t j = 0; j < prog.main_w; j++) {
            const Ext g = kb::ext_load(gkr_pows + 4 * j);
            const K* c = main + (uint64_t)j * h;
            s0 = kb::ext_add(s0, O::scale(g, O::load(c, 2 * i)));
            if (has_o) s1 = kb::ext_add(s1, O::scale(g, O::load(c, 2 * i + 1)));
        }
        for (uint32_t j = 0; j < prog.prep_w; j++) {
            const Ext g = kb::ext_load(gkr_pows + 4 * (prog.main_w + j));
            const K* c = prep + (uint64_t)j * h;
            s0 = kb::ext_add(s0, O::scale(g, O::load(c, 2 * i)));
            if (has_o) s1 = kb::ext_add(s1, O::scale(g, O::load(c, 2 * i + 1)));
        }
        acc[3] = kb::ext_add(acc[3], kb::ext_mul(s0, e));
        acc[4] = kb::ext_add(acc[4], kb::ext_mul(s1, e));
    }
    // block reduction: warp shuffles, then one thread per word over the per-warp sums
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 5; a++)
#pragma unroll
        for (int l = 0; l < 4; l++) {
            uint32_t v = acc[a].c[l];
            for (int s = 16; s > 0; s >>= 1) v = kb::add(v, __shfl_down_sync(0xffffffffu, v, s));
            if (lane == 0) red[a][l][warp] = v;
        }
    __syncthreads();
    if (threadIdx.x < 36) {
        // word w of the block's 36: node = w / 12, slot = (w / 4) % 3, limb = w % 4
        const int node = threadIdx.x / 12, slot = (threadIdx.x >> 2) % 3, l = threadIdx.x & 3;
        const int a = slot == 0 ? node : (node == 0 ? 2 + slot : -1);
        uint32_t v = 0;
        if (a >= 0)
            for (int w = 0; w < ZC_BLOCK / 32; w++) v = kb::add(v, red[a][l][w]);
        partial[(uint64_t)blockIdx.x * 36 + threadIdx.x] = v;
    }
}

// out[(job * 3 + node) * 3 + slot] = sum over the job's blocks
__global__ void __launch_bounds__(128) zc_reduce_kernel(const ZcJob* __restrict__ jobs, const uint32_t* __restrict__ partial, uint32_t* __restrict__ out,
                                                        Mail mail) {
    const ZcJob job = jobs[blockIdx.x];
    __shared__ uint32_t red[36][4];
    const int slot = threadIdx.x >> 2, part = threadIdx.x & 3;  // 32 groups of 4 threads; 36 words = 9 ext -> loop
    for (int w = slot; w < 36; w += 32) {
        uint32_t v = 0;
        for (uint32_t b = part; b < job.nblk; b += 4) v = kb::add(v, partial[(uint64_t)(job.blk_start + b) * 36 + w]);
        red[w][part] = v;
    }
    __syncthreads();
    if (threadIdx.x < 36) {
        const uint32_t* r = red[threadIdx.x];
        out[blockIdx.x * 36 + threadIdx.x] = kb::add(kb::add(r[0], r[1]), kb::add(r[2], r[3]));
    }
    sp1_mail_done(mail);  // `out` is the mailbox payload: the host polls the flag instead of copy + synchronise
}

// out[j][i] = in[j][2i] + alpha (in[j][2i+1] - in[j][2i]),  i < ceil(h/2)   (column-major, EF out; main columns then preprocessed)
template <class K>
__global__ void __launch_bounds__(256) zc_fix_kernel(const ZcFixJob* __restrict__ jobs, int n_jobs, Ext alpha) {
    using O = Ops<K>;
    const ZcFixJob job = jobs[find_job(jobs, n_jobs, blockIdx.x)];
    const uint64_t h = job.h, nh = (h + 1) / 2;
    // a block covers 256 consecutive row pairs of ONE column: (column, chunk) from the block index with one 32-bit division
    // (a flat element index would cost a 64-bit division per element, comparable to the two field operations of the fold itself)
    const uint32_t bpc = (uint32_t)((nh + 255) / 256);
    const uint32_t lb = blockIdx.x - job.blk_start;
    const uint64_t j = lb / bpc;
    const uint64_t i = (uint64_t)(lb - (uint32_t)j * bpc) * 256 + threadIdx.x;
    if (i >= nh) return;
    const uint64_t t = j * nh + i;
    const K* in = j < job.main_w ? static_cast<const K*>(job.main) + j * h : static_cast<const K*>(job.prep) + (j - job.main_w) * h;
    K a = O::load(in, 2 * i);
    K b = (2 * i + 1 < h) ? O::load(in, 2 * i + 1) : O::zero();
    Ext r;
    if constexpr (sizeof(K) == 4) r = kb::ext_add(kb::ext_from_base(a), kb::ext_mul_base(alpha, kb::sub(b, a)));
    else r = kb::ext_add(a, kb::ext_mul(alpha, kb::ext_sub(b, a)));
    kb::ext_store(job.out + 4 * t, r);
}

// After round 0: the pre-batched column of every chip in the first EF arena,
//   B[i] = sum_j g_j (col_j[2i] + alpha (col_j[2i+1] - col_j[2i])) = sum_j g_j a_j + alpha sum_j g_j (b_j - a_j)      (base-field a, b)
// one thread per output row, EF x F products only.  job.out = the chip's B column; job.main / job.prep = the BASE columns.
__global__ void __launch_bounds__(256) zc_batch0_kernel(const ZcFixJob* __restrict__ jobs, int n_jobs, const uint32_t* __restrict__ gkr_pows, Ext alpha) {
    const ZcFixJob job = jobs[find_job(jobs, n_jobs, blockIdx.x)];
    const uint64_t h = job.h, nh = (h + 1) / 2;
    const uint64_t i = (uint64_t)(blockIdx.x - job.blk_start) * 256 + threadIdx.x;
    if (i >= nh) return;
    const bool has_o = 2 * i + 1 < h;
    Ext sa = kb::ext_zero(), sd = kb::ext_zero();
    const uint32_t* main = static_cast<const uint32_t*>(job.main);
    const uint32_t* prep = static_cast<const uint32_t*>(job.prep);
    for (uint32_t j = 0; j < job.main_w + job.prep_w; j++) {
        const uint32_t* c = j < job.main_w ? main + (uint64_t)j * h : prep + (uint64_t)(j - job.main_w) * h;
        const uint32_t a = __ldg(c + 2 * i), b = has_o ? __ldg(c + 2 * i + 1) : 0u;
        const Ext g = kb::ext_load(gkr_pows + 4 * j);
        sa = kb::ext_add(sa, kb::ext_mul_base(g, a));
        sd = kb::ext_add(sd, kb::ext_mul_base(g, kb::sub(b, a)));
    }
    kb::ext_store(job.out + 4 * i, kb::ext_add(sa, kb::ext_mul(alpha, sd)));
}

// host interpreter on the all-zero row (padded_row_adjustment, shard.rs:520-537): Σ powers[alpha_idx] * reg
E4 host_eval_zero_row(const HostProg& p, const uint32_t* pv, const std::vector<E4>& powers, uint32_t n_regs) {
    std::vector<uint32_t> regs(n_regs ? n_regs : 1, 0);
    for (const DagInstr& in : p.instrs) {
        switch (in.opcode) {
            case BC_LOAD_LEAF: regs[in.out] = 0; break;
            case BC_LOAD_CONST: regs[in.out] = p.consts[in.a]; break;
            case BC_LOAD_PUBLIC: regs[in.out] = pv[p.publics[in.a]]; break;
            case BC_ADD_F: regs[in.out] = hf::add(regs[in.a], regs[in.b]); break;
            case BC_SUB_F: regs[in.out] = hf::sub(regs[in.a], regs[in.b]); break;
            case BC_MUL_F: regs[in.out] = hf::mul(regs[in.a], regs[in.b]); break;
            case BC_NEG_F: regs[in.out] = hf::neg(regs[in.a]); break;
        }
    }
    E4 acc;
    for (size_t i = 0; i < p.assert_regs.size(); i++) acc = acc + powers[p.assert_alphas[i]] * regs[p.assert_regs[i]];
    return acc;
}

struct VGeq {
    uint32_t threshold = 0; E4 geq_c, eq_c;
    VGeq fix_last(const E4& a) const {
        VGeq r; r.threshold = threshold >> 1; r.geq_c = geq_c;
        r.eq_c = (threshold & 1) == 0 ? (E4::one() - a) * eq_c : a * (eq_c + geq_c) - geq_c;
        return r;
    }
    E4 at(uint64_t idx) const { return idx < threshold ? E4() : (idx == threshold ? eq_c + geq_c : geq_c); }
};

}  // namespace

sp1b200_machine::~sp1b200_machine() {
    if (interactions) sp1b200_free_interactions(interactions);
    cudaFree(d_arena);
    cudaFree(d_zc_arena);
    cudaFree(d_chips);
}

extern "C" {

// Upload a machine's constraint bytecode once (replaces upload_machine_bytecode, sp1-gpu/crates/zerocheck/src/prover.rs).
// blob words: [n_chips] then per chip: main_w prep_w n_constraints n_regs n_instrs n_leaves n_consts n_publics n_asserts,
// instrs (2 words = one 8-byte DagInstr), leaves (2 words = LeafRef), consts (Montgomery), publics, assert_regs, assert_alphas.
sp1b200_err sp1b200_machine_create(sp1b200_ctx* ctx, const uint32_t* h_blob, uint64_t n_words, sp1b200_machine** out) { SP1_DEVICE_GUARD(ctx);
    auto m = std::make_unique<sp1b200_machine>();
    SP1_CUDA(cudaMalloc((void**)&m->d_arena, n_words * 4 + 16));
    SP1_CUDA(cudaMemcpyAsync(m->d_arena, h_blob, n_words * 4, cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t* b = h_blob;
    const uint32_t* end = h_blob + n_words;
    auto dev = [&](const uint32_t* hp) { return m->d_arena + (hp - h_blob); };
    if (n_words < 1 || !h_blob) return sp1b200_set_error("machine_create: empty blob");
    uint32_t n = *b++;
    for (uint32_t c = 0; c < n; c++) {
        if ((uint64_t)(end - b) < 9) return sp1b200_set_error("machine_create: truncated blob (header of chip %u)", c);
        ChipProg p{}; HostProg hp;
        p.main_w = *b++; p.prep_w = *b++; p.n_constraints = *b++; p.n_regs = *b++;
        const uint64_t ni = *b++, nl = *b++, nc = *b++, np = *b++, na = *b++;
        // all size arithmetic in 64 bits against the words that are left (a 32-bit sum could wrap past the check)
        if (2 * ni + 2 * nl + nc + np + 2 * na > (uint64_t)(end - b)) return sp1b200_set_error("machine_create: truncated blob (chip %u)", c);
        if (p.n_regs > 65536) return sp1b200_set_error("machine_create: chip %u declares %u registers (16-bit register indices)", c, p.n_regs);
        p.n_instrs = (uint32_t)ni; p.n_asserts = (uint32_t)na;
        p.instrs = reinterpret_cast<const DagInstr*>(dev(b)); hp.instrs.resize(ni); memcpy(hp.instrs.data(), b, ni * 8); b += 2 * ni;
        p.leaves = reinterpret_cast<const LeafRef*>(dev(b)); hp.leaves.resize(nl); memcpy(hp.leaves.data(), b, nl * 8); b += 2 * nl;
        p.consts = dev(b); hp.consts.assign(b, b + nc); b += nc;
        p.publics = dev(b); hp.publics.assign(b, b + np); b += np;
        p.assert_regs = dev(b); hp.assert_regs.assign(b, b + na); b += na;
        p.assert_alphas = dev(b); hp.assert_alphas.assign(b, b + na); b += na;
        // a blob exported for a different chip set must become an error, not an out-of-bounds read on host or device
        for (const LeafRef& l : hp.leaves) {
            if (l.source != LEAF_MAIN && l.source != LEAF_PREP) return sp1b200_set_error("machine_create: chip %u: leaf source %u (expected 2 = preprocessed or 4 = main)", c, l.source);
            if (l.col >= (l.source == LEAF_MAIN ? p.main_w : p.prep_w)) return sp1b200_set_error("machine_create: chip %u: leaf column %u outside the %s width", c, l.col, l.source == LEAF_MAIN ? "main" : "preprocessed");
        }
        for (size_t k = 0; k < hp.instrs.size(); k++) {
            const DagInstr& in = hp.instrs[k];
            if (in.out >= p.n_regs) return sp1b200_set_error("machine_create: chip %u instr %zu: output register %u >= n_regs %u", c, k, in.out, p.n_regs);
            bool ok = true;
            switch (in.opcode) {
                case BC_LOAD_LEAF: ok = in.a < nl; break;
                case BC_LOAD_CONST: ok = in.a < nc; break;
                case BC_LOAD_PUBLIC: ok = in.a < np; break;
                case BC_ADD_F: case BC_SUB_F: case BC_MUL_F: ok = in.a < p.n_regs && in.b < p.n_regs; break;
                case BC_NEG_F: ok = in.a < p.n_regs; break;
                default: return sp1b200_set_error("machine_create: chip %u instr %zu: unknown opcode %u", c, k, in.opcode);
            }
            if (!ok) return sp1b200_set_error("machine_create: chip %u instr %zu: operand out of range (opcode %u, a %u, b %u)", c, k, in.opcode, in.a, in.b);
        }
        for (size_t k = 0; k < hp.assert_regs.size(); k++) {
            if (hp.assert_regs[k] >= p.n_regs) return sp1b200_set_error("machine_create: chip %u assert %zu: register %u >= n_regs %u", c, k, hp.assert_regs[k], p.n_regs);
            if (hp.assert_alphas[k] >= p.n_constraints) return sp1b200_set_error("machine_create: chip %u assert %zu: alpha index %u >= n_constraints %u", c, k, hp.assert_alphas[k], p.n_constraints);
        }
        m->chips.push_back(p); m->host.push_back(std::move(hp));
    }
    {
        std::vector<uint32_t> widths;
        for (auto& c : m->chips) { widths.push_back(c.main_w); widths.push_back(c.prep_w); }
        widths.push_back(0);
        m->interactions = sp1b200_parse_interactions(b, end, n, widths.data());
        if (!m->interactions) return sp1b200_last_error();   // message set by the parser
    }
    // re-schedule every chip's program for the shared-memory register file (zc_lower.hpp) and upload the streams
    std::vector<ZcInstr> all;
    std::vector<size_t> zc_off(n);
    for (uint32_t c = 0; c < n; c++) {
        ZcLowered L = zc_lower(m->host[c]);
        if (!L.error.empty()) return sp1b200_set_error("machine_create: chip %u: %s", c, L.error.c_str());
        zc_off[c] = all.size();
        m->chips[c].n_zc = (uint32_t)L.instrs.size();
        m->chips[c].zc_regs = L.n_regs;
        all.insert(all.end(), L.instrs.begin(), L.instrs.end());
        // pieces for the short rounds: the asserts split into up to ZC_MAX_PIECES contiguous groups of >= 4, each lowered on its own
        const size_t na = m->host[c].assert_regs.size();
        const size_t np_ = std::min<size_t>(ZC_MAX_PIECES, na / 4);
        if (np_ >= 2 && L.instrs.size() >= 128) {
            for (size_t q = 0; q < np_; q++) {
                ZcLowered P = zc_lower(m->host[c], 24, na * q / np_, na * (q + 1) / np_);
                if (!P.error.empty()) return sp1b200_set_error("machine_create: chip %u: %s", c, P.error.c_str());
                m->host[c].zc_pieces.emplace_back((uint32_t)(all.size() - zc_off[c]), (uint32_t)P.instrs.size());
                m->chips[c].zc_regs = std::max(m->chips[c].zc_regs, P.n_regs);
                all.insert(all.end(), P.instrs.begin(), P.instrs.end());
            }
        }
    }
    SP1_CUDA(cudaMalloc(&m->d_zc_arena, all.size() * sizeof(ZcInstr) + 16));
    if (!all.empty()) SP1_CUDA(cudaMemcpyAsync(m->d_zc_arena, all.data(), all.size() * sizeof(ZcInstr), cudaMemcpyHostToDevice, ctx->stream));
    for (uint32_t c = 0; c < n; c++) m->chips[c].zc = static_cast<const ZcInstr*>(m->d_zc_arena) + zc_off[c];
    SP1_CUDA(cudaMalloc((void**)&m->d_chips, (n ? n : 1) * sizeof(ChipProg)));
    if (n) SP1_CUDA(cudaMemcpyAsync(m->d_chips, m->chips.data(), n * sizeof(ChipProg), cudaMemcpyHostToDevice, ctx->stream));
    SP1_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = m.release();
    return nullptr;
}
void sp1b200_machine_free(sp1b200_ctx*, sp1b200_machine* m) { delete m; }
// peak register pressure of a chip's re-scheduled program (tests / diagnostics)
uint32_t sp1b200_machine_chip_regs(const sp1b200_machine* m, uint32_t chip) { return chip < m->chips.size() ? m->chips[chip].zc_regs : 0; }
uint32_t sp1b200_machine_num_chips(const sp1b200_machine* m) { return (uint32_t)m->chips.size(); }

// ShardProver::zerocheck (crates/hypercube/src/prover/shard.rs:474-646).
// d_main[k] / d_prep[k]: device pointers, column-major [w x heights[k]] base-field columns (prep may be NULL when prep_w == 0);
// h_alpha / h_gamma: the constraint- and opening-batching challenges already sampled by the caller (shard.rs:707-709);
// h_claims: per chip Σ_j gamma^(j+1) opening_j (main then preprocessed) from LogUp-GKR; h_gkr_point: max_log_row_count ext.
// Output words: sumcheck proof {n_polys, per poly {n_coeffs, coeffs}, claimed_sum, point, eval} | per chip {prep evals, main evals}.
sp1b200_err sp1b200_zerocheck(sp1b200_ctx* ctx, const sp1b200_machine* m, const uint64_t* h_heights, const uint32_t* const* d_main,
                              const uint32_t* const* d_prep, const uint32_t* h_pv, uint32_t n_pv, const uint32_t* h_gkr_point,
                              const uint32_t* h_alpha, const uint32_t* h_gamma, const uint32_t* h_claims, uint32_t* h_chal, uint32_t* h_out,
                              uint64_t cap, uint64_t* h_words) { SP1_DEVICE_GUARD(ctx);
    const uint32_t mlr = ctx->params.max_log_row_count;
    const size_t nchips = m->chips.size();
    for (size_t k = 0; k < nchips; k++)
        for (uint32_t pi : m->host[k].publics)
            if (pi >= n_pv) return sp1b200_set_error("zerocheck: chip %zu reads public value %u but only %u were passed", k, pi, n_pv);
    cudaStream_t st = ctx->stream;
    DevFree mem(ctx);
    HostChallenger ch;
    SP1_TRY(ch.init(ctx, h_chal));
    PhaseTimer t_all(ctx, "zerocheck.total");
    HostAccum acc_wait(ctx, "zerocheck.host_wait"), acc_math(ctx, "zerocheck.host_math"), acc_setup(ctx, "zerocheck.host_setup");
    auto t_setup = std::make_unique<HostSpan>(acc_setup);
    const E4 alpha = E4::load(h_alpha), gamma = E4::load(h_gamma);

    struct St {
        uint64_t h;
        std::vector<E4> zeta; E4 eq_adj = E4::one(), pra; VGeq vg;
    };
    std::vector<St> S(nchips);
    size_t maxc = 0, maxw = 0, total_w = 0, total_c = 0;
    for (auto& c : m->chips) {
        maxc = std::max<size_t>(maxc, c.n_constraints); maxw = std::max<size_t>(maxw, c.main_w + c.prep_w);
        total_w += c.main_w + c.prep_w; total_c += c.n_constraints ? c.n_constraints : 1;
    }
    std::vector<E4> pw(maxc ? maxc : 1); pw[0] = E4::one();
    for (size_t i = 1; i < pw.size(); i++) pw[i] = pw[i - 1] * alpha;
    std::vector<E4> gw(maxw ? maxw : 1); gw[0] = gamma;
    for (size_t i = 1; i < gw.size(); i++) gw[i] = gw[i - 1] * gamma;
    uint32_t *d_pv, *d_gw, *d_ap;
    SP1_TRY(mem.alloc((void**)&d_pv, (n_pv ? n_pv : 1) * 4));
    if (n_pv) SP1_CUDA(cudaMemcpyAsync(d_pv, h_pv, n_pv * 4, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_gw, gw.size() * 16));
    SP1_CUDA(cudaMemcpyAsync(d_gw, gw.data(), gw.size() * 16, cudaMemcpyHostToDevice, st));
    std::vector<E4> gp(mlr);
    for (uint32_t i = 0; i < mlr; i++) gp[i] = E4::load(h_gkr_point + 4 * i);
    // per chip: reversed alpha powers (one upload), state, regions of the two EF ping-pong arenas, slot in the final-values buffer
    std::vector<E4> all_ap; all_ap.reserve(total_c);
    std::vector<size_t> ap_off(nchips), woff(nchips);
    std::vector<uint64_t> boff0(nchips), boff1(nchips);
    uint64_t b0 = 0, b1 = 0; size_t wsum = 0;
    for (size_t k = 0; k < nchips; k++) {
        const ChipProg& p = m->chips[k];
        St& s = S[k];
        s.h = h_heights[k];
        if (s.h > ((uint64_t)1 << mlr)) return sp1b200_set_error("zerocheck: chip %zu height exceeds 2^%u", k, mlr);
        if (p.zc_regs > ZC_GLOBAL_REGS) return sp1b200_set_error("zerocheck: chip %zu needs %u live registers (> %d)", k, p.zc_regs, ZC_GLOBAL_REGS);
        s.zeta = gp;
        std::vector<E4> rev(pw.begin(), pw.begin() + p.n_constraints);
        std::reverse(rev.begin(), rev.end());
        ap_off[k] = all_ap.size();
        all_ap.insert(all_ap.end(), rev.begin(), rev.end());
        if (rev.empty()) all_ap.push_back(E4());
        s.pra = host_eval_zero_row(m->host[k], h_pv, rev, p.n_regs);
        s.vg.threshold = (uint32_t)s.h; s.vg.geq_c = E4::one();
        const uint64_t nh = (s.h + 1) / 2;
        const size_t w = p.main_w + p.prep_w;
        boff0[k] = b0; b0 += (uint64_t)(w + 1) * nh * 4;               // + the pre-batched opening column B (zc_batch0_kernel)
        boff1[k] = b1; b1 += (uint64_t)(w + 1) * ((nh + 1) / 2) * 4;
        woff[k] = wsum; wsum += w;
    }
    SP1_TRY(mem.alloc((void**)&d_ap, all_ap.size() * 16));
    SP1_CUDA(cudaMemcpyAsync(d_ap, all_ap.data(), all_ap.size() * 16, cudaMemcpyHostToDevice, st));
    uint32_t *d_buf[2], *d_final;
    SP1_TRY(mem.alloc((void**)&d_buf[0], b0 * 4 + 16));
    SP1_TRY(mem.alloc((void**)&d_buf[1], b1 * 4 + 16));
    SP1_TRY(mem.alloc((void**)&d_final, (wsum ? wsum : 1) * 16));
    // eq table over the first mlr-1 coordinates of the gkr point, halved every round
    uint32_t *d_point, *d_E[2];
    SP1_TRY(mem.alloc((void**)&d_point, mlr * 16));
    SP1_CUDA(cudaMemcpyAsync(d_point, h_gkr_point, mlr * 16, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_E[0], ((size_t)16 << (mlr - 1))));
    SP1_TRY(mem.alloc((void**)&d_E[1], ((size_t)16 << (mlr > 1 ? mlr - 2 : 0))));
    SP1_LAUNCH(ctx, eq_table_kernel, blocks_for((uint64_t)1 << (mlr - 1)), 256, 0, d_point, (int)mlr - 1, d_E[0]);
    int ecur = 0;

    // ---- the whole launch plan is known up front (heights halve deterministically): job tables of every round, one upload ----
    // tiers of the shared-memory register file (registers per thread); chips above the last tier use the local-memory kernel
    static const uint32_t TIER_REGS[3] = {8, 16, 32};  // x 3 nodes x 16 B x 128 threads = 48 / 96 / 192 KiB per block (EF rounds)
    auto tier_of = [&](uint32_t regs) { for (int t = 0; t < 3; t++) if (regs <= TIER_REGS[t]) return t; return regs <= (uint32_t)ZC_LOCAL_REGS ? 3 : 4; };
    size_t ws_bytes = 0;  // global register-file workspace: worst launch of the last tier (EF rounds: 16 B per register and node)
    struct Launch { size_t job0; uint32_t n_jobs, blocks, regs; int tier; };
    struct RoundPlan { std::vector<Launch> sums; size_t fix0; uint32_t fix_jobs, fix_blocks; std::vector<uint32_t> chip_of_job; size_t job0; };
    std::vector<RoundPlan> plan(mlr);
    std::vector<ZcJob> jobs;
    std::vector<ZcFixJob> fjobs, bjobs;      // bjobs: zc_batch0_kernel (after round 0)
    uint32_t batch_blocks = 0;
    const unsigned MAXB = 148 * 4;
    uint32_t max_blocks = 1, max_jobs = 1;
    {
        std::vector<uint64_t> hcur(nchips);
        for (size_t k = 0; k < nchips; k++) hcur[k] = S[k].h;
        for (uint32_t rd = 0; rd < mlr; rd++) {
            RoundPlan& R = plan[rd];
            R.job0 = jobs.size();
            auto in_main = [&](size_t k) -> const void* {
                if (rd == 0) return d_main[k];
                return (rd & 1 ? d_buf[0] + boff0[k] : d_buf[1] + boff1[k]);
            };
            auto in_prep = [&](size_t k) -> const void* {
                const ChipProg& p = m->chips[k];
                if (rd == 0) return p.prep_w ? d_prep[k] : nullptr;
                // EF arenas: main columns, preprocessed columns, then B - contiguous (also when the chip has no preprocessed column)
                return static_cast<const uint32_t*>(in_main(k)) + (uint64_t)p.main_w * hcur[k] * 4;
            };
            auto in_batch = [&](size_t k) -> const void* {
                if (rd == 0) return nullptr;
                const ChipProg& p = m->chips[k];
                return static_cast<const uint32_t*>(in_main(k)) + (uint64_t)(p.main_w + p.prep_w) * hcur[k] * 4;
            };
            uint32_t blocks_round = 0;
            for (int tier = 0; tier < 5; tier++) {
                Launch Lc{jobs.size(), 0, 0, 0, tier};
                for (size_t k = 0; k < nchips; k++) {
                    const ChipProg& p = m->chips[k];
                    if (!hcur[k] || tier_of(p.zc_regs) != tier) continue;
                    unsigned nb = blocks_for((hcur[k] + 1) / 2, ZC_BLOCK);
                    if (nb > MAXB) nb = MAXB;
                    if (tier == 4 && nb > ZC_GLOBAL_MAXB) nb = ZC_GLOBAL_MAXB;
                    // short rounds: a thread would interpret the whole program for its row pair (hundreds of microseconds for the
                    // wide chips); the self-contained pieces run side by side instead, one job each
                    const auto& pieces = m->host[k].zc_pieces;
                    if (nb <= 16 && !pieces.empty()) {
                        for (size_t q = 0; q < pieces.size(); q++) {
                            ZcJob j{in_main(k), in_prep(k), d_ap + 4 * ap_off[k], hcur[k], Lc.blocks, nb, (uint32_t)k, q == 0 ? 1u : 0u,
                                    pieces[q].first, pieces[q].first + pieces[q].second, in_batch(k)};
                            jobs.push_back(j);
                            R.chip_of_job.push_back((uint32_t)k);
                            Lc.n_jobs++; Lc.blocks += nb;
                        }
                    } else {
                        ZcJob j{in_main(k), in_prep(k), d_ap + 4 * ap_off[k], hcur[k], Lc.blocks, nb, (uint32_t)k, 1u, 0u, p.n_zc, in_batch(k)};
                        jobs.push_back(j);
                        R.chip_of_job.push_back((uint32_t)k);
                        Lc.n_jobs++; Lc.blocks += nb;
                    }
                    Lc.regs = std::max(Lc.regs, p.zc_regs);
                }
                if (Lc.n_jobs) {
                    R.sums.push_back(Lc); blocks_round += Lc.blocks;
                    if (tier == 4) ws_bytes = std::max(ws_bytes, (size_t)Lc.blocks * Lc.regs * 3 * ZC_BLOCK * 16);
                }
            }
            max_blocks = std::max(max_blocks, blocks_round);
            max_jobs = std::max<uint32_t>(max_jobs, (uint32_t)R.chip_of_job.size());
            R.fix0 = fjobs.size(); R.fix_jobs = 0; R.fix_blocks = 0;
            for (size_t k = 0; k < nchips; k++) {
                const ChipProg& p = m->chips[k];
                if (!hcur[k]) continue;
                const uint64_t nh = (hcur[k] + 1) / 2;
                uint32_t* out = rd + 1 == mlr ? d_final + 4 * woff[k] : (rd & 1 ? d_buf[1] + boff1[k] : d_buf[0] + boff0[k]);
                // EF rounds fold the pre-batched column B along with the chip's columns (it sits right after the preprocessed columns, so
                // it is simply one more "preprocessed" column of the fix job); the last round's output is the opened values only
                const uint32_t fold_b = (rd > 0 && rd + 1 < mlr) ? 1u : 0u;
                ZcFixJob f{in_main(k), in_prep(k), out, hcur[k], p.main_w, p.prep_w + fold_b, R.fix_blocks, 0};
                fjobs.push_back(f);
                R.fix_jobs++; R.fix_blocks += blocks_for(nh, 256) * (p.main_w + p.prep_w + fold_b);   // one column per block row (zc_fix_kernel)
                if (rd == 0 && mlr > 1) {   // B of the first EF round, from the base columns
                    ZcFixJob bj{d_main[k], m->chips[k].prep_w ? d_prep[k] : nullptr, d_buf[0] + boff0[k] + (uint64_t)(p.main_w + p.prep_w) * nh * 4, hcur[k],
                                p.main_w, p.prep_w, batch_blocks, 0};
                    bjobs.push_back(bj);
                    batch_blocks += blocks_for(nh, 256);
                }
                hcur[k] = nh;
            }
        }
    }
    ZcJob* d_jobs; ZcFixJob *d_fjobs, *d_bjobs; uint32_t *d_partial, *d_sums;
    SP1_TRY(mem.alloc((void**)&d_jobs, (jobs.size() + 1) * sizeof(ZcJob)));
    SP1_TRY(mem.alloc((void**)&d_fjobs, (fjobs.size() + 1) * sizeof(ZcFixJob)));
    SP1_TRY(mem.alloc((void**)&d_bjobs, (bjobs.size() + 1) * sizeof(ZcFixJob)));
    if (!bjobs.empty()) SP1_CUDA(cudaMemcpyAsync(d_bjobs, bjobs.data(), bjobs.size() * sizeof(ZcFixJob), cudaMemcpyHostToDevice, st));
    if (!jobs.empty()) SP1_CUDA(cudaMemcpyAsync(d_jobs, jobs.data(), jobs.size() * sizeof(ZcJob), cudaMemcpyHostToDevice, st));
    if (!fjobs.empty()) SP1_CUDA(cudaMemcpyAsync(d_fjobs, fjobs.data(), fjobs.size() * sizeof(ZcFixJob), cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_partial, (size_t)max_blocks * 36 * 4));
    if ((size_t)max_jobs * 36 > SP1_MAIL_WORDS) return sp1b200_set_error("zerocheck: %u chips exceed the mailbox payload", max_jobs);
    d_sums = sp1b200_mail_dev(ctx);
    SP1_CUDA(cudaMemsetAsync(d_final, 0, (wsum ? wsum : 1) * 16, st));
    void* d_ws = nullptr;
    if (ws_bytes) SP1_TRY(mem.alloc(&d_ws, ws_bytes));
    auto launch_sum = [&](const Launch& Lc, bool ext, uint32_t* part) -> sp1b200_err {
        auto go = [&](auto kern, size_t smem) -> sp1b200_err {
            // the static reduction buffer counts against the 48 KiB default as well: opt in early
            if (smem > 32 * 1024) SP1_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            SP1_LAUNCH(ctx, kern, Lc.blocks, ZC_BLOCK, smem, d_jobs + Lc.job0, (int)Lc.n_jobs, m->d_chips, d_pv, d_gw, d_E[ecur], part, d_ws,
                       Lc.regs);
            return nullptr;
        };
        if (Lc.tier == 4) return ext ? go(zc_sum_kernel<Ext, RF_GLOBAL, false>, 0) : go(zc_sum_kernel<uint32_t, RF_GLOBAL, true>, 0);
        if (Lc.tier == 3) return ext ? go(zc_sum_kernel<Ext, RF_LOCAL, false>, 0) : go(zc_sum_kernel<uint32_t, RF_LOCAL, true>, 0);
        const size_t regs = Lc.regs;  // the file is sized by the launch's worst chip: regs x 3 nodes x block
        return ext ? go(zc_sum_kernel<Ext, RF_SMEM, false>, regs * 3 * ZC_BLOCK * 16) : go(zc_sum_kernel<uint32_t, RF_SMEM, true>, regs * 3 * ZC_BLOCK * 4);
    };

    t_setup.reset();
    E4 lambda; ch.sample_ext(lambda.c);
    std::vector<E4> round_claims(nchips);
    E4 claimed_sum;
    for (size_t k = 0; k < nchips; k++) { round_claims[k] = E4::load(h_claims + 4 * k); claimed_sum = claimed_sum * lambda + round_claims[k]; }
    SumcheckProof sc;
    std::vector<E4> ys((size_t)nchips * 4);  // per chip: round polynomial values at the nodes 0, 1, 2, 4
    std::vector<uint32_t> hs((size_t)max_jobs * 36);
    std::vector<E4> chip_sums(nchips * 9);
    const E4 two = E4::from_base(hf::to_monty(2)), four = E4::from_base(hf::to_monty(4)), three = E4::from_base(hf::to_monty(3));
    for (uint32_t rd = 0; rd < mlr; rd++) {
        const RoundPlan& R = plan[rd];
        // every chip's partial sums: one launch per register-file tier, one reduction each, one copy back
        {
            uint32_t blk = 0, seq = 0; size_t jb = 0;
            for (const Launch& Lc : R.sums) {
                SP1_TRY(launch_sum(Lc, rd > 0, d_partial + (size_t)blk * 36));
                const Mail mail = sp1b200_mail_next(ctx); seq = mail.seq;
                SP1_LAUNCH(ctx, zc_reduce_kernel, Lc.n_jobs, 128, 0, d_jobs + Lc.job0, d_partial + (size_t)blk * 36, d_sums + jb * 36, mail);
                blk += Lc.blocks; jb += Lc.n_jobs;
            }
            if (jb) {  // launches complete in stream order: the last sequence number covers every tier
                HostSpan sp(acc_wait);
                SP1_TRY(sp1b200_mail_wait(ctx, seq));
                memcpy(hs.data(), sp1b200_mail_host(ctx), jb * 36 * 4);
            }
        }
        HostSpan sp_math(acc_math);
        // a chip's sums = the sums of its jobs (one per piece of its instruction stream)
        std::fill(chip_sums.begin(), chip_sums.end(), E4());
        for (size_t j = 0; j < R.chip_of_job.size(); j++)
            for (int w9 = 0; w9 < 9; w9++) chip_sums[(size_t)R.chip_of_job[j] * 9 + w9] = chip_sums[(size_t)R.chip_of_job[j] * 9 + w9] + E4::load(&hs[j * 36 + 4 * w9]);
        // Every chip's round polynomial goes through the same five nodes {0, 1, 2, 4, b} (b depends only on the shared point),
        // and interpolation is linear: combine the chips' node values with the lambda powers first, interpolate ONCE.
        const E4 last = gp[mlr - 1 - rd];
        const E4 bnode = (E4::one() - last) * hf::inv(E4::one() - (last + last));
        const E4 nodes[5] = {E4(), E4::one(), two, four, bnode};
        E4 basis[5][5];
        hf::lagrange_basis<5>(nodes, basis);
        const E4 f0 = E4::one() - last, f2 = last * hf::to_monty(3) - E4::one(), f4 = last * hf::to_monty(7) - three;
        E4 Y[4];  // lambda-combined values at nodes 0, 1, 2, 4 (the value at b is zero by construction)
        for (size_t k = 0; k < nchips; k++) {
            St& s = S[k];
            E4* y = &ys[4 * k];
            if (s.h == 0) { y[0] = y[1] = y[2] = y[3] = E4(); }
            else {
                // sums: [node][slot] ; y_t = C_t + A + t (B - A) with A, B the opening-batching term at 0 and 1
                const E4* q = &chip_sums[k * 9];
                const E4 A = q[1], B = q[2];
                E4 y0 = q[0] + A;
                E4 y2 = q[3] + (B + B) - A;
                E4 y4 = q[6] + B * four - A * three;
                const uint64_t th = (s.h + 1) / 2 - 1;
                const uint64_t esize = (uint64_t)1 << (s.zeta.size() - 1);
                // E[th] = eq(bits of th, zeta[0 .. len-1)) (most significant bit first): 21 host products instead of a device read + sync
                E4 eth;
                if (th < esize) {
                    const size_t kk = s.zeta.size() - 1;
                    eth = E4::one();
                    for (size_t t = 0; t < kk; t++) eth = eth * (((th >> (kk - 1 - t)) & 1) ? s.zeta[t] : E4::one() - s.zeta[t]);
                }
                const E4 msb = s.eq_adj * eth;
                const E4 v0 = s.vg.fix_last(E4()).at(th), v2 = s.vg.fix_last(two).at(th), v4 = s.vg.fix_last(four).at(th);
                y0 = y0 * (f0 * s.eq_adj) - s.pra * v0 * msb * f0;
                y2 = y2 * (f2 * s.eq_adj) - s.pra * v2 * msb * f2;
                y4 = y4 * (f4 * s.eq_adj) - s.pra * v4 * msb * f4;
                y[0] = y0; y[1] = round_claims[k] - y0; y[2] = y2; y[3] = y4;
            }
            for (int i = 0; i < 4; i++) Y[i] = (k ? Y[i] * lambda : E4()) + y[i];
        }
        E4 rlc[5];
        for (int c5 = 0; c5 < 5; c5++) for (int i = 0; i < 4; i++) rlc[c5] = rlc[c5] + basis[i][c5] * Y[i];
        const E4 a = sc.round(ch, rlc, 5);
        const Ext da = to_ext(a);
        if (R.fix_jobs) {
            if (rd == 0) {
                SP1_LAUNCH(ctx, zc_fix_kernel<uint32_t>, R.fix_blocks, 256, 0, d_fjobs + R.fix0, (int)R.fix_jobs, da);
                if (!bjobs.empty()) SP1_LAUNCH(ctx, zc_batch0_kernel, batch_blocks, 256, 0, d_bjobs, (int)bjobs.size(), d_gw, da);
            } else SP1_LAUNCH(ctx, zc_fix_kernel<Ext>, R.fix_blocks, 256, 0, d_fjobs + R.fix0, (int)R.fix_jobs, da);
        }
        E4 La[4];  // L_i(a) for the four non-zero nodes
        for (int i = 0; i < 4; i++) La[i] = hf::eval_poly<5>(basis[i], a);
        for (size_t k = 0; k < nchips; k++) {
            St& s = S[k];
            const E4* y = &ys[4 * k];
            round_claims[k] = y[0] * La[0] + y[1] * La[1] + y[2] * La[2] + y[3] * La[3];
            s.vg = s.vg.fix_last(a);
            if (s.h == 0) continue;
            s.eq_adj = s.eq_adj * (a * last + (E4::one() - a) * (E4::one() - last));
            s.zeta.pop_back();
            s.h = (s.h + 1) / 2;
        }
        if (rd + 1 < mlr) {
            const uint64_t n_out = (uint64_t)1 << (mlr - 2 - rd);
            SP1_LAUNCH(ctx, halve_eq_kernel, blocks_for(n_out), 256, 0, d_E[ecur], n_out, d_E[ecur ^ 1]);
            ecur ^= 1;
        }
    }
    E4 final_eval;
    for (auto& c : round_claims) final_eval = final_eval * lambda + c;
    std::vector<uint32_t> words;
    sc.emit(words, claimed_sum, final_eval);
    // opened values: one EF row per chip (main columns then preprocessed, zeros for absent chips), fetched with one copy;
    // observed and emitted prep-first as the reference does
    std::vector<uint32_t> fin((wsum ? wsum : 1) * 4);
    SP1_CUDA(cudaMemcpyAsync(fin.data(), d_final, fin.size() * 4, cudaMemcpyDeviceToHost, st));
    SP1_CUDA(cudaStreamSynchronize(st));
    ch.observe(hf::to_monty(nchips));
    for (size_t k = 0; k < nchips; k++) {
        const ChipProg& p = m->chips[k];
        const uint32_t* mv = &fin[4 * woff[k]];
        const uint32_t* pvv = mv + 4 * (size_t)p.main_w;
        ch.observe(hf::to_monty(p.prep_w)); ch.observe_n(pvv, (size_t)p.prep_w * 4);
        ch.observe(hf::to_monty(p.main_w)); ch.observe_n(mv, (size_t)p.main_w * 4);
        words.insert(words.end(), pvv, pvv + (size_t)p.prep_w * 4);
        words.insert(words.end(), mv, mv + (size_t)p.main_w * 4);
    }
    t_all.stop();
    ch.store(h_chal);
    if (h_words) *h_words = words.size();
    if (words.size() > cap) return sp1b200_set_error("zerocheck: output needs %zu words, capacity %llu", words.size(), (unsigned long long)cap);
    if (h_out) memcpy(h_out, words.data(), words.size() * 4);
    return nullptr;
}

}  // extern "C"
