// Multilinear and sumcheck building blocks shared by the prover phases (pcs.cu, jagged.cu, gkr.cu, zerocheck.cu).
// Everything sits in an anonymous namespace: each translation unit compiles its own internal copy of these kernels, so no
// device code is linked across translation units.
#pragma once
#include "ctx.cuh"
#include "challenger.cuh"
#include "hostfield.hpp"
#include "kb31.cuh"
#include <vector>

namespace {

// E[j] = prod_t (j_t ? x_t : 1 - x_t), point[0] <-> MSB of j
__global__ void eq_table_kernel(const uint32_t* __restrict__ point, int k, uint32_t* __restrict__ E) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ((uint64_t)1 << k)) return;
    kb::Ext acc = kb::ext_one();
    for (int t = 0; t < k; t++) {
        kb::Ext x = kb::ext_load(point + 4 * t);
        bool bit = (j >> (k - 1 - t)) & 1;
        acc = kb::ext_mul(acc, bit ? x : kb::ext_sub(kb::ext_one(), x));
    }
    kb::ext_store(E + 4 * j, acc);
}

// E'[j] = E[2j] + E[2j+1]  (drops the last coordinate of the eq point)
__global__ void halve_eq_kernel(const uint32_t* __restrict__ E, uint64_t n_out, uint32_t* __restrict__ Eo) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_out) return;
    kb::ext_store(Eo + 4 * j, kb::ext_add(kb::ext_load(E + 8 * j), kb::ext_load(E + 8 * j + 4)));
}

// out[j] = in[2j] + alpha (in[2j+1] - in[2j])  (fixes the last variable of a multilinear at alpha)
__global__ void fix_last_kernel(const uint32_t* __restrict__ in, uint64_t n_out, kb::Ext alpha, uint32_t* __restrict__ out) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_out) return;
    const kb::Ext a = kb::ext_load(in + 8 * j), b = kb::ext_load(in + 8 * j + 4);
    kb::ext_store(out + 4 * j, kb::ext_add(a, kb::ext_mul(alpha, kb::ext_sub(b, a))));
}

// Last step of a round kernel: sums the N ext values over the block and posts them to the mailbox payload `partial`
// (4 N words per block) so that the host transcript polls instead of copy + synchronise (ctx.cuh).  Warp shuffles and one
// barrier: the late rounds are latency-bound, where a shared-memory tree would cost eight barriers.
template <int N>
__device__ __forceinline__ void block_post_sums(const kb::Ext (&v)[N], uint32_t* __restrict__ partial, const Mail& mail) {
    __shared__ uint32_t red[4 * N][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t w[4 * N];
#pragma unroll
    for (int i = 0; i < N; i++)
#pragma unroll
        for (int l = 0; l < 4; l++) w[4 * i + l] = v[i].c[l];
#pragma unroll
    for (int k = 0; k < 4 * N; k++) {
        uint32_t x = w[k];
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) x = kb::add(x, __shfl_down_sync(0xffffffffu, x, sft));
        if (lane == 0) red[k][warp] = x;
    }
    __syncthreads();
    if (threadIdx.x < 4 * N) {
        uint32_t x = 0;
        for (int q = 0; q < (int)(blockDim.x >> 5); q++) x = kb::add(x, red[threadIdx.x][q]);
        partial[blockIdx.x * 4 * N + threadIdx.x] = x;
    }
    sp1_mail_done(mail);
}

// index of the job that owns block `blk`: the last one with blk_start <= blk (jobs sorted by blk_start, jobs[0].blk_start = 0)
template <class J>
__device__ __forceinline__ int find_job(const J* __restrict__ jobs, int n, uint32_t blk) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (jobs[mid].blk_start <= blk) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- per-column evaluations of base-field tables: out[c] = sum_{r < rows} eq[r] * col_c[r] -----------------------------------
// A block takes one chunk of COL_EVAL_ROWS rows of one table (column-major), keeps its eq values in registers and walks all the
// table's columns (coalesced column-major reads, 4 products per 64-bit accumulator and reduction); per-column block sums go to
// partial[(blk_of_table)][col], a second launch adds the chunks.
constexpr int COL_EVAL_ROWS_PER_THREAD = 16;
constexpr int COL_EVAL_ROWS = 256 * COL_EVAL_ROWS_PER_THREAD;
struct ColEvalJob { const uint32_t* cols; uint64_t h; uint32_t w, blk_start, nblk, out_col; uint64_t part_off; };

__global__ void __launch_bounds__(256) column_evals_partial_kernel(const ColEvalJob* __restrict__ jobs, int n_jobs, const uint32_t* __restrict__ eq,
                                                                   uint32_t* __restrict__ partial) {
    const ColEvalJob job = jobs[find_job(jobs, n_jobs, blockIdx.x)];
    const uint32_t chunk = blockIdx.x - job.blk_start;
    const uint64_t row0 = (uint64_t)chunk * COL_EVAL_ROWS + threadIdx.x;
    uint4 e[COL_EVAL_ROWS_PER_THREAD];
#pragma unroll
    for (int k = 0; k < COL_EVAL_ROWS_PER_THREAD; k++) {
        const uint64_t r = row0 + (uint64_t)k * 256;
        e[k] = r < job.h ? __ldg(reinterpret_cast<const uint4*>(eq + 4 * r)) : make_uint4(0, 0, 0, 0);
    }
    __shared__ uint32_t red[8][4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* outp = partial + (job.part_off + (uint64_t)chunk * job.w) * 4;
    for (uint32_t c = 0; c < job.w; c++) {
        const uint32_t* col = job.cols + (uint64_t)c * job.h;
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll
        for (int k4 = 0; k4 < COL_EVAL_ROWS_PER_THREAD; k4 += 4) {
            uint64_t s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll
            for (int k = k4; k < k4 + 4; k++) {
                const uint64_t r = row0 + (uint64_t)k * 256;
                const uint32_t x = r < job.h ? __ldg(col + r) : 0u;
                s0 = kb::mac(x, e[k].x, s0); s1 = kb::mac(x, e[k].y, s1); s2 = kb::mac(x, e[k].z, s2); s3 = kb::mac(x, e[k].w, s3);
            }
            a0 = kb::add(a0, kb::monty_reduce2(s0)); a1 = kb::add(a1, kb::monty_reduce2(s1));
            a2 = kb::add(a2, kb::monty_reduce2(s2)); a3 = kb::add(a3, kb::monty_reduce2(s3));
        }
        for (int sft = 16; sft > 0; sft >>= 1) {
            a0 = kb::add(a0, __shfl_down_sync(0xffffffffu, a0, sft)); a1 = kb::add(a1, __shfl_down_sync(0xffffffffu, a1, sft));
            a2 = kb::add(a2, __shfl_down_sync(0xffffffffu, a2, sft)); a3 = kb::add(a3, __shfl_down_sync(0xffffffffu, a3, sft));
        }
        __syncthreads();  // previous column's red[] has been consumed
        if (lane == 0) { red[warp][0] = a0; red[warp][1] = a1; red[warp][2] = a2; red[warp][3] = a3; }
        __syncthreads();
        if (threadIdx.x < 4) {
            uint32_t v = 0;
            for (int w = 0; w < 8; w++) v = kb::add(v, red[w][threadIdx.x]);
            outp[4 * c + threadIdx.x] = v;
        }
    }
}
// out[(job.out_col + c)] = sum over the table's chunks; one block per table, thread -> (column, limb)
__global__ void __launch_bounds__(256) column_evals_reduce_kernel(const ColEvalJob* __restrict__ jobs, const uint32_t* __restrict__ partial,
                                                                  uint32_t* __restrict__ out) {
    const ColEvalJob job = jobs[blockIdx.x];
    for (uint32_t t = threadIdx.x; t < job.w * 4; t += blockDim.x) {
        uint32_t v = 0;
        for (uint32_t b = 0; b < job.nblk; b++) v = kb::add(v, partial[(job.part_off + (uint64_t)b * job.w) * 4 + t]);
        out[(uint64_t)job.out_col * 4 + t] = v;
    }
}

// one table for column_evals: `width` columns of `rows` base-field cells each, column-major at `cols`
struct ColTable { const uint32_t* cols; uint64_t rows; uint32_t width, out_col; };

// d_out[t.out_col + c] = sum_{r < t.rows} d_eq[r] * column c of t, for every table t, in two launches; d_out holds n_cols ext
// elements, and the columns of tables without rows (and any column no table names) are zero.
inline sp1b200_err column_evals(sp1b200_ctx* ctx, DevFree& mem, const std::vector<ColTable>& tables, const uint32_t* d_eq, size_t n_cols,
                                uint32_t* d_out) {
    std::vector<ColEvalJob> jobs;
    uint32_t blk = 0;
    uint64_t part = 0;
    for (const ColTable& t : tables) {
        if (!t.rows) continue;
        const uint32_t nb = (uint32_t)((t.rows + COL_EVAL_ROWS - 1) / COL_EVAL_ROWS);
        jobs.push_back(ColEvalJob{t.cols, t.rows, t.width, blk, nb, t.out_col, part});
        blk += nb; part += (uint64_t)nb * t.width;
    }
    SP1_CUDA(cudaMemsetAsync(d_out, 0, n_cols * 16, ctx->stream));
    if (jobs.empty()) return nullptr;
    ColEvalJob* d_jobs;
    uint32_t* d_part;
    SP1_TRY(mem.alloc((void**)&d_jobs, jobs.size() * sizeof(ColEvalJob)));
    SP1_TRY(mem.alloc((void**)&d_part, part * 16));
    SP1_CUDA(cudaMemcpyAsync(d_jobs, jobs.data(), jobs.size() * sizeof(ColEvalJob), cudaMemcpyHostToDevice, ctx->stream));
    SP1_LAUNCH(ctx, column_evals_partial_kernel, blk, 256, 0, d_jobs, (int)jobs.size(), d_eq, d_part);
    SP1_LAUNCH(ctx, column_evals_reduce_kernel, (unsigned)jobs.size(), 256, 0, d_jobs, d_part, d_out);
    return nullptr;
}

// host side of block_post_sums: waits for the launch with sequence number `seq` and adds up its nblk blocks
template <int N>
sp1b200_err mail_sums(sp1b200_ctx* ctx, uint32_t seq, unsigned nblk, hf::E4 (&out)[N]) {
    SP1_TRY(sp1b200_mail_wait(ctx, seq));
    const uint32_t* h = sp1b200_mail_host(ctx);
    for (hf::E4& x : out) x = hf::E4();
    for (unsigned k = 0; k < nblk; k++)
        for (int i = 0; i < N; i++) out[i] = out[i] + hf::E4::load(&h[4 * (N * k + i)]);
    return nullptr;
}

inline kb::Ext to_ext(const hf::E4& e) { return kb::Ext{{e.c[0], e.c[1], e.c[2], e.c[3]}}; }

// Transcript side of one sumcheck and its proof words, PartialSumcheckProof (slop/crates/sumcheck/src/proof.rs):
//   n_polys | per round {n_coeffs, coeffs} | claimed_sum | point (most recent challenge first) | eval
// The caller computes each round polynomial and the claim it implies at the returned challenge.
struct SumcheckProof {
    std::vector<uint32_t> polys;
    std::vector<hf::E4> point;

    // observes the round polynomial, records it, samples the round's challenge and returns it
    hf::E4 round(HostChallenger& ch, const hf::E4* coeffs, int n) {
        for (int i = 0; i < n; i++) ch.observe_n(coeffs[i].c, 4);
        polys.push_back((uint32_t)n);
        for (int i = 0; i < n; i++) polys.insert(polys.end(), coeffs[i].c, coeffs[i].c + 4);
        hf::E4 alpha;
        ch.sample_ext(alpha.c);
        point.insert(point.begin(), alpha);
        return alpha;
    }
    void emit(std::vector<uint32_t>& out, const hf::E4& claimed_sum, const hf::E4& eval) const {
        out.push_back((uint32_t)point.size());
        out.insert(out.end(), polys.begin(), polys.end());
        out.insert(out.end(), claimed_sum.c, claimed_sum.c + 4);
        for (const hf::E4& x : point) out.insert(out.end(), x.c, x.c + 4);
        out.insert(out.end(), eval.c, eval.c + 4);
    }
};

}  // namespace
