// Stacked PCS + BaseFold prover on the device.
// Reference behaviour: slop/crates/stacked/src/prover.rs:59-160 (commit, batch evaluations),
// slop/crates/basefold-prover/src/prover.rs:102-270 (protocol), fri.rs:30-168 (batch, commit_phase_round),
// slop/crates/multilinear/src/{fold.rs:12-26, restrict.rs:75-87, lagrange.rs:19-45};
// the GPU twin it replaces: sp1-gpu/crates/basefold/src/fri.rs:117-477 + sys/lib/basefold/basefold.cu.
// Differences in HOW (results identical): the batched codeword is kept limb-major ([4][m], so FRI leaves are
// read with coalesced 8-byte loads and no transposeEvenOdd pass), the codeword is folded directly (p3
// fold_even_odd rule, pinned by slop/crates/basefold/src/verifier.rs:309-386) instead of re-encoding the folded
// MLE each round, the eq table for fixed_at_zero is built once and halved per round, and the PoW witnesses are
// the deterministic minimum (or replayed).
#include "sumcheck.cuh"
#include "poseidon2.cuh"
#include <array>
#include <memory>
#include <vector>

struct sp1b200_commit {
    uint64_t ncols = 0;
    uint32_t log_h = 0, log_blowup = 0;
    uint32_t* d_mles = nullptr;      // [ncols x 2^log_h], owned copy if owns_mles
    bool owns_mles = false;
    uint32_t* d_codeword = nullptr;  // [ncols x 2^(log_h+log_blowup)] or NULL (recomputed on demand)
    uint32_t* d_layers = nullptr;    // (2^(log_h+log_blowup+1) - 1) digests
    uint32_t root[8], commit[8];
};

namespace {

using kb::Ext;

__device__ __forceinline__ uint32_t root_pow(const uint32_t* __restrict__ TH, const uint32_t* __restrict__ TL, uint32_t e) {
    uint32_t hi = __ldg(TH + (e >> 12));
    uint32_t lo = e & 4095u;
    return lo ? kb::mul(hi, __ldg(TL + lo)) : hi;
}

// out[i] (+)= sum_c coeff[c] * cols[c][i]   ; out as Ext AoS [h]
__global__ void __launch_bounds__(256) batch_columns_kernel(const uint32_t* __restrict__ cols, uint64_t ncols, uint64_t h,
                                                            const uint32_t* __restrict__ coeffs, uint32_t* __restrict__ out,
                                                            int accumulate) {
    extern __shared__ uint32_t scoef[];
    for (uint64_t t = threadIdx.x; t < ncols * 4; t += blockDim.x) scoef[t] = coeffs[t];
    __syncthreads();
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h) return;
    uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    if (accumulate) { uint4 v = *reinterpret_cast<const uint4*>(out + 4 * i); a0 = v.x; a1 = v.y; a2 = v.z; a3 = v.w; }
    const uint32_t* p = cols + i;
    uint64_t c = 0;
    // two products (< 2^62 each) fit a 64-bit accumulator before one Montgomery reduction
    for (; c + 2 <= ncols; c += 2) {
        uint32_t x = __ldg(p + c * h), y = __ldg(p + (c + 1) * h);
        const uint32_t* k0 = scoef + 4 * c;
        a0 = kb::add(a0, kb::monty_reduce2((uint64_t)x * k0[0] + (uint64_t)y * k0[4]));
        a1 = kb::add(a1, kb::monty_reduce2((uint64_t)x * k0[1] + (uint64_t)y * k0[5]));
        a2 = kb::add(a2, kb::monty_reduce2((uint64_t)x * k0[2] + (uint64_t)y * k0[6]));
        a3 = kb::add(a3, kb::monty_reduce2((uint64_t)x * k0[3] + (uint64_t)y * k0[7]));
    }
    if (c < ncols) {
        uint32_t x = __ldg(p + c * h);
        const uint32_t* k0 = scoef + 4 * c;
        a0 = kb::add(a0, kb::mul(x, k0[0])); a1 = kb::add(a1, kb::mul(x, k0[1]));
        a2 = kb::add(a2, kb::mul(x, k0[2])); a3 = kb::add(a3, kb::mul(x, k0[3]));
    }
    *reinterpret_cast<uint4*>(out + 4 * i) = make_uint4(a0, a1, a2, a3);
}

// Ext AoS [h] -> limb-major [4][h]
__global__ void split_limbs_kernel(const uint32_t* __restrict__ aos, uint64_t h, uint32_t* __restrict__ limbs) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h) return;
    uint4 v = *reinterpret_cast<const uint4*>(aos + 4 * i);
    limbs[i] = v.x; limbs[h + i] = v.y; limbs[2 * h + i] = v.z; limbs[3 * h + i] = v.w;
}

// partial[blk] = sum_j E[j] * mle[2j]   (Ext x Ext), j < n
__global__ void __launch_bounds__(256) dot_even_kernel(const uint32_t* __restrict__ E, const uint32_t* __restrict__ mle, uint64_t n,
                                                       uint32_t* __restrict__ partial) {
    Ext acc = kb::ext_zero();
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (uint64_t)gridDim.x * blockDim.x) {
        Ext e = kb::ext_load(E + 4 * j);
        Ext m = kb::ext_load(mle + 8 * j);
        acc = kb::ext_add(acc, kb::ext_mul(e, m));
    }
    block_post_sums<1>({acc}, partial, Mail{});  // the FRI tree launch that follows posts the round's mail
}

// mle'[j] = mle[2j] + beta * mle[2j+1]
__global__ void fold_mle_kernel(const uint32_t* __restrict__ mle, uint64_t n_out, Ext beta, uint32_t* __restrict__ out) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_out) return;
    Ext a = kb::ext_load(mle + 8 * j), b = kb::ext_load(mle + 8 * j + 4);
    kb::ext_store(out + 4 * j, kb::ext_add(a, kb::ext_mul(beta, b)));
}

// limb-major codeword [4][m] -> folded [4][m/2]:
// f[i] = (e0 + e1)/2 + beta * (e0 - e1) / (2 x_i),  x_i = g^{bitrev(i, log_m - 1)},  g of order m = 2^log_m
__global__ void fold_codeword_kernel(const uint32_t* __restrict__ cw, int log_m, Ext beta_half, uint32_t half,
                                     const uint32_t* __restrict__ TH, const uint32_t* __restrict__ TL, uint32_t* __restrict__ out) {
    const uint64_t m = (uint64_t)1 << log_m, mo = m >> 1;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= mo) return;
    Ext e0, e1;
#pragma unroll
    for (int l = 0; l < 4; l++) {
        uint2 v = *reinterpret_cast<const uint2*>(cw + l * m + 2 * i);
        e0.c[l] = v.x; e1.c[l] = v.y;
    }
    uint32_t br = log_m > 1 ? (__brev((uint32_t)i) >> (32 - (log_m - 1))) : 0;
    // x_i^-1 = w24^( -(br << (24 - log_m)) )
    uint32_t e = (0x1000000u - (br << (24 - log_m))) & 0xffffffu;
    uint32_t xinv = root_pow(TH, TL, e);
    Ext s = kb::ext_mul_base(kb::ext_add(e0, e1), half);
    Ext d = kb::ext_mul_base(kb::ext_sub(e0, e1), xinv);
    Ext f = kb::ext_add(s, kb::ext_mul(beta_half, d));
#pragma unroll
    for (int l = 0; l < 4; l++) out[l * mo + i] = f.c[l];
}

// values[q][c] = codeword[c][idx[q]]
__global__ void gather_columns_kernel(const uint32_t* __restrict__ cw, uint64_t ncols, uint64_t M, const uint32_t* __restrict__ idx,
                                      uint32_t nq, uint32_t* __restrict__ out) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)nq * ncols) return;
    uint32_t q = (uint32_t)(t / ncols);
    uint64_t c = t - (uint64_t)q * ncols;
    out[t] = cw[c * M + idx[q]];
}

// paths[q][k] = layer_k[(idx[q] >> k) ^ 1]
__global__ void gather_paths_kernel(const uint32_t* __restrict__ layers, uint32_t log_h, const uint32_t* __restrict__ idx, uint32_t nq,
                                    uint32_t* __restrict__ out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq * log_h * 8) return;
    uint32_t w = t & 7, k = (t >> 3) % log_h, q = (t >> 3) / log_h;
    uint64_t off = ((uint64_t)2 << log_h) - ((uint64_t)2 << (log_h - k));  // digests before layer k
    out[t] = layers[(off + ((idx[q] >> k) ^ 1)) * 8 + w];
}

// values[q][0..8) = (cw[2 idx] limbs, cw[2 idx + 1] limbs)
__global__ void gather_fri_values_kernel(const uint32_t* __restrict__ cw, uint64_t m, const uint32_t* __restrict__ idx, uint32_t nq,
                                         uint32_t* __restrict__ out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq * 8) return;
    uint32_t q = t >> 3, w = t & 7;
    out[t] = cw[(w & 3) * m + 2 * (uint64_t)idx[q] + (w >> 2)];
}

}  // namespace

extern "C" {

sp1b200_err sp1b200_stacked_commit(sp1b200_ctx* ctx, const uint32_t* dense_any, uint64_t ncols, int keep_codeword,
                                   uint32_t* h_commit8, sp1b200_commit** out) { SP1_DEVICE_GUARD(ctx);
    if (!ncols) return sp1b200_set_error("stacked_commit: ncols == 0");
    const uint32_t log_h = ctx->params.log_stacking_height, b = ctx->params.log_blowup;
    const size_t n = (size_t)ncols << log_h, M = n << b;
    auto c = std::make_unique<sp1b200_commit>();
    c->ncols = ncols; c->log_h = log_h; c->log_blowup = b;
    if (sp1b200_is_device_ptr(dense_any)) {
        c->d_mles = const_cast<uint32_t*>(dense_any);  // borrowed: caller keeps the trace resident (reference: main_virtual_tensor)
    } else {
        SP1_CUDA(cudaMallocFromPoolAsync((void**)&c->d_mles, n * sizeof(uint32_t), ctx->pool, ctx->stream));
        c->owns_mles = true;
        SP1_CUDA(cudaMemcpyAsync(c->d_mles, dense_any, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    }
    SP1_CUDA(cudaMallocFromPoolAsync((void**)&c->d_codeword, M * sizeof(uint32_t), ctx->pool, ctx->stream));
    const size_t nd = ((size_t)2 << (log_h + b)) - 1;
    SP1_CUDA(cudaMallocFromPoolAsync((void**)&c->d_layers, nd * 8 * sizeof(uint32_t), ctx->pool, ctx->stream));
    uint32_t* d_rc;
    SP1_CUDA(cudaMallocFromPoolAsync((void**)&d_rc, 64, ctx->pool, ctx->stream));
    {
        PhaseTimer t(ctx, "commit.rs_encode");
        SP1_TRY(sp1b200_rs_encode_device(ctx, c->d_mles, ncols, log_h, b, c->d_codeword));
        t.stop();
    }
    {
        PhaseTimer t(ctx, "commit.merkle");
        SP1_TRY(sp1b200_merkle_commit_device(ctx, c->d_codeword, ncols, log_h + b, c->d_layers, d_rc));
        t.stop();
    }
    uint32_t rc[16];
    SP1_CUDA(cudaMemcpyAsync(rc, d_rc, 64, cudaMemcpyDeviceToHost, ctx->stream));
    SP1_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFreeAsync(d_rc, ctx->stream);
    memcpy(c->root, rc, 32); memcpy(c->commit, rc + 8, 32);
    if (!keep_codeword) { cudaFreeAsync(c->d_codeword, ctx->stream); c->d_codeword = nullptr; }
    if (h_commit8) memcpy(h_commit8, c->commit, 32);
    *out = c.release();
    return nullptr;
}

void sp1b200_commit_free(sp1b200_ctx* ctx, sp1b200_commit* c) { SP1_DEVICE_GUARD(ctx);
    if (!c) return;
    if (c->owns_mles) cudaFreeAsync(c->d_mles, ctx->stream);
    if (c->d_codeword) cudaFreeAsync(c->d_codeword, ctx->stream);
    if (c->d_layers) cudaFreeAsync(c->d_layers, ctx->stream);
    delete c;
}

sp1b200_err sp1b200_stacked_prove(sp1b200_ctx* ctx, sp1b200_commit* const* rounds, uint32_t n_rounds, const uint32_t* h_point,
                                  uint32_t n_point, const uint32_t* h_replay, uint32_t* h_chal, uint32_t* h_proof,
                                  uint64_t cap, uint64_t* h_words) { SP1_DEVICE_GUARD(ctx);
    using hf::E4;
    if (!n_rounds) return sp1b200_set_error("stacked_prove: no rounds");
    const uint32_t log_h = rounds[0]->log_h, b = rounds[0]->log_blowup;
    for (uint32_t r = 0; r < n_rounds; r++)
        if (rounds[r]->log_h != log_h || rounds[r]->log_blowup != b) return sp1b200_set_error("stacked_prove: inconsistent rounds");
    if (n_point < log_h) return sp1b200_set_error("stacked_prove: point has %u < %u coordinates", n_point, log_h);
    if (log_h == 0) return sp1b200_set_error("stacked_prove: log_stacking_height 0 unsupported");
    const bool replay = ctx->params.grind_mode == 1;
    if (replay && !h_replay) return sp1b200_set_error("stacked_prove: grind_mode=replay needs witnesses");
    const uint64_t h = (uint64_t)1 << log_h, M = h << b;
    const uint32_t nq = ctx->params.num_queries;
    cudaStream_t st = ctx->stream;
    DevFree mem(ctx);
    HostChallenger ch;
    SP1_TRY(ch.init(ctx, h_chal));
    std::vector<uint32_t> proof;
    auto put = [&](const uint32_t* p, size_t n) { proof.insert(proof.end(), p, p + n); };

    // stack point (last log_h coordinates) on device + eq table
    uint32_t *d_point, *d_E, *d_E2;
    SP1_TRY(mem.alloc((void**)&d_point, log_h * 16));
    SP1_CUDA(cudaMemcpyAsync(d_point, h_point + 4 * (n_point - log_h), log_h * 16, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_E, h * 16));
    SP1_TRY(mem.alloc((void**)&d_E2, (h / 2) * 16));
    PhaseTimer t_all(ctx, "open.total");
    SP1_LAUNCH(ctx, eq_table_kernel, blocks_for(h), 256, 0, d_point, (int)log_h, d_E);

    // ---- stacked layer: per-column evaluations at the stack point (batch_evaluations) -------------------------
    uint64_t total_cols = 0;
    for (uint32_t r = 0; r < n_rounds; r++) total_cols += rounds[r]->ncols;
    std::vector<uint32_t> evals(total_cols * 4);
    {
        std::vector<ColTable> tables;
        uint64_t off = 0;
        for (uint32_t r = 0; r < n_rounds; r++) {
            tables.push_back(ColTable{rounds[r]->d_mles, h, (uint32_t)rounds[r]->ncols, (uint32_t)off});
            off += rounds[r]->ncols;
        }
        uint32_t* d_ev;
        SP1_TRY(mem.alloc((void**)&d_ev, total_cols * 16));
        SP1_TRY(column_evals(ctx, mem, tables, d_E, total_cols, d_ev));
        SP1_CUDA(cudaMemcpyAsync(evals.data(), d_ev, total_cols * 16, cudaMemcpyDeviceToHost, st));
        SP1_CUDA(cudaStreamSynchronize(st));
    }
    // prove_untrusted_evaluations: observe every claim
    ch.observe_n(evals.data(), evals.size());

    // ---- BaseFold ---------------------------------------------------------------------------------------------
    uint32_t batch_w, pow_w;
    if (replay) {
        batch_w = h_replay[0];
        if (!ch.check_witness(ctx->params.batch_pow_bits, batch_w)) return sp1b200_set_error("stacked_prove: replayed batch witness invalid");
    } else SP1_TRY(ch.grind(ctx->params.batch_pow_bits, &batch_w));

    const unsigned nb = hf::log2_ceil(total_cols);
    std::vector<E4> bp(nb);
    for (auto& x : bp) ch.sample_ext(x.c);
    std::vector<E4> coeffs = hf::partial_lagrange(bp);
    E4 claim;
    for (uint64_t c = 0; c < total_cols; c++) claim = claim + E4::load(&evals[4 * c]) * coeffs[c];

    uint32_t *d_coef, *d_mle, *d_mle2, *d_limbs;
    SP1_TRY(mem.alloc((void**)&d_coef, total_cols * 16));
    SP1_CUDA(cudaMemcpyAsync(d_coef, coeffs.data(), total_cols * 16, cudaMemcpyHostToDevice, st));
    SP1_TRY(mem.alloc((void**)&d_mle, h * 16));
    SP1_TRY(mem.alloc((void**)&d_mle2, (h / 2) * 16));
    SP1_TRY(mem.alloc((void**)&d_limbs, h * 16));
    {
        PhaseTimer t(ctx, "open.batch");
        uint64_t off = 0;
        for (uint32_t r = 0; r < n_rounds; r++) {
            // columns are processed in groups so that the coefficient slice fits shared memory
            for (uint64_t c0 = 0; c0 < rounds[r]->ncols; c0 += 2048) {
                uint64_t nc = rounds[r]->ncols - c0 < 2048 ? rounds[r]->ncols - c0 : 2048;
                SP1_LAUNCH(ctx, batch_columns_kernel, blocks_for(h), 256, nc * 16, rounds[r]->d_mles + c0 * h, nc, h,
                           d_coef + (off + c0) * 4, d_mle, (int)(r > 0 || c0 > 0));
            }
            off += rounds[r]->ncols;
        }
        t.stop();
    }
    SP1_LAUNCH(ctx, split_limbs_kernel, blocks_for(h), 256, 0, d_mle, h, d_limbs);
    // codewords of all fold rounds, limb-major, back to back: sizes M, M/2, ..., 4  (4 limbs each)
    uint32_t* d_cw_all;
    SP1_TRY(mem.alloc((void**)&d_cw_all, 2 * M * 16));
    SP1_TRY(sp1b200_rs_encode_device(ctx, d_limbs, 4, log_h, b, d_cw_all));
    // digest layers of all fold-round trees: round r has M >> (r+1) leaves
    uint32_t* d_trees;
    SP1_TRY(mem.alloc((void**)&d_trees, 2 * M * 32));

    uint32_t d_h = hf::to_monty(log_h);
    ch.observe(d_h);
    std::vector<E4> point(log_h);
    for (uint32_t i = 0; i < log_h; i++) point[i] = E4::load(h_point + 4 * (n_point - log_h + i));
    const uint32_t half = hf::inv(hf::to_monty(2));
    std::vector<uint32_t> uni;                      // univariate messages
    std::vector<uint32_t> fri_commits;              // d x 8
    std::vector<uint32_t*> cw_ptr(log_h + 1), tree_ptr(log_h);
    std::vector<std::array<uint32_t, 8>> fri_roots(log_h);
    uint32_t *d_part, *d_rc;
    SP1_TRY(mem.alloc((void**)&d_part, 1024 * 16));
    SP1_TRY(mem.alloc((void**)&d_rc, 64));
    uint32_t *cur_mle = d_mle, *nxt_mle = d_mle2, *cur_E = d_E, *nxt_E = d_E2;
    {
        uint64_t off = 0, toff = 0;
        for (uint32_t r = 0; r <= log_h; r++) { cw_ptr[r] = d_cw_all + off; off += 4 * (M >> r); }
        for (uint32_t r = 0; r < log_h; r++) { tree_ptr[r] = d_trees + toff; toff += 8 * (((uint64_t)2 * (M >> (r + 1))) - 1); }
    }
    PhaseTimer t_fri(ctx, "open.fri_rounds");
    for (uint32_t r = 0; r < log_h; r++) {
        const uint64_t n_cur = h >> r;         // current mle length
        const uint64_t m_cur = M >> r;         // current codeword length
        const E4 last = point.back();
        point.pop_back();
        // E for the remaining point: halve (E_{k} -> E_{k-1})
        SP1_LAUNCH(ctx, halve_eq_kernel, blocks_for(n_cur / 2), 256, 0, cur_E, n_cur / 2, nxt_E);
        std::swap(cur_E, nxt_E);
        unsigned nblk = (unsigned)((n_cur / 2 + 255) / 256);
        if (nblk > 1024) nblk = 1024;
        // the round's two results travel through the mailbox: payload [0,16) root + commitment, [16, 16 + 4 nblk) dot partials
        uint32_t* mail_dev = sp1b200_mail_dev(ctx);
        SP1_LAUNCH(ctx, dot_even_kernel, nblk, 256, 0, cur_E, cur_mle, n_cur / 2, mail_dev + 16);
        // leaves + tree of the current codeword: leaf hashing fused into the first subtree launch, <= 3 launches per tree
        const uint32_t log_leaves = log_h + b - r - 1;
        const Mail mail = sp1b200_mail_next(ctx);
        SP1_TRY(sp1b200_fri_tree_device(ctx, cw_ptr[r], m_cur, tree_ptr[r], log_leaves, mail_dev, mail));
        SP1_TRY(sp1b200_mail_wait(ctx, mail.seq));
        const uint32_t* mh = sp1b200_mail_host(ctx);
        uint32_t rc[16];
        memcpy(rc, mh, 64);
        std::vector<uint32_t> parts(mh + 16, mh + 16 + (size_t)nblk * 4);
        E4 zero_val;
        for (unsigned k = 0; k < nblk; k++) zero_val = zero_val + E4::load(&parts[4 * k]);
        E4 one_val = (claim - zero_val) * hf::inv(last) + zero_val;
        uni.insert(uni.end(), zero_val.c, zero_val.c + 4);
        uni.insert(uni.end(), one_val.c, one_val.c + 4);
        ch.observe_n(zero_val.c, 4); ch.observe_n(one_val.c, 4);
        ch.observe_n(rc + 8, 8);
        fri_commits.insert(fri_commits.end(), rc + 8, rc + 16);
        memcpy(fri_roots[r].data(), rc, 32);
        E4 beta; ch.sample_ext(beta.c);
        SP1_LAUNCH(ctx, fold_codeword_kernel, blocks_for(m_cur / 2), 256, 0, cw_ptr[r], (int)(log_h + b - r), to_ext(beta * half), half,
                   ctx->d_TH, ctx->d_TL, cw_ptr[r + 1]);
        SP1_LAUNCH(ctx, fold_mle_kernel, blocks_for(n_cur / 2), 256, 0, cur_mle, n_cur / 2, to_ext(beta), nxt_mle);
        std::swap(cur_mle, nxt_mle);
        claim = zero_val + beta * one_val;
    }
    // final_poly = codeword[0] of the last (length 2^b) codeword, limb-major with stride 2^b
    uint32_t fin[4];
    {
        std::vector<uint32_t> lastcw(4 << b);
        SP1_CUDA(cudaMemcpyAsync(lastcw.data(), cw_ptr[log_h], (4 << b) * 4, cudaMemcpyDeviceToHost, st));
        SP1_CUDA(cudaStreamSynchronize(st));
        for (int l = 0; l < 4; l++) fin[l] = lastcw[(size_t)l << b];
    }
    t_fri.stop();
    ch.observe_n(fin, 4);
    if (replay) {
        pow_w = h_replay[1];
        if (!ch.check_witness(ctx->params.pow_bits, pow_w)) return sp1b200_set_error("stacked_prove: replayed pow witness invalid");
    } else SP1_TRY(ch.grind(ctx->params.pow_bits, &pow_w));
    std::vector<uint32_t> idx(nq);
    for (auto& q : idx) q = ch.sample_bits(log_h + b);

    // ---- assemble: univariate messages, fri commitments -----------------------------------------------------------
    put(uni.data(), uni.size());
    put(fri_commits.data(), fri_commits.size());

    // ---- query phase -------------------------------------------------------------------------------------------------
    PhaseTimer t_q(ctx, "open.queries");
    uint32_t* d_idx;
    SP1_TRY(mem.alloc((void**)&d_idx, nq * 4));
    SP1_CUDA(cudaMemcpyAsync(d_idx, idx.data(), nq * 4, cudaMemcpyHostToDevice, st));
    const uint32_t LH = log_h + b;
    for (uint32_t r = 0; r < n_rounds; r++) {
        sp1b200_commit* c = rounds[r];
        uint32_t* cw = c->d_codeword;
        DevFree tmp(ctx);
        if (!cw) {  // recompute (drop_ldes)
            SP1_TRY(tmp.alloc((void**)&cw, (c->ncols << LH) * 4));
            SP1_TRY(sp1b200_rs_encode_device(ctx, c->d_mles, c->ncols, log_h, b, cw));
        }
        uint32_t *d_vals, *d_paths;
        SP1_TRY(tmp.alloc((void**)&d_vals, nq * c->ncols * 4));
        SP1_TRY(tmp.alloc((void**)&d_paths, (size_t)nq * LH * 32));
        SP1_LAUNCH(ctx, gather_columns_kernel, blocks_for(nq * c->ncols), 256, 0, cw, c->ncols, M, d_idx, nq, d_vals);
        SP1_LAUNCH(ctx, gather_paths_kernel, blocks_for((uint64_t)nq * LH * 8), 256, 0, c->d_layers, LH, d_idx, nq, d_paths);
        std::vector<uint32_t> vals(nq * c->ncols), paths((size_t)nq * LH * 8);
        SP1_CUDA(cudaMemcpyAsync(vals.data(), d_vals, vals.size() * 4, cudaMemcpyDeviceToHost, st));
        SP1_CUDA(cudaMemcpyAsync(paths.data(), d_paths, paths.size() * 4, cudaMemcpyDeviceToHost, st));
        SP1_CUDA(cudaStreamSynchronize(st));
        put(vals.data(), vals.size());
        put(c->root, 8);
        uint32_t meta[2] = {LH, (uint32_t)c->ncols};
        put(meta, 2);
        put(paths.data(), paths.size());
    }
    for (uint32_t r = 0; r < log_h; r++) {
        for (auto& q : idx) q >>= 1;
        SP1_CUDA(cudaMemcpyAsync(d_idx, idx.data(), nq * 4, cudaMemcpyHostToDevice, st));
        const uint32_t lh = LH - r - 1;
        DevFree tmp(ctx);
        uint32_t *d_vals, *d_paths;
        SP1_TRY(tmp.alloc((void**)&d_vals, nq * 32));
        SP1_TRY(tmp.alloc((void**)&d_paths, (size_t)nq * (lh ? lh : 1) * 32));
        SP1_LAUNCH(ctx, gather_fri_values_kernel, blocks_for(nq * 8), 256, 0, cw_ptr[r], M >> r, d_idx, nq, d_vals);
        if (lh) SP1_LAUNCH(ctx, gather_paths_kernel, blocks_for((uint64_t)nq * lh * 8), 256, 0, tree_ptr[r], lh, d_idx, nq, d_paths);
        std::vector<uint32_t> vals(nq * 8), paths((size_t)nq * lh * 8);
        SP1_CUDA(cudaMemcpyAsync(vals.data(), d_vals, vals.size() * 4, cudaMemcpyDeviceToHost, st));
        if (lh) SP1_CUDA(cudaMemcpyAsync(paths.data(), d_paths, paths.size() * 4, cudaMemcpyDeviceToHost, st));
        SP1_CUDA(cudaStreamSynchronize(st));
        put(vals.data(), vals.size());
        put(fri_roots[r].data(), 8);
        uint32_t meta[2] = {lh, 8};
        put(meta, 2);
        put(paths.data(), paths.size());
    }
    t_q.stop();
    put(fin, 4);
    put(&pow_w, 1);
    put(&batch_w, 1);
    put(evals.data(), evals.size());
    t_all.stop();

    ch.store(h_chal);
    if (h_words) *h_words = proof.size();
    if (proof.size() > cap) return sp1b200_set_error("stacked_prove: proof needs %zu words, capacity %llu", proof.size(), (unsigned long long)cap);
    if (h_proof) memcpy(h_proof, proof.data(), proof.size() * 4);
    return nullptr;
}

}  // extern "C"
