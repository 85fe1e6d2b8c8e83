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
