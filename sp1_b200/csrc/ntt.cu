// Reed-Solomon encode of stacked trace columns: zero-pad x 2^b, forward DFT over the 2^(L+b)-th roots,
// output rows bit-reversed.  Replaces the per-column host loop of batch_coset_dft
// (sp1-gpu/crates/sys/include/ntt/sppark.cuh:49-107: bit-reverse, LDE-spread, 3 CT steps, bit-reverse again,
// ~6 launches per column) with a batched two-step decimation-in-frequency transform that never
// materialises the zero padding and needs no bit-reversal pass:
//
//   input index j = hi * 2^L2 + lo,   frequency k = k_a + 2^(L1+b) * k_b,   k_a = k1 * 2^b + r
//   step A:  Y[q][lo]  = sum_hi (x[hi,lo] * zeta^(hi r)) * theta^(hi k1)       (size-2^L1 DIF per coset r)
//            row q = bitrev_b(r) * 2^L1 + bitrev_L1(k1) = bitrev_(L1+b)(k_a)
//   step B:  Z[q][.]   = DIF_2^L2( Y[q][lo] * omega^(lo k_a) )  in place         (contiguous rows)
//   output index bitrev_(L+b)(k) = q * 2^L2 + bitrev_L2(k_b)  -- exactly the reference's bit-reversed order
//   (slop/crates/dft/src/p3.rs:27-48, slop/crates/basefold/src/verifier.rs:320-326).
//
// Step B runs in place on the step-A output of the same column group while it is still L2-resident
// (B200: 126 MB L2; one 2^23-row column is 32 MB), so the intermediate never costs an HBM round trip.
#include "ctx.cuh"
#include "kb31.cuh"

namespace {

__device__ __forceinline__ uint32_t root_pow(const uint32_t* __restrict__ TH, const uint32_t* __restrict__ TL, uint32_t e) {
    uint32_t hi = __ldg(TH + (e >> 12));
    uint32_t lo = e & 4095u;
    return lo ? kb::mul(hi, __ldg(TL + lo)) : hi;
}

__global__ void init_tables_kernel(uint32_t* TH, uint32_t* TL) {
    // w = 3^127 generates the 2^24-th roots (sppark/ntt/parameters/koala_bear.h:5-36, checked in tests)
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 4096) return;
    uint32_t w = kb::pow(kb::to_monty_c(3), 127);
    TL[i] = kb::pow(w, i);
    TH[i] = kb::pow(w, (uint64_t)i << 12);
}

// ---- generic step A: coset expansion + size-2^L1 DIF over the strided (hi) axis ---------------------------
// grid (2^L2 / T, ncols), dynamic smem 2^L1 * T words
__global__ void rs_step_a_generic(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int L1, int L2, int b, int T,
                                  const uint32_t* __restrict__ TH, const uint32_t* __restrict__ TL) {
    extern __shared__ uint32_t sm[];
    const int L = L1 + L2;
    const size_t n = (size_t)1 << L, M = n << b;
    const uint32_t* col_in = in + (size_t)blockIdx.y * n;
    uint32_t* col_out = out + (size_t)blockIdx.y * M;
    const uint32_t lo0 = blockIdx.x * T;
    const int H = 1 << L1;
    const int tile = H * T;
    for (int r = 0; r < (1 << b); r++) {
        const uint32_t rr = __brev((uint32_t)r) >> (32 - b);
        for (int idx = threadIdx.x; idx < tile; idx += blockDim.x) {
            int hi = idx / T, lo = idx - hi * T;
            uint32_t x = col_in[((size_t)hi << L2) + lo0 + lo];
            if (r && hi) x = kb::mul(x, root_pow(TH, TL, ((uint32_t)hi * r) << (24 - L1 - b)));
            sm[idx] = x;
        }
        __syncthreads();
        for (int s = L1; s >= 1; s--) {
            const int half = 1 << (s - 1);
            for (int w = threadIdx.x; w < (H / 2) * T; w += blockDim.x) {
                int bf = w / T, lo = w - bf * T;
                int j = bf & (half - 1), blk = bf >> (s - 1);
                int i0 = ((blk << s) + j) * T + lo, i1 = i0 + half * T;
                uint32_t a = sm[i0], c = sm[i1];
                sm[i0] = kb::add(a, c);
                uint32_t d = kb::sub(a, c);
                sm[i1] = j ? kb::mul(d, __ldg(TH + ((uint32_t)j << (12 - s)))) : d;
            }
            __syncthreads();
        }
        for (int idx = threadIdx.x; idx < tile; idx += blockDim.x) {
            int p = idx / T, lo = idx - p * T;
            col_out[(((size_t)rr << L1) + p << L2) + lo0 + lo] = sm[idx];
        }
        __syncthreads();
    }
}

// ---- generic step B: twist + size-2^L2 DIF on contiguous rows, in place ---------------------------------
// grid (2^(L1+b), ncols), dynamic smem 2^L2 words
__global__ void rs_step_b_generic(uint32_t* __restrict__ buf, int L1, int L2, int b, const uint32_t* __restrict__ TH,
                                  const uint32_t* __restrict__ TL) {
    extern __shared__ uint32_t sm[];
    const int L = L1 + L2;
    const size_t M = (size_t)1 << (L + b);
    const uint32_t q = blockIdx.x;
    const uint32_t ka = (L1 + b) ? (__brev(q) >> (32 - (L1 + b))) : 0;
    uint32_t* row = buf + (size_t)blockIdx.y * M + ((size_t)q << L2);
    const int W = 1 << L2;
    for (int lo = threadIdx.x; lo < W; lo += blockDim.x) {
        uint32_t x = row[lo];
        uint32_t e = ((uint32_t)lo * ka) << (24 - L - b);
        if (e) x = kb::mul(x, root_pow(TH, TL, e));
        sm[lo] = x;
    }
    __syncthreads();
    for (int s = L2; s >= 1; s--) {
        const int half = 1 << (s - 1);
        for (int w = threadIdx.x; w < W / 2; w += blockDim.x) {
            int j = w & (half - 1), blk = w >> (s - 1);
            int i0 = (blk << s) + j, i1 = i0 + half;
            uint32_t a = sm[i0], c = sm[i1];
            sm[i0] = kb::add(a, c);
            uint32_t d = kb::sub(a, c);
            sm[i1] = j ? kb::mul(d, __ldg(TH + ((uint32_t)j << (12 - s)))) : d;
        }
        __syncthreads();
    }
    for (int lo = threadIdx.x; lo < W; lo += blockDim.x) row[lo] = sm[lo];
}

// ==== fast path: radix-8 butterflies in registers, 2-3 shared-memory exchanges per transform =================

// (a - c) * w with the difference left unreduced in (0, 2p): valid Montgomery operand since w < p
// (measured alternatives, 16 columns of 2^21: this subtractive Montgomery form 1.253 ms; additive wide form 1.337 ms; Shoup
// twiddles slower still — DESIGN.md 3.1)
__device__ __forceinline__ uint32_t submul(uint32_t a, uint32_t c, uint32_t w) { return kb::mul(a - c + kb::P, w); }

// in-place radix-8 decimation-in-frequency butterfly on v[0..8) (v[j], j bit 2 = most significant of the 3 index bits)
__device__ __forceinline__ void dif8(uint32_t (&v)[8], const uint32_t (&wA)[4], const uint32_t (&wB)[2], uint32_t wC) {
#pragma unroll
    for (int j = 0; j < 4; j++) { uint32_t a = v[j], c = v[j + 4]; v[j] = kb::add(a, c); v[j + 4] = submul(a, c, wA[j]); }
#pragma unroll
    for (int h = 0; h < 8; h += 4)
#pragma unroll
        for (int j = 0; j < 2; j++) { uint32_t a = v[h + j], c = v[h + j + 2]; v[h + j] = kb::add(a, c); v[h + j + 2] = submul(a, c, wB[j]); }
#pragma unroll
    for (int h = 0; h < 8; h += 2) { uint32_t a = v[h], c = v[h + 1]; v[h] = kb::add(a, c); v[h + 1] = submul(a, c, wC); }
}

// twiddles for a radix-8 pass whose top stage has 2^s points and whose elements are spaced `stride` apart:
// local element j sits at offset j*stride + low inside its 2^s block  (stride = 2^(s-3))
__device__ __forceinline__ void load_tw8(const uint32_t* __restrict__ TH, int s, uint32_t low, uint32_t (&wA)[4], uint32_t (&wB)[2],
                                         uint32_t& wC) {
    const uint32_t stride = 1u << (s - 3);
#pragma unroll
    for (int j = 0; j < 4; j++) wA[j] = __ldg(TH + ((j * stride + low) << (12 - s)));
#pragma unroll
    for (int j = 0; j < 2; j++) wB[j] = __ldg(TH + ((j * stride + low) << (13 - s)));
    wC = __ldg(TH + (low << (14 - s)));
}

// ---- fast step B: one 2048-point row per block of 256 threads, in place --------------------------------
__device__ __forceinline__ int swzB(int e) { return e ^ (((e >> 5) & 7) << 2); }

__global__ void __launch_bounds__(256) rs_step_b_2048(uint32_t* __restrict__ buf, int L1, int b, const uint32_t* __restrict__ TH,
                                                      const uint32_t* __restrict__ TL) {
    __shared__ uint32_t sm[2048];
    constexpr int L2 = 11;
    const int L = L1 + L2;
    const size_t M = (size_t)1 << (L + b);
    const uint32_t q = blockIdx.x;
    const uint32_t ka = (L1 + b) ? (__brev(q) >> (32 - (L1 + b))) : 0;
    uint32_t* row = buf + (size_t)blockIdx.y * M + ((size_t)q << L2);
    const int t = threadIdx.x;
    uint32_t v[8], wA[4], wB[2], wC;
    // pass 1: bits 10..8, straight from global, with the inter-step twist omega^(lo * ka)
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = row[j * 256 + t];
    if (ka) {
        const int sh = 24 - L - b;
        uint32_t tw = root_pow(TH, TL, ((uint32_t)t * ka) << sh);
        const uint32_t step = root_pow(TH, TL, ((256u * ka) << sh) & 0xffffffu);
#pragma unroll
        for (int j = 0; j < 8; j++) { v[j] = kb::mul(v[j], tw); if (j < 7) tw = kb::mul(tw, step); }
    }
    load_tw8(TH, 11, t, wA, wB, wC);
    dif8(v, wA, wB, wC);
#pragma unroll
    for (int j = 0; j < 8; j++) sm[swzB(j * 256 + t)] = v[j];
    __syncthreads();
    // pass 2: bits 7..5
    {
        const int low = t & 31, hib = t >> 5;
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = sm[swzB(hib * 256 + j * 32 + low)];
        load_tw8(TH, 8, low, wA, wB, wC);
        dif8(v, wA, wB, wC);
#pragma unroll
        for (int j = 0; j < 8; j++) sm[swzB(hib * 256 + j * 32 + low)] = v[j];
    }
    __syncthreads();
    // pass 3: bits 4..2
    {
        const int low = t & 3, hib = t >> 2;
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = sm[swzB(hib * 32 + j * 4 + low)];
        load_tw8(TH, 5, low, wA, wB, wC);
        dif8(v, wA, wB, wC);
#pragma unroll
        for (int j = 0; j < 8; j++) sm[swzB(hib * 32 + j * 4 + low)] = v[j];
    }
    __syncthreads();
    // pass 4: bits 1..0 (radix 4, only non-trivial twiddle is the 4th root), two groups per thread, 16-byte I/O
    const uint32_t w4 = __ldg(TH + 1024);
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const int g = t + k * 256;
        uint4 x = *reinterpret_cast<const uint4*>(&sm[swzB(4 * g)]);
        uint32_t a0 = kb::add(x.x, x.z), a1 = kb::add(x.y, x.w);
        uint32_t a2 = kb::sub(x.x, x.z), a3 = submul(x.y, x.w, w4);
        uint4 y = make_uint4(kb::add(a0, a1), kb::sub(a0, a1), kb::add(a2, a3), kb::sub(a2, a3));
        *reinterpret_cast<uint4*>(row + 4 * g) = y;
    }
}

// ---- fast step A: tile of 8 consecutive lo x all 2^L1 hi, L1 = 3*NP + 1, 2^L1 threads ----------------------
__device__ __forceinline__ int swzA(int e) { return e ^ (((e >> 7) & 1) << 4); }

// MINB = 2 caps the kernel at 32 registers (9 words spill to local memory) so that two 1024-thread blocks share an SM
template <int L1, int MINB = 1>
__global__ void __launch_bounds__(1 << L1, MINB) rs_step_a_fast(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int L2, int b,
                                                          const uint32_t* __restrict__ TH, const uint32_t* __restrict__ TL) {
    static_assert(L1 % 3 == 1 && L1 >= 7, "L1 = 3k+1, at least two radix-8 passes");
    constexpr int NP = L1 / 3;           // radix-8 passes; the last stage (hi bit 0) is a warp shuffle
    constexpr int TILE = 8 << L1;
    extern __shared__ uint32_t smA[];    // 2 x TILE words (double buffer across cosets)
    const int L = L1 + L2;
    const size_t n = (size_t)1 << L, M = n << b;
    const uint32_t* col_in = in + (size_t)blockIdx.y * n;
    uint32_t* col_out = out + (size_t)blockIdx.y * M;
    const uint32_t lo0 = blockIdx.x * 8;
    const int u = threadIdx.x, lo = u & 7, x = u >> 3;  // x: low L1-3 bits of hi in pass-1 layout
    uint32_t src[8], v[8], wA[4], wB[2], wC;
#pragma unroll
    for (int j = 0; j < 8; j++) src[j] = col_in[((size_t)(j * (1 << (L1 - 3)) + x) << L2) + lo0 + lo];
    const int sh = 24 - L1 - b;
    for (int r = 0; r < (1 << b); r++) {
        uint32_t* sm = smA + (r & 1) * TILE;
        const uint32_t rr = __brev((uint32_t)r) >> (32 - b);
        if (r == 0) {
#pragma unroll
            for (int j = 0; j < 8; j++) v[j] = src[j];
        } else {
            uint32_t tw = root_pow(TH, TL, ((uint32_t)x * r) << sh);
            const uint32_t step = root_pow(TH, TL, ((uint32_t)r << (L1 - 3)) << sh);
#pragma unroll
            for (int j = 0; j < 8; j++) { v[j] = kb::mul(src[j], tw); if (j < 7) tw = kb::mul(tw, step); }
        }
        // pass 0: hi bits L1-1 .. L1-3
        load_tw8(TH, L1, x, wA, wB, wC);
        dif8(v, wA, wB, wC);
#pragma unroll
        for (int j = 0; j < 8; j++) sm[swzA(j * (TILE / 8) + u)] = v[j];
        __syncthreads();
#pragma unroll
        for (int k = 1; k < NP; k++) {
            const int hb = L1 - 1 - 3 * k;            // top hi bit of this pass
            const int nlow = hb - 2;                  // hi bits below the pass
            const int low = x & ((1 << nlow) - 1), high = x >> nlow;
            const int base = ((high << (hb + 1)) + low) * 8 + lo;
            const int stride = 8 << nlow;
#pragma unroll
            for (int j = 0; j < 8; j++) v[j] = sm[swzA(base + j * stride)];
            load_tw8(TH, hb + 1, low, wA, wB, wC);
            dif8(v, wA, wB, wC);
            if (k < NP - 1) {
#pragma unroll
                for (int j = 0; j < 8; j++) sm[swzA(base + j * stride)] = v[j];
                __syncthreads();
            } else {
                // last stage: hi bit 0 lives in bit 3 of the thread index -> partner lane = lane ^ 8, twiddle 1
                const bool odd = (x & 1);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint32_t o = __shfl_xor_sync(0xffffffffu, v[j], 8);
                    uint32_t res = odd ? kb::sub(o, v[j]) : kb::add(v[j], o);
                    const uint32_t p = (uint32_t)((high << 4) + j * 2 + (x & 1));
                    col_out[((((size_t)rr << L1) + p) << L2) + lo0 + lo] = res;
                }
            }
        }
        // double buffering: the next coset writes the other half; the barrier after its pass 0 protects reuse
    }
}

}  // namespace

template <int L1, int MINB = 1>
static sp1b200_err launch_step_a_fast(sp1b200_ctx* ctx, const uint32_t* in, uint32_t* out, int L2, int b, unsigned nc) {
    const size_t smem = 2 * (size_t)(8 << L1) * sizeof(uint32_t);
    SP1_CUDA(cudaFuncSetAttribute(rs_step_a_fast<L1, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 g((1u << L2) / 8, nc);
    SP1_LAUNCH(ctx, (rs_step_a_fast<L1, MINB>), g, 1 << L1, smem, in, out, L2, b, ctx->d_TH, ctx->d_TL);
    return nullptr;
}

sp1b200_err sp1b200_init_tables(sp1b200_ctx* ctx) {
    SP1_CUDA(cudaMalloc(&ctx->d_TH, 4096 * sizeof(uint32_t)));
    SP1_CUDA(cudaMalloc(&ctx->d_TL, 4096 * sizeof(uint32_t)));
    SP1_LAUNCH(ctx, init_tables_kernel, 16, 256, 0, ctx->d_TH, ctx->d_TL);
    return nullptr;
}

// device-pointer implementation; d_msg [ncols x 2^log_h], d_out [ncols x 2^(log_h+log_blowup)]
sp1b200_err sp1b200_rs_encode_device(sp1b200_ctx* ctx, const uint32_t* d_msg, uint64_t ncols, uint32_t log_h,
                                     uint32_t log_blowup, uint32_t* d_out) {
    if (log_blowup < 1 || log_blowup > 4) return sp1b200_set_error("rs_encode: log_blowup %u unsupported (1..4)", log_blowup);
    if (log_h + log_blowup > 24) return sp1b200_set_error("rs_encode: 2^%u exceeds the two-adicity 2^24", log_h + log_blowup);
    if (ncols == 0) return nullptr;
    const int L = (int)log_h, b = (int)log_blowup;
    const int L2 = L < 11 ? L : 11;
    const int L1 = L - L2;
    if (L1 > 12) return sp1b200_set_error("rs_encode: log_h %u too large", log_h);
    int T = 16;
    if ((1 << L2) < T) T = 1 << L2;
    while (((size_t)T << L1) * 4 > 160 * 1024) T >>= 1;
    const size_t smemA = ((size_t)T << L1) * sizeof(uint32_t);
    const size_t smemB = ((size_t)1 << L2) * sizeof(uint32_t);
    SP1_CUDA(cudaFuncSetAttribute(rs_step_a_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    const size_t n = (size_t)1 << L, M = n << b;
    // column groups sized so that a group's step-A output stays L2-resident for step B (<= 64 MiB)
    size_t group = (64ull << 20) / (M * sizeof(uint32_t));
    if (group < 1) group = 1;
    if (group > 65535) group = 65535;
    int threadsA = (int)(((size_t)T << L1) / 2);
    if (threadsA > 1024) threadsA = 1024;
    if (threadsA < 32) threadsA = 32;
    int threadsB = (1 << L2) / 2;
    if (threadsB > 1024) threadsB = 1024;
    if (threadsB < 32) threadsB = 32;
    const bool fast = L2 == 11;
    for (uint64_t c0 = 0; c0 < ncols; c0 += group) {
        unsigned nc = (unsigned)((ncols - c0 < group) ? (ncols - c0) : group);
        dim3 gA((1u << L2) / T, nc), gB(1u << (L1 + b), nc);
        // two 1024-thread blocks per SM (32 registers, 9 words of spill) measured 7.42 ms against 7.79 ms for the 52-register build on
        // the 95 columns of S2 (profiles/bench_r02_occ*.json)
        if (fast && L1 == 10) SP1_TRY((launch_step_a_fast<10, 2>(ctx, d_msg + c0 * n, d_out + c0 * M, L2, b, nc)));
        else if (fast && L1 == 7) SP1_TRY(launch_step_a_fast<7>(ctx, d_msg + c0 * n, d_out + c0 * M, L2, b, nc));
        else SP1_LAUNCH(ctx, rs_step_a_generic, gA, threadsA, smemA, d_msg + c0 * n, d_out + c0 * M, L1, L2, b, T, ctx->d_TH, ctx->d_TL);
        if (fast) SP1_LAUNCH(ctx, rs_step_b_2048, gB, 256, 0, d_out + c0 * M, L1, b, ctx->d_TH, ctx->d_TL);
        else SP1_LAUNCH(ctx, rs_step_b_generic, gB, threadsB, smemB, d_out + c0 * M, L1, L2, b, ctx->d_TH, ctx->d_TL);
    }
    return nullptr;
}
