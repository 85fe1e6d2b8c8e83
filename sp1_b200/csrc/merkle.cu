// Poseidon2 Merkle tensor commitment over a column-major [width x 2^log_h] matrix.
// Replaces leafHashPacked / compress / computePaths / computeOpenings of
// sp1-gpu/crates/sys/lib/merkle_tree/merkle_tree.cu:27-257; semantics are p3's first_digest_layer +
// compress_and_inject as driven by slop/crates/merkle-tree/src/p3sync.rs:40-170:
//   leaf i   = PaddingFreeSponge(mat[0][i], mat[1][i], ..., mat[width-1][i])     (rate 8, overwrite mode)
//   layer k  = compress(layer k-1 [2j], layer k-1 [2j+1])
//   commit   = compress(root, hash([log_h, width]))
// Digest layers are stored bottom-up in one buffer (layer k at digest offset 2^(log_h+1) - 2^(log_h-k+1)),
// 8 words (32 B) per digest.
#include "ctx.cuh"
#include "poseidon2.cuh"

namespace {

__global__ void permute_states_kernel(uint32_t* states, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t s[16];
    uint4* p = reinterpret_cast<uint4*>(states + i * 16);
#pragma unroll
    for (int k = 0; k < 4; k++) { uint4 v = p[k]; s[4 * k] = v.x; s[4 * k + 1] = v.y; s[4 * k + 2] = v.z; s[4 * k + 3] = v.w; }
    p2::permute(s);
#pragma unroll
    for (int k = 0; k < 4; k++) p[k] = make_uint4(s[4 * k], s[4 * k + 1], s[4 * k + 2], s[4 * k + 3]);
}

__device__ __forceinline__ void store_digest(uint32_t* dst, const uint32_t (&s)[16]) {
    uint4* p = reinterpret_cast<uint4*>(dst);
    p[0] = make_uint4(s[0], s[1], s[2], s[3]);
    p[1] = make_uint4(s[4], s[5], s[6], s[7]);
}

// one thread per row; consecutive threads read consecutive words of each column (coalesced)
__global__ void __launch_bounds__(256) leaf_hash_kernel(const uint32_t* __restrict__ mat, uint64_t width, uint32_t log_h,
                                                        uint32_t* __restrict__ digests) {
    const uint64_t h = (uint64_t)1 << log_h;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= h) return;
    uint32_t s[16];
#pragma unroll
    for (int k = 0; k < 16; k++) s[k] = 0;
    const uint32_t* p = mat + i;
    uint64_t c = 0;
    for (; c + 8 <= width; c += 8) {
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = __ldg(p + (c + k) * h);
        p2::permute(s);
    }
    if (c < width) {
#pragma unroll
        for (int k = 0; k < 8; k++)
            if (c + k < width) s[k] = __ldg(p + (c + k) * h);
        p2::permute(s);
    }
    store_digest(digests + i * 8, s);
}

// parents[j] = compress(children[2j], children[2j+1]): one thread per parent, full occupancy (32 registers) — used for the wide
// layers of a tree, where throughput matters; the narrow top goes through merkle_subtree_kernel (fewer launches)
__global__ void __launch_bounds__(256) compress_layer_kernel(const uint32_t* __restrict__ children, uint32_t* __restrict__ parents,
                                                             uint64_t n_parents) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_parents) return;
    uint32_t s[16];
    const uint4* p = reinterpret_cast<const uint4*>(children + j * 16);
#pragma unroll
    for (int k = 0; k < 4; k++) { uint4 v = __ldg(p + k); s[4 * k] = v.x; s[4 * k + 1] = v.y; s[4 * k + 2] = v.z; s[4 * k + 3] = v.w; }
    p2::permute(s);
    store_digest(parents + j * 8, s);
}
// FRI-round leaves: leaf i = hash(cw[2i] limbs, cw[2i+1] limbs) -- one permutation (8 words = rate), limb-major codeword of length m
__global__ void __launch_bounds__(256) fri_leaf_hash_kernel(const uint32_t* __restrict__ cw, uint64_t m, uint32_t* __restrict__ digests) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m / 2) return;
    uint32_t s[16];
#pragma unroll
    for (int l = 0; l < 4; l++) {
        const uint2 v = *reinterpret_cast<const uint2*>(cw + l * m + 2 * i);
        s[l] = v.x; s[4 + l] = v.y;
    }
#pragma unroll
    for (int k = 8; k < 16; k++) s[k] = 0;
    p2::permute(s);
    store_digest(digests + i * 8, s);
}

// ---- subtree kernel: up to 9 compress levels per launch ------------------------------------------------------------------------
// A block takes 512 consecutive digests of layer k0 (or, MODE 1, the 512 FRI leaves it first hashes from the limb-major
// codeword: leaf i = hash(cw[2i] limbs, cw[2i+1] limbs), one permutation) and climbs: level j halves the active threads, parents
// travel through shared memory and every level is also written to its layer of the tree buffer.  A 2^23-leaf tree takes 3
// launches instead of 23 (the reference launches one `compress` per layer, merkle_tree.cu:74-94), small FRI trees one.
// The block that produces the root also forms the commitment compress(root, hash([log_h, width])) and posts the mailbox.
__device__ __forceinline__ void digest_to_smem(uint32_t* dst, const uint32_t (&s)[16]) {
    uint4* p = reinterpret_cast<uint4*>(dst);
    p[0] = make_uint4(s[0], s[1], s[2], s[3]);
    p[1] = make_uint4(s[4], s[5], s[6], s[7]);
}
template <int MODE>
__global__ void __launch_bounds__(256) merkle_subtree_kernel(const uint32_t* __restrict__ src, uint64_t m, uint32_t* __restrict__ layers,
                                                             uint32_t log_h, uint32_t k0, uint32_t L, int finalize, uint32_t width,
                                                             uint32_t* __restrict__ out16, Mail mail) {
    __shared__ __align__(16) uint32_t buf[2][256 * 8];
    const uint64_t n_leaves = (uint64_t)1 << log_h;
    auto layer_ptr = [&](uint32_t k) { return layers + (2 * n_leaves - (2 * n_leaves >> k)) * 8; };
    const uint32_t t = threadIdx.x;
    uint32_t s[16];
    // level 1
    {
        const uint64_t n_par = n_leaves >> (k0 + 1);
        const uint64_t j = (uint64_t)blockIdx.x * 256 + t;
        if (j < n_par) {
            if (MODE == 1) {
                uint32_t* leaf = layer_ptr(0);
                uint32_t d0[8];
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {
                    const uint64_t i = 2 * j + hh;
#pragma unroll
                    for (int l = 0; l < 4; l++) {
                        const uint2 v = *reinterpret_cast<const uint2*>(src + l * m + 2 * i);
                        s[l] = v.x; s[4 + l] = v.y;
                    }
#pragma unroll
                    for (int k = 8; k < 16; k++) s[k] = 0;
                    p2::permute(s);
                    store_digest(leaf + i * 8, s);
                    if (hh == 0) {
#pragma unroll
                        for (int k = 0; k < 8; k++) d0[k] = s[k];
                    }
                }
#pragma unroll
                for (int k = 0; k < 8; k++) { s[8 + k] = s[k]; s[k] = d0[k]; }
            } else {
                const uint4* p = reinterpret_cast<const uint4*>(layer_ptr(k0) + j * 16);
#pragma unroll
                for (int k = 0; k < 4; k++) { uint4 v = __ldg(p + k); s[4 * k] = v.x; s[4 * k + 1] = v.y; s[4 * k + 2] = v.z; s[4 * k + 3] = v.w; }
            }
            p2::permute(s);
            store_digest(layer_ptr(k0 + 1) + j * 8, s);
            digest_to_smem(&buf[0][t * 8], s);
        }
    }
    for (uint32_t lev = 2; lev <= L; lev++) {
        __syncthreads();
        const uint32_t n_local = 256u >> (lev - 1);
        const uint64_t n_par = n_leaves >> (k0 + lev);
        const uint64_t j = (uint64_t)blockIdx.x * n_local + t;
        if (t < n_local && j < n_par) {
            const uint4* p = reinterpret_cast<const uint4*>(&buf[lev & 1][t * 16]);
#pragma unroll
            for (int k = 0; k < 4; k++) { uint4 v = p[k]; s[4 * k] = v.x; s[4 * k + 1] = v.y; s[4 * k + 2] = v.z; s[4 * k + 3] = v.w; }
            p2::permute(s);
            store_digest(layer_ptr(k0 + lev) + j * 8, s);
            digest_to_smem(&buf[(lev & 1) ^ 1][t * 8], s);
        }
    }
    if (finalize) {
        if (t == 0 && blockIdx.x == 0) {
            // s[0..8) is the root (thread 0 computed the last level)
            uint32_t root[8], hsh[16];
#pragma unroll
            for (int k = 0; k < 8; k++) root[k] = s[k];
#pragma unroll
            for (int k = 0; k < 16; k++) hsh[k] = 0;
            hsh[0] = kb::from_canonical(log_h);
            hsh[1] = kb::from_canonical(width);
            p2::permute(hsh);
#pragma unroll
            for (int k = 0; k < 8; k++) { s[k] = root[k]; s[8 + k] = hsh[k]; }
            p2::permute(s);
#pragma unroll
            for (int k = 0; k < 8; k++) { out16[k] = root[k]; out16[8 + k] = s[k]; }
        }
        sp1_mail_done(mail);
    }
}

// commit = compress(root, hash([log_h, width]))
__global__ void tcs_commitment_kernel(const uint32_t* __restrict__ root, uint32_t log_h, uint32_t width, uint32_t* __restrict__ out16) {
    if (threadIdx.x || blockIdx.x) return;
    uint32_t s[16];
#pragma unroll
    for (int k = 0; k < 16; k++) s[k] = 0;
    s[0] = kb::from_canonical(log_h);
    s[1] = kb::from_canonical(width);
    p2::permute(s);
    uint32_t t[16];
#pragma unroll
    for (int k = 0; k < 8; k++) { t[k] = root[k]; t[8 + k] = s[k]; }
    p2::permute(t);
#pragma unroll
    for (int k = 0; k < 8; k++) { out16[k] = root[k]; out16[8 + k] = t[k]; }
}

}  // namespace

sp1b200_err sp1b200_permute_device(sp1b200_ctx* ctx, uint32_t* d_states, uint64_t n) {
    if (!n) return nullptr;
    SP1_LAUNCH(ctx, permute_states_kernel, (unsigned)((n + 255) / 256), 256, 0, d_states, n);
    return nullptr;
}

// d_layers: (2^(log_h+1) - 1) digests; d_root_commit16: 16 words (root, commitment)
sp1b200_err sp1b200_merkle_commit_device(sp1b200_ctx* ctx, const uint32_t* d_mat, uint64_t width, uint32_t log_h,
                                         uint32_t* d_layers, uint32_t* d_root_commit16) {
    if (width == 0) return sp1b200_set_error("merkle_commit: empty matrix");
    if (width >= kb::P || log_h > 30) return sp1b200_set_error("merkle_commit: shape out of range");
    const uint64_t h = (uint64_t)1 << log_h;
    {
        PhaseTimer t(ctx, "merkle.leaf_hash");  // the step's dominant kernel: timed alone for the roofline line of bench.py
        SP1_LAUNCH(ctx, leaf_hash_kernel, (unsigned)((h + 255) / 256), 256, 0, d_mat, width, log_h, d_layers);
        t.stop();
    }
    return sp1b200_merkle_tree_from_leaves_device(ctx, d_layers, log_h, (uint32_t)width, d_root_commit16);
}


// climbs from layer 0 (MODE 0: already filled; MODE 1: FRI leaves hashed from the codeword `src` of length m) to the root
// Layers with more than 2^SUBTREE_LOG nodes go through the flat one-thread-per-node kernels (full occupancy: the fused subtree
// kernel reaches 2.7 Gperm/s on a 2^22-leaf tree against 4.4 for the flat ones, profiles/launches_r01_final_S2.txt); the narrow
// top of every tree, where launch count and not throughput matters, is climbed by the subtree kernel.
constexpr uint32_t SUBTREE_LOG = 16;
template <int MODE>
static sp1b200_err build_tree(sp1b200_ctx* ctx, const uint32_t* src, uint64_t m, uint32_t* d_layers, uint32_t log_h, uint32_t width,
                              uint32_t* d_root_commit16, Mail mail) {
    const uint64_t h = (uint64_t)1 << log_h;
    auto layer_ptr = [&](uint32_t k) { return d_layers + (2 * h - (2 * h >> k)) * 8; };
    uint32_t k0 = 0;
    bool leaves_done = (MODE == 0);
    if (MODE == 1 && log_h > SUBTREE_LOG) {
        SP1_LAUNCH(ctx, fri_leaf_hash_kernel, (unsigned)((h + 255) / 256), 256, 0, src, m, d_layers);
        leaves_done = true;
    }
    while (leaves_done && log_h - k0 > SUBTREE_LOG) {
        const uint64_t n_par = h >> (k0 + 1);
        SP1_LAUNCH(ctx, compress_layer_kernel, (unsigned)((n_par + 255) / 256), 256, 0, layer_ptr(k0), layer_ptr(k0 + 1), n_par);
        k0++;
    }
    while (k0 < log_h) {
        const uint32_t L = log_h - k0 < 9 ? log_h - k0 : 9;
        const uint64_t n_children = (uint64_t)1 << (log_h - k0);
        const unsigned blocks = (unsigned)(n_children > 512 ? n_children / 512 : 1);
        const int fin = (k0 + L == log_h);
        const Mail none{nullptr, nullptr, 0};
        if (!leaves_done && k0 == 0) SP1_LAUNCH(ctx, merkle_subtree_kernel<1>, blocks, 256, 0, src, m, d_layers, log_h, k0, L, fin, width, d_root_commit16, fin ? mail : none);
        else SP1_LAUNCH(ctx, merkle_subtree_kernel<0>, blocks, 256, 0, nullptr, (uint64_t)0, d_layers, log_h, k0, L, fin, width, d_root_commit16, fin ? mail : none);
        k0 += L;
    }
    return nullptr;
}

// d_layers: leaf layer (2^log_h digests) already filled; builds the compress layers above it and
// root/commitment with the given matrix width
sp1b200_err sp1b200_merkle_tree_from_leaves_device(sp1b200_ctx* ctx, uint32_t* d_layers, uint32_t log_h, uint32_t width,
                                                   uint32_t* d_root_commit16) {
    if (log_h == 0) { SP1_LAUNCH(ctx, tcs_commitment_kernel, 1, 32, 0, d_layers, log_h, width, d_root_commit16); return nullptr; }
    return build_tree<0>(ctx, nullptr, 0, d_layers, log_h, width, d_root_commit16, Mail{nullptr, nullptr, 0});
}
// FRI round tree: leaves hashed from the limb-major codeword cw (length m = 2^(log_leaves+1) per limb), all layers, root and
// commitment (width 8); the launch that forms the root posts `mail` (flag may be NULL)
sp1b200_err sp1b200_fri_tree_device(sp1b200_ctx* ctx, const uint32_t* d_cw, uint64_t m, uint32_t* d_layers, uint32_t log_leaves,
                                    uint32_t* d_root_commit16, Mail mail) {
    if (log_leaves == 0) return sp1b200_set_error("fri_tree: a round needs at least two leaves");
    return build_tree<1>(ctx, d_cw, m, d_layers, log_leaves, 8, d_root_commit16, mail);
}
