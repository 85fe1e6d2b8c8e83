// Context / runtime shared by all kernels: one CUDA stream, stream-ordered pool allocations,
// root-of-unity tables, launch counter and per-phase CUDA-event timing.
// Replaces the role of sp1-gpu/crates/cuda (TaskScope = stream + cudaMallocAsync pool) and
// sp1-gpu/crates/sys/lib/runtime/{stream,memory,mem_pool}.cu for this path.
#pragma once
#include <cuda_runtime.h>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "../../include/sp1b200.h"

struct sp1b200_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaMemPool_t pool = nullptr;  // this context's own stream-ordered pool: contexts proving concurrently never wait on each other's frees
    sp1b200_params params{};
    // TH[i] = w^(i * 2^12), TL[j] = w^j  with w = two-adic generator of order 2^24 (Montgomery words)
    uint32_t* d_TH = nullptr;
    uint32_t* d_TL = nullptr;
    uint64_t launches = 0;
    std::map<std::string, float> phase_ms;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // mailbox: pinned + mapped host memory the round kernels write their few result words into, followed by a sequence flag;
    // the host transcript polls the flag instead of issuing a copy + stream synchronise per sumcheck round
    uint32_t* h_mail = nullptr;         // [0] flag, payload from MAIL_HDR
    uint32_t* d_mail = nullptr;         // device alias of h_mail
    uint32_t* d_mail_counter = nullptr; // device memory: blocks finished in the current posting kernel
    uint32_t mail_seq = 0;
    // double-buffered upload slots: host traces of the NEXT shard are copied on `copy_stream` while the current one is proven
    cudaStream_t copy_stream = nullptr;
    uint32_t* d_slot[2] = {nullptr, nullptr};
    uint64_t slot_words[2] = {0, 0};
    cudaEvent_t slot_ready[2] = {nullptr, nullptr};   // recorded on copy_stream after the upload
    cudaEvent_t slot_free[2] = {nullptr, nullptr};    // recorded on stream when the consumer (prove_shard) is done with the slot
    bool slot_pending[2] = {false, false};
    std::unique_ptr<uint32_t[]> shard_scratch;  // host staging of the three variable-length proof sections (shard.cu), reused across shards
};
constexpr size_t SP1_MAIL_HDR = 16;               // words before the payload (64-byte aligned payload)
constexpr size_t SP1_MAIL_WORDS = 1 << 16;        // payload capacity in words (256 KiB)

struct Mail { uint32_t* flag; uint32_t* counter; uint32_t seq; };
inline Mail sp1b200_mail_next(sp1b200_ctx* c) { return Mail{c->d_mail, c->d_mail_counter, ++c->mail_seq}; }
inline uint32_t* sp1b200_mail_dev(sp1b200_ctx* c) { return c->d_mail + SP1_MAIL_HDR; }
inline const uint32_t* sp1b200_mail_host(sp1b200_ctx* c) { return c->h_mail + SP1_MAIL_HDR; }
extern "C" sp1b200_err sp1b200_mail_wait(sp1b200_ctx* c, uint32_t seq);

#ifdef __CUDACC__
// Last step of a posting kernel, called by EVERY thread after the block's payload words were stored through the device
// alias: the last block to arrive publishes the sequence number (system-scope release) and re-arms the counter.
__device__ __forceinline__ void sp1_mail_done(const Mail& m) {
    if (!m.flag) return;  // launch-uniform: this launch does not post
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0 && threadIdx.z == 0) {
        const unsigned total = gridDim.x * gridDim.y * gridDim.z;
        const unsigned prev = atomicAdd(m.counter, 1u);
        if (prev == total - 1) {
            *m.counter = 0;
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t*>(m.flag) = m.seq;
        }
    }
}
#endif

const char* sp1b200_set_error(const char* fmt, ...);
const char* sp1b200_last_error();   // the calling thread's most recent message

// Every extern "C" entry point that takes a context runs with the context's device current and restores the caller's device on
// exit: the CUDA current device is per host thread and defaults to 0, so a host runtime that drives several GPUs from one process
// (worker threads, tokio spawn_blocking) would otherwise allocate and launch on the wrong device.
struct Sp1DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit Sp1DeviceGuard(int dev) {
        if (dev < 0) return;
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~Sp1DeviceGuard() { if (switched) cudaSetDevice(prev); }
    Sp1DeviceGuard(const Sp1DeviceGuard&) = delete;
    Sp1DeviceGuard& operator=(const Sp1DeviceGuard&) = delete;
};
#define SP1_DEVICE_GUARD(c) Sp1DeviceGuard _sp1_device_guard((c) ? (c)->device : -1)

#define SP1_CUDA(call)                                                                            \
    do {                                                                                          \
        cudaError_t _e = (call);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return sp1b200_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
    } while (0)

#define SP1_TRY(call)                   \
    do {                                \
        sp1b200_err _m = (call);        \
        if (_m) return _m;              \
    } while (0)

// launch wrapper: counts the launch and checks the launch error
#define SP1_LAUNCH(ctx, kernel, grid, block, smem, ...)                        \
    do {                                                                       \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);       \
        (ctx)->launches++;                                                     \
        SP1_CUDA(cudaGetLastError());                                          \
    } while (0)

struct PhaseTimer {
    sp1b200_ctx* ctx;
    const char* name;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool done = false;
    PhaseTimer(sp1b200_ctx* c, const char* n) : ctx(c), name(n) {
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, c->stream);
    }
    // call after the phase's last launch; synchronises on the end event
    void stop() {
        if (done) return;
        done = true;
        cudaEventRecord(e1, ctx->stream);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        ctx->phase_ms[name] = ms;
    }
    ~PhaseTimer() { cudaEventDestroy(e0); cudaEventDestroy(e1); }
};

// host wall-clock accumulator reported next to the CUDA-event phases (where the host waits or computes inside a phase)
struct HostAccum {
    sp1b200_ctx* ctx; const char* name; double ms = 0;
    HostAccum(sp1b200_ctx* c, const char* n) : ctx(c), name(n) {}
    ~HostAccum() { ctx->phase_ms[name] = (float)ms; }
};
struct HostSpan {
    HostAccum& a; std::chrono::steady_clock::time_point t0;
    explicit HostSpan(HostAccum& acc) : a(acc), t0(std::chrono::steady_clock::now()) {}
    ~HostSpan() { a.ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

// resolves a host-or-device pointer to a device pointer, staging through a temporary if needed
struct DevBuf {
    sp1b200_ctx* ctx = nullptr;
    void* d = nullptr;
    void* host = nullptr;  // original host pointer if staged
    size_t bytes = 0;
    bool owned = false;
    sp1b200_err in(sp1b200_ctx* c, const void* any, size_t nbytes);        // for inputs (copies H2D if host)
    sp1b200_err out(sp1b200_ctx* c, void* any, size_t nbytes);             // for outputs (allocates if host)
    sp1b200_err finish();                                                  // D2H copy-back for outputs, free
    ~DevBuf();
};

// stream-ordered scratch allocations from the context's pool, freed (stream-ordered) when the scope ends
struct DevFree {
    sp1b200_ctx* ctx;
    std::vector<void*> ptrs;
    explicit DevFree(sp1b200_ctx* c) : ctx(c) {}
    ~DevFree() { for (void* p : ptrs) cudaFreeAsync(p, ctx->stream); }
    sp1b200_err alloc(void** p, size_t bytes) {
        SP1_CUDA(cudaMallocFromPoolAsync(p, bytes ? bytes : 4, ctx->pool, ctx->stream));
        ptrs.push_back(*p);
        return nullptr;
    }
};
inline unsigned blocks_for(uint64_t n, unsigned bs = 256) { return (unsigned)((n + bs - 1) / bs); }

bool sp1b200_is_device_ptr(const void* p);
extern "C" int sp1b200_upload_acquire(sp1b200_ctx* c, const void* d_ptr);
extern "C" void sp1b200_upload_release(sp1b200_ctx* c, int slot);

// device-pointer implementations behind the C entry points, called across translation units (ntt.cu, merkle.cu)
sp1b200_err sp1b200_init_tables(sp1b200_ctx* ctx);
sp1b200_err sp1b200_rs_encode_device(sp1b200_ctx* ctx, const uint32_t* d_msg, uint64_t ncols, uint32_t log_h, uint32_t log_blowup,
                                     uint32_t* d_out);
sp1b200_err sp1b200_permute_device(sp1b200_ctx* ctx, uint32_t* d_states, uint64_t n);
sp1b200_err sp1b200_merkle_commit_device(sp1b200_ctx* ctx, const uint32_t* d_mat, uint64_t width, uint32_t log_h, uint32_t* d_layers,
                                         uint32_t* d_root_commit16);
sp1b200_err sp1b200_merkle_tree_from_leaves_device(sp1b200_ctx* ctx, uint32_t* d_layers, uint32_t log_h, uint32_t width,
                                                   uint32_t* d_root_commit16);
sp1b200_err sp1b200_fri_tree_device(sp1b200_ctx* ctx, const uint32_t* d_cw, uint64_t m, uint32_t* d_layers, uint32_t log_leaves,
                                    uint32_t* d_root_commit16, Mail mail);
