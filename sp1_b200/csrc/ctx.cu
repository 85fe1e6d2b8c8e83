// Context, memory and the kernel-level C entry points of include/sp1b200.h.
#include "ctx.cuh"
#include <atomic>
#include <sched.h>
#include <chrono>
#include <cstring>
#include <cstdarg>
#include <cstring>
#include <cstdlib>

static thread_local char g_err[1024];

const char* sp1b200_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return g_err;
}

const char* sp1b200_last_error() { return g_err; }

bool sp1b200_is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

sp1b200_err DevBuf::in(sp1b200_ctx* c, const void* any, size_t nbytes) {
    ctx = c; bytes = nbytes;
    if (nbytes == 0) { d = nullptr; return nullptr; }
    if (sp1b200_is_device_ptr(any)) { d = const_cast<void*>(any); owned = false; return nullptr; }
    SP1_CUDA(cudaMallocFromPoolAsync(&d, nbytes, c->pool, c->stream));
    owned = true;
    SP1_CUDA(cudaMemcpyAsync(d, any, nbytes, cudaMemcpyHostToDevice, c->stream));
    return nullptr;
}
sp1b200_err DevBuf::out(sp1b200_ctx* c, void* any, size_t nbytes) {
    ctx = c; bytes = nbytes;
    if (nbytes == 0) { d = nullptr; return nullptr; }
    if (sp1b200_is_device_ptr(any)) { d = any; owned = false; return nullptr; }
    SP1_CUDA(cudaMallocFromPoolAsync(&d, nbytes, c->pool, c->stream));
    owned = true; host = any;
    return nullptr;
}
sp1b200_err DevBuf::finish() {
    if (owned && host) {
        SP1_CUDA(cudaMemcpyAsync(host, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        SP1_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (owned) { cudaFreeAsync(d, ctx->stream); owned = false; }
    return nullptr;
}
DevBuf::~DevBuf() {
    if (owned) cudaFreeAsync(d, ctx->stream);
}

extern "C" {

const char* sp1b200_version(void) { return "sp1-b200 0.1 (sp1 v6.4.0 hypercube core-shard path, sm_100a)"; }

void sp1b200_default_core_params(sp1b200_params* p) {
    p->log_stacking_height = 21; p->max_log_row_count = 22; p->log_blowup = 2; p->num_queries = 124;
    p->pow_bits = 16; p->batch_pow_bits = 5; p->gkr_pow_bits = 12; p->grind_mode = 0;
}

static sp1b200_err ctx_init(sp1b200_ctx* c, int device, const sp1b200_params* params) {
    cudaDeviceProp prop;
    SP1_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return sp1b200_set_error("ctx_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    if (params) c->params = *params; else sp1b200_default_core_params(&c->params);
    SP1_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    SP1_CUDA(cudaEventCreate(&c->ev0));
    SP1_CUDA(cudaEventCreate(&c->ev1));
    // a private stream-ordered pool per context; freed blocks stay in it instead of going back to the driver
    {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        SP1_CUDA(cudaMemPoolCreate(&c->pool, &props));
        uint64_t thresh = UINT64_MAX;
        SP1_CUDA(cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &thresh));
    }
    SP1_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        SP1_CUDA(cudaEventCreateWithFlags(&c->slot_ready[i], cudaEventDisableTiming));
        SP1_CUDA(cudaEventCreateWithFlags(&c->slot_free[i], cudaEventDisableTiming));
    }
    SP1_CUDA(cudaHostAlloc((void**)&c->h_mail, (SP1_MAIL_HDR + SP1_MAIL_WORDS) * 4, cudaHostAllocMapped | cudaHostAllocPortable));
    memset(c->h_mail, 0, (SP1_MAIL_HDR + SP1_MAIL_WORDS) * 4);
    SP1_CUDA(cudaHostGetDevicePointer((void**)&c->d_mail, c->h_mail, 0));
    SP1_CUDA(cudaMalloc((void**)&c->d_mail_counter, 64));
    SP1_CUDA(cudaMemset(c->d_mail_counter, 0, 64));
    SP1_TRY(sp1b200_init_tables(c));
    SP1_CUDA(cudaStreamSynchronize(c->stream));
    return nullptr;
}

sp1b200_err sp1b200_ctx_create(int device, const sp1b200_params* params, sp1b200_ctx** out) {
    if (!out) return sp1b200_set_error("ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    SP1_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return sp1b200_set_error("ctx_create: device %d not present (%d devices)", device, ndev);
    Sp1DeviceGuard guard(device);
    sp1b200_ctx* c = new sp1b200_ctx();
    c->device = device;
    sp1b200_err e = ctx_init(c, device, params);
    if (e) {  // every failure exit releases what was created so far (destroy null-checks each member)
        sp1b200_ctx_destroy(c);
        return e;
    }
    *out = c;
    return nullptr;
}

void sp1b200_ctx_destroy(sp1b200_ctx* c) {
    if (!c) return;
    SP1_DEVICE_GUARD(c);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->d_TH) cudaFree(c->d_TH);
    if (c->d_TL) cudaFree(c->d_TL);
    if (c->d_mail_counter) cudaFree(c->d_mail_counter);
    if (c->h_mail) cudaFreeHost(c->h_mail);
    if (c->copy_stream) { cudaStreamSynchronize(c->copy_stream); cudaStreamDestroy(c->copy_stream); }
    for (int i = 0; i < 2; i++) {
        if (c->d_slot[i]) cudaFree(c->d_slot[i]);
        if (c->slot_ready[i]) cudaEventDestroy(c->slot_ready[i]);
        if (c->slot_free[i]) cudaEventDestroy(c->slot_free[i]);
    }
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->pool) cudaMemPoolDestroy(c->pool);
    cudaGetLastError();
    delete c;
}

// Spin on the mailbox flag until the posting kernel with sequence number `seq` has published its payload.  The stream is
// queried every few thousand spins so that a faulted kernel turns into an error instead of a hang.
sp1b200_err sp1b200_mail_wait(sp1b200_ctx* c, uint32_t seq) {
    volatile uint32_t* flag = c->h_mail;
    static const bool no_poll = [] { const char* e = getenv("SP1B200_MAIL_SYNC"); return e && e[0] == '1'; }();
    if (no_poll) {  // profiling aid: wait with a stream synchronise instead of spinning (tools that serialise launches)
        SP1_CUDA(cudaStreamSynchronize(c->stream));
        if (*flag != seq) return sp1b200_set_error("mail_wait: sequence %u was not posted (flag = %u)", seq, *flag);
        return nullptr;
    }
    const auto t0 = std::chrono::steady_clock::now();
    for (uint64_t spins = 0;; spins++) {
        if (*flag == seq) { std::atomic_thread_fence(std::memory_order_acquire); return nullptr; }
        if ((spins & 0x3fff) == 0x3fff) {
            cudaError_t q = cudaStreamQuery(c->stream);
            if (q != cudaSuccess && q != cudaErrorNotReady) return sp1b200_set_error("mail_wait: stream error: %s", cudaGetErrorString(q));
            if (q == cudaSuccess && *flag != seq) {
                // stream drained but the flag did not arrive: re-check once after a full fence, then fail loudly
                std::atomic_thread_fence(std::memory_order_seq_cst);
                if (*flag == seq) return nullptr;
                return sp1b200_set_error("mail_wait: stream idle but sequence %u was never posted (flag = %u)", seq, *flag);
            }
            if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 60.0)
                return sp1b200_set_error("mail_wait: timed out waiting for sequence %u", seq);
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        // several contexts per GPU and several GPUs per host mean tens of polling threads: give the core away now and then so
        // that an oversubscribed host (cgroup CPU quota) still schedules the threads that have work (free when nobody waits)
        if ((spins & 0x3ff) == 0x3ff) sched_yield();
    }
}

// Start copying a shard's traces from (pinned) host memory into upload slot `slot` on the copy stream and return the slot's
// device pointer.  The copy overlaps whatever the main stream is doing (normally the proof of the previous shard); a later
// call on the main stream that consumes the pointer (sp1b200_prove_shard / sp1b200_jagged_commit) waits for it in stream
// order, and the slot is not overwritten before its previous consumer has finished.
sp1b200_err sp1b200_upload_begin(sp1b200_ctx* c, const uint32_t* h_src, uint64_t n_words, int slot, uint32_t** d_out) { SP1_DEVICE_GUARD(c);
    if (slot < 0 || slot > 1) return sp1b200_set_error("upload_begin: slot must be 0 or 1");
    if (!h_src || !d_out) return sp1b200_set_error("upload_begin: NULL argument");
    if (c->slot_words[slot] < n_words) {
        SP1_CUDA(cudaStreamSynchronize(c->stream));
        SP1_CUDA(cudaStreamSynchronize(c->copy_stream));
        cudaFree(c->d_slot[slot]); c->d_slot[slot] = nullptr; c->slot_words[slot] = 0;
        SP1_CUDA(cudaMalloc((void**)&c->d_slot[slot], (n_words ? n_words : 1) * 4));
        c->slot_words[slot] = n_words;
    }
    SP1_CUDA(cudaStreamWaitEvent(c->copy_stream, c->slot_free[slot], 0));  // a never-recorded event is complete
    SP1_CUDA(cudaMemcpyAsync(c->d_slot[slot], h_src, n_words * 4, cudaMemcpyHostToDevice, c->copy_stream));
    SP1_CUDA(cudaEventRecord(c->slot_ready[slot], c->copy_stream));
    c->slot_pending[slot] = true;
    *d_out = c->d_slot[slot];
    return nullptr;
}
// stream-ordered wait for a pending upload if `d_ptr` is one of the slots; returns the slot index or -1
int sp1b200_upload_acquire(sp1b200_ctx* c, const void* d_ptr) { SP1_DEVICE_GUARD(c);
    for (int i = 0; i < 2; i++)
        if (d_ptr && d_ptr == c->d_slot[i]) {
            if (c->slot_pending[i]) { cudaStreamWaitEvent(c->stream, c->slot_ready[i], 0); c->slot_pending[i] = false; }
            return i;
        }
    return -1;
}
void sp1b200_upload_release(sp1b200_ctx* c, int slot) { SP1_DEVICE_GUARD(c);
    if (slot >= 0 && slot < 2) cudaEventRecord(c->slot_free[slot], c->stream);
}

sp1b200_err sp1b200_ctx_sync(sp1b200_ctx* c) { SP1_DEVICE_GUARD(c);
    SP1_CUDA(cudaStreamSynchronize(c->stream));
    if (c->copy_stream) SP1_CUDA(cudaStreamSynchronize(c->copy_stream));
    return nullptr;
}
void* sp1b200_ctx_stream(sp1b200_ctx* c) { return (void*)c->stream; }
uint64_t sp1b200_launch_count(sp1b200_ctx* c) { return c->launches; }
float sp1b200_last_phase_ms(sp1b200_ctx* c, const char* phase) {
    auto it = c->phase_ms.find(phase);
    return it == c->phase_ms.end() ? -1.0f : it->second;
}

sp1b200_err sp1b200_malloc(sp1b200_ctx* c, size_t bytes, void** d_out) { SP1_DEVICE_GUARD(c);
    SP1_CUDA(cudaMallocFromPoolAsync(d_out, bytes, c->pool, c->stream));
    return nullptr;
}
sp1b200_err sp1b200_free(sp1b200_ctx* c, void* d_ptr) { SP1_DEVICE_GUARD(c);
    if (d_ptr) SP1_CUDA(cudaFreeAsync(d_ptr, c->stream));
    return nullptr;
}
sp1b200_err sp1b200_memcpy_h2d(sp1b200_ctx* c, void* d_dst, const void* h_src, size_t bytes) { SP1_DEVICE_GUARD(c);
    SP1_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, c->stream));
    return nullptr;
}
sp1b200_err sp1b200_memcpy_d2h(sp1b200_ctx* c, void* h_dst, const void* d_src, size_t bytes) { SP1_DEVICE_GUARD(c);
    SP1_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, c->stream));
    SP1_CUDA(cudaStreamSynchronize(c->stream));
    return nullptr;
}

sp1b200_err sp1b200_poseidon2_permute(sp1b200_ctx* c, uint32_t* states_any, uint64_t n) { SP1_DEVICE_GUARD(c);
    DevBuf b;
    SP1_TRY(b.in(c, states_any, n * 16 * sizeof(uint32_t)));
    if (b.owned) b.host = states_any;
    PhaseTimer t(c, "poseidon2_permute");
    SP1_TRY(sp1b200_permute_device(c, (uint32_t*)b.d, n));
    t.stop();
    return b.finish();
}

sp1b200_err sp1b200_rs_encode(sp1b200_ctx* c, const uint32_t* msg_any, uint64_t ncols, uint32_t log_h, uint32_t log_blowup,
                              uint32_t* out_any) { SP1_DEVICE_GUARD(c);
    DevBuf in, out;
    size_t n = (size_t)ncols << log_h;
    SP1_TRY(in.in(c, msg_any, n * sizeof(uint32_t)));
    SP1_TRY(out.out(c, out_any, (n << log_blowup) * sizeof(uint32_t)));
    PhaseTimer t(c, "rs_encode");
    SP1_TRY(sp1b200_rs_encode_device(c, (const uint32_t*)in.d, ncols, log_h, log_blowup, (uint32_t*)out.d));
    t.stop();
    SP1_TRY(out.finish());
    return in.finish();
}

sp1b200_err sp1b200_merkle_commit(sp1b200_ctx* c, const uint32_t* mat_any, uint64_t width, uint32_t log_h, uint32_t* d_layers_out,
                                  uint32_t* h_root8, uint32_t* h_commit8) { SP1_DEVICE_GUARD(c);
    DevBuf in;
    SP1_TRY(in.in(c, mat_any, ((size_t)width << log_h) * sizeof(uint32_t)));
    uint32_t* layers = d_layers_out;
    size_t nd = ((size_t)2 << log_h) - 1;
    if (!layers) SP1_CUDA(cudaMallocFromPoolAsync((void**)&layers, nd * 8 * sizeof(uint32_t), c->pool, c->stream));
    uint32_t* d_rc;
    SP1_CUDA(cudaMallocFromPoolAsync((void**)&d_rc, 16 * sizeof(uint32_t), c->pool, c->stream));
    PhaseTimer t(c, "merkle_commit");
    sp1b200_err e = sp1b200_merkle_commit_device(c, (const uint32_t*)in.d, width, log_h, layers, d_rc);
    t.stop();
    uint32_t rc[16];
    if (!e) {
        cudaError_t ce = cudaMemcpyAsync(rc, d_rc, sizeof(rc), cudaMemcpyDeviceToHost, c->stream);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->stream);
        if (ce != cudaSuccess) e = sp1b200_set_error("merkle_commit: %s", cudaGetErrorString(ce));
    }
    cudaFreeAsync(d_rc, c->stream);
    if (!d_layers_out) cudaFreeAsync(layers, c->stream);
    if (e) return e;
    if (h_root8) memcpy(h_root8, rc, 32);
    if (h_commit8) memcpy(h_commit8, rc + 8, 32);
    return in.finish();
}

}  // extern "C"
