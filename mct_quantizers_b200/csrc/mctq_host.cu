// mctq_host.cu -- process-wide state, introspection entry points and the host-buffer (staged) operators.
#include <mutex>
#include <stdint.h>

#include "mctq_common.cuh"
#include <nvtx3/nvToolsExt.h>

namespace mctq {
std::atomic<int64_t> g_launches{0};
int g_pdl = 1;              // 0 off, 1 programmatic dependent launch (wait first), opt-in: 2 + loads before the wait, 3 + no wait at all for launches independent of everything still in flight
int g_nvtx = 0;             // key 9

// ---- dependent-launch bookkeeping (see mctq_common.cuh): per (device, stream), the memory ranges of the library's launches
// since -- and including -- the last one that waited for its predecessor BEFORE touching memory (a "late" launch: when its
// first CTA passes the wait, everything enqueued before it has completed).  Every launch after it may still be running
// together with it, so a new launch is checked against the whole chain.
namespace {
struct Span { uintptr_t lo, hi; };
struct ChainLaunch {
    int n_in, n_out;        // -1 / -1: ranges unknown (multi-tensor plans): nothing may overlap with it
    int prepare;            // a mctq_*_prepare kernel: its output is a parameter blob
    Span in[2], out[2];
};
// a waiting launch + launches that overlap with it, then a waiting one again (longer chains measured no faster: DESIGN.md §5)
constexpr int kChainMax = 3;
struct StreamChain {
    cudaStream_t st;
    int device;
    uint64_t stamp;
    int n;
    ChainLaunch l[kChainMax];
};
constexpr int kLastSlots = 16;
StreamChain g_chain[kLastSlots];
uint64_t g_chain_stamp = 0;
std::mutex g_chain_mu;

inline bool overlaps(const Span& a, const Span& b) { return a.lo < b.hi && b.lo < a.hi; }
}  // namespace

NvtxRange::NvtxRange(const char* name) : on(g_nvtx != 0) { if (on) nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { if (on) nvtxRangePop(); }

void pdl_forget_streams() {
    std::lock_guard<std::mutex> lock(g_chain_mu);
    for (auto& c : g_chain) c.stamp = 0;
}

static int plan_launch(cudaStream_t st, const IoSpan* in, int n_in, const IoSpan* out, int n_out, const IoSpan* tables, uint32_t* tab_early,
                       int is_prepare) {
    if (tab_early) *tab_early = 0;
    if (g_pdl == 0) return 0;
    int device = 0;
    if (cudaGetDevice(&device) != cudaSuccess) { cudaGetLastError(); return 0; }
    ChainLaunch me;
    me.n_in = me.n_out = -1;
    me.prepare = is_prepare;
    if (in && out) {
        me.n_in = me.n_out = 0;
        for (int i = 0; i < n_in && i < 2; ++i)
            if (in[i].p && in[i].bytes) me.in[me.n_in++] = {reinterpret_cast<uintptr_t>(in[i].p), reinterpret_cast<uintptr_t>(in[i].p) + in[i].bytes};
        for (int j = 0; j < n_out && j < 2; ++j)
            if (out[j].p && out[j].bytes) me.out[me.n_out++] = {reinterpret_cast<uintptr_t>(out[j].p), reinterpret_cast<uintptr_t>(out[j].p) + out[j].bytes};
    }
    std::lock_guard<std::mutex> lock(g_chain_mu);
    StreamChain* slot = nullptr;
    StreamChain* victim = &g_chain[0];
    for (int i = 0; i < kLastSlots; ++i) {
        StreamChain& c = g_chain[i];
        if (c.stamp && c.st == st && c.device == device) { slot = &c; break; }
        if (c.stamp < victim->stamp) victim = &c;
    }
    // 0 late (wait, then everything), 1 early (loads before the wait), 2 free (no wait until the CTA's last instruction)
    int order = 0;
    if (g_pdl >= 2 && slot && me.n_in >= 0) {
        bool raw = false, other = false, unknown = false;       // input produced by the chain / output collides with the chain
        for (int k = 0; k < slot->n; ++k) {
            const ChainLaunch& c = slot->l[k];
            if (c.n_in < 0) { unknown = true; break; }
            for (int i = 0; i < me.n_in; ++i)
                for (int j = 0; j < c.n_out; ++j) raw |= overlaps(me.in[i], c.out[j]);
            for (int i = 0; i < me.n_out; ++i) {
                for (int j = 0; j < c.n_out; ++j) other |= overlaps(me.out[i], c.out[j]);
                for (int j = 0; j < c.n_in; ++j) other |= overlaps(me.out[i], c.in[j]);
            }
        }
        if (!unknown && !raw) order = (g_pdl >= 3 && !other && slot->n < kChainMax) ? 2 : 1;
    }
    // Parameter tables (prepared blobs) are private to the library: only mctq_*_prepare writes them, and it declares the
    // blob as its output here.  Unless such a launch is still in the chain, the tables were complete before the chain's
    // first launch passed its wait, so a kernel may stage them BEFORE its own wait -- whatever other libraries enqueue
    // on the stream (they never touch a blob), hence legal in the default mode too.  "Unknown" launches (multi-tensor
    // plans) write tensors, never blobs.
    if (tables && tab_early && slot) {
        // tables->p == nullptr: "several blobs" (multi-tensor plans) -- any prepare kernel in the chain counts
        const Span t = {reinterpret_cast<uintptr_t>(tables->p), reinterpret_cast<uintptr_t>(tables->p) + tables->bytes};
        bool fresh = false;
        for (int k = 0; k < slot->n; ++k) {
            const ChainLaunch& c = slot->l[k];
            if (!c.prepare) continue;
            if (!tables->p) fresh = true;
            for (int j = 0; j < c.n_out; ++j) fresh |= overlaps(t, c.out[j]);
        }
        *tab_early = fresh ? 0u : 1u;
    }
    // a stream this table has never seen (or whose entry was evicted): the predecessor may be one of our launches that
    // is no longer remembered -> late order
    if (!slot) { slot = victim; slot->n = 0; }
    slot->st = st;
    slot->device = device;
    slot->stamp = ++g_chain_stamp;
    if (order == 2) {
        slot->l[slot->n++] = me;                     // runs alongside the whole chain
    } else {
        // a launch that waits (before its stores at the latest) ends the overlap: whoever follows can only meet this launch
        slot->l[0] = me;
        slot->n = 1;
    }
    return order;
}

int pdl_plan_launch(cudaStream_t st, const IoSpan* in, int n_in, const IoSpan* out, int n_out, const IoSpan* tables, uint32_t* tab_early) {
    return plan_launch(st, in, n_in, out, n_out, tables, tab_early, 0);
}

void pdl_note_prepare(cudaStream_t st, const void* blob, size_t bytes) {
    const IoSpan out[1] = {{blob, bytes}};
    const IoSpan none[1] = {{nullptr, 0}};
    plan_launch(st, none, 0, out, 1, nullptr, nullptr, 1);
}
}  // namespace mctq

using namespace mctq;

extern "C" {

int mctq_abi_version(void) { return MCTQ_ABI_VERSION; }

const char* mctq_build_info(void) {
    return "libmctq_sm100 abi=1 arch=sm_100a threads=256 vec=16B fmad=off";
}

int64_t mctq_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int mctq_set_tuning(int key, int value) {
    int prev;
    switch (key) {
        case 3: prev = g_pdl; if (value < 0 || value > 3) return MCTQ_E_BADARG; g_pdl = value; pdl_forget_streams(); return prev;
        case 9: prev = g_nvtx; g_nvtx = value ? 1 : 0; return prev;
        default: return MCTQ_E_BADARG;
    }
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------- host staging
namespace {
constexpr int kHostStreams = 3;                      // data streams (= staging slots) of the pipeline (6: see pick_chunk_elems)
constexpr size_t kHostChunkBytesIn = 32u << 20;      // largest input chunk (slot size); small tensors use smaller chunks
constexpr size_t kParamAreaBytes = 16u << 20;        // head of the staging buffer: parameters (device side)
// The parameter area is a ring of kRing entries so that the uploads of call i + 1 never overwrite what the kernels of
// call i are still reading (calls overlap in deferred mode).  Entry layout: [scale | thr : 1.5 MB][zp : 1.5 MB][LUT table : 1 MB].
constexpr int kRing = 4;
constexpr size_t kRingEntryBytes = kParamAreaBytes / kRing;
constexpr size_t kRingArrayBytes = 1536u << 10;
constexpr size_t kRingTableBytes = 1u << 20;

struct HostCtx {
    int device = -1;
    cudaStream_t st[kHostStreams] = {};
    cudaStream_t st_par = nullptr;                   // parameter uploads: never queued behind a data chunk
    cudaEvent_t params_ready = nullptr;
    int deferred = 0;                                // calls return without synchronising (mctq_host_set_deferred)
    uint64_t next_chunk = 0;                         // round-robin position over the streams / slots, continues across calls
    uint64_t ring_pos = 0;
    uint8_t* pin = nullptr;                          // pinned host mirror of the parameter ring
    cudaEvent_t uploaded[kRing] = {};                // the H2D copy out of pin entry e has finished
    cudaEvent_t released[kRing][kHostStreams] = {};  // the last kernel of stream i that reads device entry e has finished
    std::mutex mu;                                   // host-buffer calls of one device are serialised (ctypes drops the GIL)
};
HostCtx g_hctx[16];

int host_ctx(int device, HostCtx** out) {
    if (device < 0 || device >= 16) return MCTQ_E_NODEVICE;
    HostCtx& c = g_hctx[device];
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return (int)e;
    std::lock_guard<std::mutex> init_lock(c.mu);
    if (c.device != device) {
        for (int i = 0; i < kHostStreams; ++i) {
            e = cudaStreamCreateWithFlags(&c.st[i], cudaStreamNonBlocking);
            if (e != cudaSuccess) return (int)e;
        }
        e = cudaStreamCreateWithFlags(&c.st_par, cudaStreamNonBlocking);
        if (e != cudaSuccess) return (int)e;
        e = cudaEventCreateWithFlags(&c.params_ready, cudaEventDisableTiming);
        if (e != cudaSuccess) return (int)e;
        e = cudaHostAlloc(reinterpret_cast<void**>(&c.pin), kParamAreaBytes, cudaHostAllocDefault);
        if (e != cudaSuccess) return (int)e;
        for (int r = 0; r < kRing; ++r) {
            e = cudaEventCreateWithFlags(&c.uploaded[r], cudaEventDisableTiming);
            if (e != cudaSuccess) return (int)e;
            for (int i = 0; i < kHostStreams; ++i) {
                e = cudaEventCreateWithFlags(&c.released[r][i], cudaEventDisableTiming);
                if (e != cudaSuccess) return (int)e;
            }
        }
        c.device = device;
    }
    *out = &c;
    return 0;
}
size_t dtype_size(int dt) { return dt == MCTQ_F32 ? 4 : 2; }

int sync_all(HostCtx* ctx) {
    cudaError_t e = cudaStreamSynchronize(ctx->st_par);
    for (int i = 0; i < kHostStreams; ++i) {
        cudaError_t e2 = cudaStreamSynchronize(ctx->st[i]);
        if (e == cudaSuccess) e = e2;
    }
    return cuda_rc(e);
}

// chunk length: about an eighth of the tensor so that uploads, kernels and downloads of neighbouring chunks overlap
// even for tensors of a few tens of MB, between 1 MB of input and the slot size, a multiple of 64 Ki elements
// (a sixteenth was measured and is slower: 67 MB 76 -> 71 GB/s, the per-transfer latency of the copy engines dominates)
// In deferred mode the pipeline does not drain between calls, so there is nothing to overlap WITHIN a tensor and whole
// slots move best: MobileNetV2 step with host tensors 87.2 GB/s with eighths, 88.8 with halves, 91.6 with whole slots
// (6 streams instead of 3 on top: 92.2, not worth 300 MB of staging).
int64_t pick_chunk_elems(int64_t n, size_t in_elem_bytes, size_t slot_elem_bytes, bool deferred) {
    const int64_t max_elems = (int64_t)(kHostChunkBytesIn / slot_elem_bytes);
    const int64_t min_elems = (int64_t)((1u << 20) / in_elem_bytes);
    const int64_t div = deferred ? 1 : 8;
    int64_t c = (n / div + 65535) / 65536 * 65536;
    if (c < min_elems) c = min_elems;
    if (c > max_elems) c = max_elems;
    return c;
}

// Small tensors in PINNED host memory skip the staging pipeline altogether: the streaming kernel reads x and writes y
// directly over PCIe through their unified virtual addresses (one launch, no fill / drain of a three-stage pipeline).
// Measured on the B200 box (profiles/r01_pcie_probe.txt), one synchronous call: 1 MB 40, 4 MB 50 vs 41, 17 MB 60 vs 51,
// 67 MB 69 vs 74, 1 GB 79 vs 88-93 GB/s (zero-copy vs copy engines) -> cut-over at 32 MB of input.  In deferred mode the
// pipeline does not drain between calls, so the copy engines win earlier: cut-over at 8 MB.
constexpr size_t kZeroCopyMaxBytesSync = 32u << 20;
constexpr size_t kZeroCopyMaxBytesDeferred = 8u << 20;

bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost && at.devicePointer == p;
}
bool zero_copy_ok(const HostCtx* ctx, const void* x_host, const void* y_host, int64_t n, size_t in_es) {
    const size_t limit = ctx->deferred ? kZeroCopyMaxBytesDeferred : kZeroCopyMaxBytesSync;
    return (size_t)n * in_es <= limit && is_pinned(x_host) && is_pinned(y_host);
}

// One host-buffer call.  Parameters (if any) go through ring entry `e` of the pinned mirror and the device parameter
// area on the dedicated parameter stream; the data goes H2D -> launch(chunk) -> D2H chunk by chunk, round-robin over the
// data streams, continuing where the previous call stopped.  In the default mode the call returns when y_host is
// complete; in deferred mode it returns as soon as everything is enqueued (mctq_host_wait completes the results), so
// that the pipeline never drains between the tensors of a model.
struct HostCall {
    HostCtx* ctx;
    uint8_t* base;           // staging buffer
    int entry = -1;          // ring entry holding this call's parameters (-1: none)
    uint8_t* d_entry = nullptr;
    uint8_t* h_entry = nullptr;

    // reserve a ring entry; returns its pinned host address to be filled before upload()
    int begin_params() {
        entry = (int)(ctx->ring_pos++ % kRing);
        d_entry = base + (size_t)entry * kRingEntryBytes;
        h_entry = ctx->pin + (size_t)entry * kRingEntryBytes;
        return cuda_rc(cudaEventSynchronize(ctx->uploaded[entry]));     // host side: the previous upload out of h_entry is done
    }
    int upload(size_t off, size_t bytes) {
        return cuda_rc(cudaMemcpyAsync(d_entry + off, h_entry + off, bytes, cudaMemcpyHostToDevice, ctx->st_par));
    }
    int before_uploads() {
        // device side: every kernel that read the previous contents of this entry has finished
        for (int i = 0; i < kHostStreams; ++i) {
            cudaError_t e = cudaStreamWaitEvent(ctx->st_par, ctx->released[entry][i], 0);
            if (e != cudaSuccess) return (int)e;
        }
        return 0;
    }
    int after_uploads() {
        cudaError_t e = cudaEventRecord(ctx->uploaded[entry], ctx->st_par);
        if (e != cudaSuccess) return (int)e;
        return cuda_rc(cudaEventRecord(ctx->params_ready, ctx->st_par));
    }

    template <class Launch>
    int run(const uint8_t* x_host, uint8_t* y_host, int64_t n, size_t in_es, size_t out_es, bool zero_copy, Launch launch) {
        cudaError_t e = cudaSuccess;
        int rc = 0;
        bool used[kHostStreams] = {};
        auto stream_for = [&](uint64_t k) {
            const int i = (int)(k % (uint64_t)kHostStreams);
            if (!used[i]) {
                used[i] = true;
                if (entry >= 0) cudaStreamWaitEvent(ctx->st[i], ctx->params_ready, 0);
            }
            return i;
        };
        if (zero_copy) {
            // the kernel reads x_host / writes y_host over PCIe through their unified virtual addresses
            const int i = stream_for(ctx->next_chunk++);
            rc = launch(x_host, y_host, n, 0, ctx->st[i]);
        } else {
            uint8_t* slots = base + kParamAreaBytes;
            const int64_t chunk_elems = pick_chunk_elems(n, in_es, in_es > out_es ? in_es : out_es, ctx->deferred != 0);
            for (int64_t off = 0; off < n; off += chunk_elems) {
                const int64_t cnt = (n - off) < chunk_elems ? (n - off) : chunk_elems;
                const int i = stream_for(ctx->next_chunk++);
                cudaStream_t st = ctx->st[i];
                uint8_t* d_in = slots + (size_t)i * 3 * kHostChunkBytesIn;
                uint8_t* d_out = d_in + kHostChunkBytesIn;
                e = cudaMemcpyAsync(d_in, x_host + off * in_es, cnt * in_es, cudaMemcpyHostToDevice, st);
                if (e != cudaSuccess) break;
                rc = launch(d_in, d_out, cnt, off, st);
                if (rc) break;
                e = cudaMemcpyAsync(y_host + off * out_es, d_out, cnt * out_es, cudaMemcpyDeviceToHost, st);
                if (e != cudaSuccess) break;
            }
        }
        if (entry >= 0)
            for (int i = 0; i < kHostStreams; ++i)
                if (used[i]) cudaEventRecord(ctx->released[entry][i], ctx->st[i]);
        if (!ctx->deferred || rc || e != cudaSuccess) {
            const int rs = sync_all(ctx);
            if (!rc && e == cudaSuccess) rc = rs;
        }
        return rc ? rc : cuda_rc(e);
    }
};
}  // namespace

extern "C" {

size_t mctq_host_staging_min_bytes(void) {
    // per stream: one input chunk + one f32-sized output chunk (LUT output of a 2-byte input is 2x larger) + parameter area
    return (size_t)kHostStreams * (kHostChunkBytesIn + 2 * kHostChunkBytesIn) + kParamAreaBytes;
}

int mctq_host_set_deferred(int device, int on) {
    HostCtx* ctx;
    int rc = host_ctx(device, &ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (ctx->deferred && !on) rc = sync_all(ctx);
    ctx->deferred = on ? 1 : 0;
    return rc;
}

int mctq_host_wait(int device) {
    MCTQ_NVTX("mctq_host_wait");
    HostCtx* ctx;
    int rc = host_ctx(device, &ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    return sync_all(ctx);
}

int mctq_fq_affine_host(const void* x_host, void* y_host, int64_t n, int x_dtype, const float* scale_host,
                        const int32_t* zp_host, int64_t C, int64_t inner, int32_t qmin, int32_t qmax,
                        void* staging_dev, size_t staging_bytes, int device) {
    MCTQ_NVTX("mctq_fq_affine_host");
    if (!x_host || !y_host || !scale_host || !zp_host || !staging_dev || n < 0 || C < 1 || inner < 1) return MCTQ_E_BADARG;
    if (x_dtype < 0 || x_dtype > 2) return MCTQ_E_DTYPE;
    if (staging_bytes < mctq_host_staging_min_bytes() || (size_t)C * 4 > kRingArrayBytes) return MCTQ_E_BADARG;
    if (n == 0) return 0;
    HostCtx* ctx;
    int rc = host_ctx(device, &ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const size_t es = dtype_size(x_dtype);
    HostCall call{ctx, reinterpret_cast<uint8_t*>(staging_dev)};
    const bool zc = zero_copy_ok(ctx, x_host, y_host, n, es);
    const uint8_t* xb = reinterpret_cast<const uint8_t*>(x_host);
    uint8_t* yb = reinterpret_cast<uint8_t*>(y_host);
    if (C == 1) {
        // per-tensor: parameters travel by value, nothing to upload
        const float s = scale_host[0];
        const int32_t z = zp_host[0];
        return call.run(xb, yb, n, es, es, zc, [&](const uint8_t* d_in, uint8_t* d_out, int64_t cnt, int64_t, cudaStream_t st) {
            return mctq_fq_affine_scalar(d_in, d_out, nullptr, cnt, x_dtype, s, z, qmin, qmax, MCTQ_CODES_NONE, st);
        });
    }
    if ((rc = call.begin_params())) return rc;
    memcpy(call.h_entry, scale_host, (size_t)C * 4);
    memcpy(call.h_entry + kRingArrayBytes, zp_host, (size_t)C * 4);
    if ((rc = call.before_uploads()) || (rc = call.upload(0, (size_t)C * 4)) || (rc = call.upload(kRingArrayBytes, (size_t)C * 4)) ||
        (rc = call.after_uploads()))
        return rc;
    const float* d_scale = reinterpret_cast<const float*>(call.d_entry);
    const int32_t* d_zp = reinterpret_cast<const int32_t*>(call.d_entry + kRingArrayBytes);
    return call.run(xb, yb, n, es, es, zc, [&](const uint8_t* d_in, uint8_t* d_out, int64_t cnt, int64_t off, cudaStream_t st) {
        return mctq_fq_affine(d_in, d_out, nullptr, cnt, x_dtype, d_scale, d_zp, C, inner, off, qmin, qmax, MCTQ_CODES_NONE, st);
    });
}

int mctq_fq_lut_host(const void* x_host, float* y_host, int64_t n, int x_dtype, const void* table_host, int K,
                     const float* thr_host, int64_t C, int64_t inner, float eps, int scalar_mode, float divisor,
                     float thr_f32, int round_to_x_dtype, void* staging_dev, size_t staging_bytes, int device) {
    MCTQ_NVTX("mctq_fq_lut_host");
    if (!x_host || !y_host || !table_host || !staging_dev || n < 0 || C < 1 || inner < 1) return MCTQ_E_BADARG;
    if (!scalar_mode && !thr_host) return MCTQ_E_BADARG;
    if (x_dtype < 0 || x_dtype > 2) return MCTQ_E_DTYPE;
    const size_t tbytes = mctq_lut_table_bytes(K);
    if (!tbytes || tbytes > kRingTableBytes) return MCTQ_E_LUT;
    if (staging_bytes < mctq_host_staging_min_bytes() || (size_t)C * 4 > kRingArrayBytes) return MCTQ_E_BADARG;
    if (n == 0) return 0;
    HostCtx* ctx;
    int rc = host_ctx(device, &ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const size_t es = dtype_size(x_dtype);
    HostCall call{ctx, reinterpret_cast<uint8_t*>(staging_dev)};
    if ((rc = call.begin_params())) return rc;
    if (!scalar_mode) memcpy(call.h_entry, thr_host, (size_t)C * 4);
    memcpy(call.h_entry + 2 * kRingArrayBytes, table_host, tbytes);
    if ((rc = call.before_uploads())) return rc;
    if (!scalar_mode && (rc = call.upload(0, (size_t)C * 4))) return rc;
    if ((rc = call.upload(2 * kRingArrayBytes, tbytes)) || (rc = call.after_uploads())) return rc;
    const float* d_thr = reinterpret_cast<const float*>(call.d_entry);
    const uint8_t* d_table = call.d_entry + 2 * kRingArrayBytes;
    const bool zc = zero_copy_ok(ctx, x_host, y_host, n, es);
    return call.run(reinterpret_cast<const uint8_t*>(x_host), reinterpret_cast<uint8_t*>(y_host), n, es, 4, zc,
                    [&](const uint8_t* d_in, uint8_t* d_out, int64_t cnt, int64_t off, cudaStream_t st) {
                        float* out = reinterpret_cast<float*>(d_out);
                        if (scalar_mode)
                            return mctq_fq_lut_scalar(d_in, out, nullptr, cnt, x_dtype, d_table, K, divisor, thr_f32, round_to_x_dtype,
                                                      MCTQ_CODES_NONE, st);
                        return mctq_fq_lut(d_in, out, nullptr, cnt, x_dtype, d_table, K, d_thr, C, inner, off, eps, MCTQ_CODES_NONE, st);
                    });
}

}  // extern "C"
