// capi.cu -- the C ABI of liblz4b200.so (include/lz4b200.h): context, batched entry points, single-block entry points.
//
// Host-memory batches are processed as a software pipeline: the block list is cut into chunks, and for each chunk
// H2D(inputs) -> kernel -> D2H(outputs) is enqueued on one of NSLOT streams, so that the copy engines (both PCIe
// directions) and the SMs work on different chunks at the same time.  There is no CPU codec in this library: if the
// device or the kernel image is unusable every entry point reports an error.
#include "../../include/lz4b200.h"
#include "kernels.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace lz4b200;

namespace {

thread_local std::string g_err = "";

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what)
{
    g_err = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return LZ4B200_E_CUDA;
}
#define CU(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)

constexpr int NSLOT = 3;                       // pipeline depth of host-memory batches
constexpr int NCOUNTER = 256;
constexpr size_t HOST_CHUNK_BYTES_DEFAULT = 128u << 20; // src + dst bytes per pipeline stage (tools/e2e_sweep.py: 128 MiB is the best of 32..512 on B200)

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + (n >> 3) + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
struct PinBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMallocHost(&p, n + 4096);
        if (e == cudaSuccess) cap = n + 4096;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Pageable host memory (a managed caller's `fixed` byte[]): cudaMemcpyAsync from / to it is staged by the driver through
// its own small pinned buffers, synchronously (measured: 4.5 GB/s round trip against 21 from pinned memory).  The library
// stages such buffers itself, a pipeline chunk at a time, with a handful of host threads doing the memcpy into / out of
// its pinned chunk buffers while the previous chunks are on the wire.
constexpr int STAGE_THREADS = 8;
constexpr size_t STAGE_PARALLEL_MIN = 4u << 20;

void par_ranges(size_t n, size_t min_parallel, const std::function<void(size_t, size_t)>& fn)
{
    if (n < min_parallel) { fn(0, n); return; }
    std::vector<std::thread> th;
    const size_t per = (n + STAGE_THREADS - 1) / STAGE_THREADS;
    for (int t = 1; t < STAGE_THREADS; t++) {
        const size_t lo = per * t, hi = std::min(n, lo + per);
        if (lo < hi) th.emplace_back(fn, lo, hi);
    }
    fn(0, std::min(n, per));
    for (auto& t : th) t.join();
}
void par_memcpy(void* dst, const void* src, size_t n)
{
    par_ranges(n, STAGE_PARALLEL_MIN, [&](size_t lo, size_t hi) { std::memcpy((uint8_t*)dst + lo, (const uint8_t*)src + lo, hi - lo); });
}
bool is_pageable(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    DevBuf src, dst, meta, packed, offs, scan;
    PinBuf hmeta, bounce, hsrc, hdst;
};

}  // namespace

struct lz4b200_ctx {
    int device = 0;
    DeviceInfo dev{};
    cudaStream_t stream = nullptr;
    uint32_t* counters = nullptr;
    int next_counter = 0;
    DevBuf hc_arena, compact_tmp;
    DevBuf stream_work, stream_table, stream_res;   // device framing: encoder slots + per-chunk metadata, chunk tables, walk result
    PinBuf stream_host;                    // their results, read back by the host
    cudaEvent_t hc_done = nullptr;         // the HC state arena is shared: HC launches are chained through this event
    cudaEvent_t compact_done = nullptr;    // likewise the scan scratch of lz4b200_compact
    int decode_lanes = 16;                 // lanes per block for device-memory batches (+100 = output-staged variant)
    bool decode_lanes_auto = true;         // host-memory batches: chosen per chunk from the compression ratio
    int encode_ctas_per_sm = 0;            // encoder warps (= blocks in flight) per SM: 0 = as many as shared memory holds tables for (14)
    int encode_variant = 2;                // same-hash detection inside a round: 1 exact votes, 2 optimistic (default)
    int encode_tune[4] = {512, 12, 8, 24}; // prefetch distance, lane_copy_max, probe_max, wide_min (lz4_encode.cuh EncTune)
    size_t host_chunk_bytes = HOST_CHUNK_BYTES_DEFAULT;
    int hc_concurrency = 131072;         // blocks in flight (one thread each, 256 KiB state): 16384 / 65536 / 131072 / 262144 -> 2.8 / 8.3 / 9.7 / 9.7 GB/s (E50)
    int hc_kernel = -1;                  // -1: chosen per batch (encode.cu launch_encode_hc_auto); 0: one thread per block (any block size); one warp per block on a static index (blocks <= 64 KiB, the rest is handed to 0): 1 = block staged in shared memory, 2 = nothing in shared memory
    int hc_warps_per_sm = 0;             // warp kernels: blocks in flight per SM (0 = 3 for kernel 1, 32 for kernel 2)
    Slot slot[NSLOT];
    int64_t launches = 0;
    std::mutex mu;

    uint32_t* counter() { uint32_t* c = counters + next_counter; next_counter = (next_counter + 4) % NCOUNTER; return c; }   // fours: [block counter, decoder pick, two more counters]
};

namespace {

struct DeviceGuard {
    int prev = -1; bool ok;
    explicit DeviceGuard(int dev) { ok = cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Decode group size from the ratio compressed/raw of a batch (tools/sweep.py): incompressible data is long literal runs
// (whole warps, 128-bit copies), nearly-empty streams are long matches, everything between is sequence-dense (the
// denser, the smaller the group: 8 lanes around ratio 0.58, 4 lanes around 0.37; both output-staged).
int lanes_for_ratio(double ratio, int64_t n_blocks, const DeviceInfo& dev)
{
    const int g = decode_lanes_for_ratio(ratio);
    // token-dense + at least half a wave of blocks: one lane per block (decode.cu lpb_pays; host chunks rarely fill whole
    // waves, so the middle class stays with the 8-lane group kernel)
    return g == 104 && n_blocks >= (int64_t)dev.num_sms * 32 * 8 ? 1 : g;
}

int run_device(lz4b200_ctx* c, const BatchArgs& a, int op /*0 enc fast, 1 enc hc, 2 dec known, 3 dec unknown*/, cudaStream_t st, int lanes = 0)
{
    if (!lanes && !c->decode_lanes_auto) lanes = c->decode_lanes;       // (0 = auto: the decoder is picked on the device)
    cudaError_t e = cudaSuccess;
    switch (op) {
    case 0: e = launch_encode_fast(a, c->counter(), c->encode_ctas_per_sm, c->encode_tune, c->encode_variant, c->dev, st, &c->launches); break;
    case 1: {
        // (chosen per batch: the thread kernel only runs for batches of blocks above 64 KiB -- 4 GiB of state at most there)
        const int conc = (int)std::min<int64_t>(c->hc_kernel < 0 ? std::min(c->hc_concurrency, 16384) : c->hc_concurrency, std::max(a.n_blocks, 1));
        const size_t need = c->hc_kernel < 0 ? hc_auto_scratch_bytes(a.n_blocks, conc, c->dev)
                          : (c->hc_kernel ? hcw_scratch_bytes(a.n_blocks, c->hc_kernel, c->hc_warps_per_sm, c->dev) : hc_scratch_bytes(conc));
        if (need > c->hc_arena.cap) {
            CU(cudaDeviceSynchronize());           // the arena may still be in use by an earlier launch
            CU(c->hc_arena.reserve(need));
        }
        // one arena per context: an HC launch may not overlap the previous one, whatever stream it was given
        CU(cudaStreamWaitEvent(st, c->hc_done, 0));
        e = c->hc_kernel < 0 ? launch_encode_hc_auto(a, c->hc_arena.p, conc, c->counter(), c->dev, st, &c->launches)
          : c->hc_kernel ? launch_encode_hcw(a, c->hc_arena.p, c->hc_kernel, c->hc_warps_per_sm, c->counter(), c->dev, st, &c->launches)
                              : launch_encode_hc(a, c->hc_arena.p, conc, c->counter(), c->dev, st, &c->launches);
        if (e == cudaSuccess) e = cudaEventRecord(c->hc_done, st);
        break;
    }
    case 2: e = launch_decode(a, true, lanes, c->counter(), c->dev, st, &c->launches); break;
    default: e = launch_decode(a, false, lanes, c->counter(), c->dev, st, &c->launches); break;
    }
    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
    return LZ4B200_OK;
}

// Host-memory batch: chunked, overlapped H2D / kernel / D2H.
// Only bytes a block PRODUCED ever reach the caller's buffer (the reference's safe codec leaves everything behind the
// return value untouched, its native ones spill at most 7 bytes): known-size decodes produce exactly dst_cap[i] bytes per
// block, so maximal runs of adjacent slots go back in one transfer each; encoders and the unknown-size decoder are
// compacted on the device (the same kernel as the packed encode), cross PCIe as one packed transfer into a pinned bounce
// buffer and are scattered to dst + dst_off[i] from there.  Chunks of at most 8 blocks copy block by block.
int run_host(lz4b200_ctx* c, const uint8_t* src, const int64_t* src_off, const int32_t* src_len,
             uint8_t* dst, const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n, int op)
{
    const bool decode = op >= 2;
    const bool src_pageable = is_pageable(src), dst_pageable = is_pageable(dst);
    int32_t b0 = 0; int k = 0;
    enum Mode { PER_BLOCK, RUNS, PACKED };
    struct Pending { int32_t b0, b1; int64_t dlo; Mode mode; int32_t* h_out; int64_t* h_off; };
    Pending pend[NSLOT]; bool busy[NSLOT] = {false, false, false};
    // whatever happens, nothing of this call is still in flight when it returns (the staging buffers are reused)
    struct Drain { lz4b200_ctx* c; ~Drain() { for (int i = 0; i < NSLOT; i++) cudaStreamSynchronize(c->slot[i].stream); } } drain{c};

    auto retire = [&](int s) -> int {
        // outputs of slot s are on the host once its event has fired; scatter out_len and (if needed) per-block payloads
        if (!busy[s]) return LZ4B200_OK;
        busy[s] = false;
        Slot& sl = c->slot[s];
        CU(cudaEventSynchronize(sl.done));
        Pending& p = pend[s];
        const int32_t m = p.b1 - p.b0;
        std::memcpy(out_len + p.b0, p.h_out, sizeof(int32_t) * (size_t)m);
        if (p.mode == PER_BLOCK) {
            for (int32_t i = p.b0; i < p.b1; i++) {
                int32_t r = out_len[i];
                int64_t nbytes = op == 2 ? (r >= 0 ? dst_cap[i] : 0) : std::max(r, 0);
                if (nbytes > 0)
                    CU(cudaMemcpyAsync(dst + dst_off[i], (uint8_t*)sl.dst.p + (dst_off[i] - p.dlo), (size_t)nbytes,
                                       cudaMemcpyDeviceToHost, sl.stream));
            }
            CU(cudaStreamSynchronize(sl.stream));
        } else if (p.mode == PACKED) {
            const int64_t total = p.h_off[m];
            if (total > 0) {
                CU(sl.bounce.reserve((size_t)total));
                CU(cudaMemcpyAsync(sl.bounce.p, sl.packed.p, (size_t)total, cudaMemcpyDeviceToHost, sl.stream));
                CU(cudaStreamSynchronize(sl.stream));
                const int64_t* h_off = p.h_off; const int32_t pb0 = p.b0; const uint8_t* bounce = (const uint8_t*)sl.bounce.p;
                par_ranges((size_t)m, total >= (int64_t)STAGE_PARALLEL_MIN ? 1 : (size_t)m + 1, [&](size_t lo, size_t hi) {
                    for (size_t i = lo; i < hi; i++) {
                        const int64_t nb = h_off[i + 1] - h_off[i];
                        if (nb > 0) std::memcpy(dst + dst_off[pb0 + (int32_t)i], bounce + h_off[i], (size_t)nb);
                    }
                });
            }
        } else if (p.mode == RUNS && dst_pageable) {
            // the runs landed in the slot's pinned buffer (same layout as the device buffer): out to the caller's memory
            int32_t r0 = p.b0;
            for (int32_t i = p.b0 + 1; i <= p.b1; i++) {
                if (i == p.b1 || dst_off[i] != dst_off[i - 1] + dst_cap[i - 1]) {
                    const int64_t lo = dst_off[r0], hi = dst_off[i - 1] + dst_cap[i - 1];
                    if (hi > lo) par_memcpy(dst + lo, (const uint8_t*)sl.hdst.p + (lo - p.dlo), (size_t)(hi - lo));
                    r0 = i;
                }
            }
        }
        return LZ4B200_OK;
    };

    while (b0 < n) {
        // ---- pick the chunk [b0, b1): bounded raw bytes ----
        int64_t bytes = 0; int32_t b1 = b0;
        while (b1 < n) {
            int64_t w = std::max<int64_t>(src_len[b1], 0) + std::max<int64_t>(dst_cap[b1], 0);
            if (b1 > b0 && bytes + w > (int64_t)c->host_chunk_bytes) break;
            bytes += w; b1++;
        }
        const int s = k % NSLOT; k++;
        int rc = retire(s); if (rc) return rc;
        Slot& sl = c->slot[s];
        const int32_t m = b1 - b0;
        int64_t slo = INT64_MAX, shi = INT64_MIN, dlo = INT64_MAX, dhi = INT64_MIN;
        for (int32_t i = b0; i < b1; i++) {
            if (src_len[i] < 0 || dst_cap[i] < 0) return fail(LZ4B200_E_ARG, "negative block length");
            slo = std::min(slo, src_off[i]); shi = std::max(shi, src_off[i] + src_len[i]);
            dlo = std::min(dlo, dst_off[i]); dhi = std::max(dhi, dst_off[i] + dst_cap[i]);
        }
        const Mode mode = m <= 8 ? PER_BLOCK : (op == 2 ? RUNS : PACKED);
        const size_t sbytes = (size_t)(shi - slo), dbytes = (size_t)(dhi - dlo);
        CU(sl.src.reserve(sbytes + 64)); CU(sl.dst.reserve(dbytes + 64));
        const size_t meta_bytes = (size_t)m * (8 + 4 + 8 + 4 + 4) + sizeof(int64_t) * (size_t)(m + 2);
        CU(sl.meta.reserve(meta_bytes)); CU(sl.hmeta.reserve(meta_bytes));
        // meta layout: int64 src_off[m] | int64 dst_off[m] | int32 src_len[m] | int32 dst_cap[m] | int32 out_len[m] | (host only) int64 packed_off[m+1]
        int64_t* h_so = (int64_t*)sl.hmeta.p; int64_t* h_do = h_so + m;
        int32_t* h_sl = (int32_t*)(h_do + m); int32_t* h_dc = h_sl + m; int32_t* h_out = h_dc + m;
        int64_t* h_off = (int64_t*)(((uintptr_t)(h_out + m) + 7) & ~(uintptr_t)7);
        for (int32_t i = 0; i < m; i++) {
            h_so[i] = src_off[b0 + i] - slo; h_do[i] = dst_off[b0 + i] - dlo;
            h_sl[i] = src_len[b0 + i]; h_dc[i] = dst_cap[b0 + i];
        }
        uint8_t* d_meta = (uint8_t*)sl.meta.p;
        CU(cudaMemcpyAsync(d_meta, sl.hmeta.p, (size_t)m * 24, cudaMemcpyHostToDevice, sl.stream));
        if (sbytes) {
            const uint8_t* from = src + slo;
            if (src_pageable && m > 8) { CU(sl.hsrc.reserve(sbytes)); par_memcpy(sl.hsrc.p, from, sbytes); from = (const uint8_t*)sl.hsrc.p; }
            CU(cudaMemcpyAsync(sl.src.p, from, sbytes, cudaMemcpyHostToDevice, sl.stream));
        }
        BatchArgs a;
        a.src = (const uint8_t*)sl.src.p; a.dst = (uint8_t*)sl.dst.p;
        a.src_off = (const int64_t*)d_meta; a.dst_off = a.src_off + m;
        a.src_len = (const int32_t*)(a.dst_off + m); a.dst_cap = a.src_len + m;
        a.out_len = (int32_t*)(a.dst_cap + m); a.n_blocks = m;
        int lanes = 0;
        if (decode && c->decode_lanes_auto) {
            double cs = 0, rs = 0;
            for (int32_t i = b0; i < b1; i++) { cs += src_len[i]; rs += dst_cap[i]; }
            lanes = lanes_for_ratio(rs > 0 ? cs / rs : 1.0, m, c->dev);
        }
        rc = run_device(c, a, op, sl.stream, lanes); if (rc) return rc;
        if (mode == PACKED) {
            CU(sl.packed.reserve(dbytes + 64)); CU(sl.offs.reserve(sizeof(int64_t) * (size_t)(m + 1))); CU(sl.scan.reserve(compact_tmp_bytes(m)));
            cudaError_t e = launch_compact(a.dst, a.dst_off, a.out_len, (uint8_t*)sl.packed.p, (int64_t*)sl.offs.p, m,
                                           sl.scan.p, sl.scan.cap, c->dev, sl.stream, &c->launches);
            if (e != cudaSuccess) return cuda_fail(e, "compact launch");
            CU(cudaMemcpyAsync(h_off, sl.offs.p, sizeof(int64_t) * (size_t)(m + 1), cudaMemcpyDeviceToHost, sl.stream));
        }
        CU(cudaMemcpyAsync(h_out, a.out_len, sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToHost, sl.stream));
        if (mode == RUNS) {
            if (dst_pageable) CU(sl.hdst.reserve(dbytes));
            int32_t r0 = b0;
            for (int32_t i = b0 + 1; i <= b1; i++) {
                if (i == b1 || dst_off[i] != dst_off[i - 1] + dst_cap[i - 1]) {
                    const int64_t lo = dst_off[r0], hi = dst_off[i - 1] + dst_cap[i - 1];
                    uint8_t* to = dst_pageable ? (uint8_t*)sl.hdst.p + (lo - dlo) : dst + lo;
                    if (hi > lo) CU(cudaMemcpyAsync(to, (uint8_t*)sl.dst.p + (lo - dlo), (size_t)(hi - lo), cudaMemcpyDeviceToHost, sl.stream));
                    r0 = i;
                }
            }
        }
        CU(cudaEventRecord(sl.done, sl.stream));
        pend[s] = Pending{b0, b1, dlo, mode, h_out, h_off}; busy[s] = true;
        b0 = b1;
    }
    for (int i = 0; i < NSLOT; i++) { int rc = retire((k + i) % NSLOT); if (rc) return rc; }
    return LZ4B200_OK;
}

// Host-memory encode with PACKED output: per chunk  H2D(raw) -> encode into device slots -> compact on the device ->
// D2H(exactly the compressed bytes).  Only compLen bytes per block cross PCIe on the way back (LZ4Stream / RPC payloads
// want the packed form anyway).  out_off[n+1] receives the byte offset of every block's payload in dst.
int run_host_encode_packed(lz4b200_ctx* c, const uint8_t* src, const int64_t* src_off, const int32_t* src_len,
                           const int32_t* dst_cap, uint8_t* dst, int64_t dst_total_cap, int64_t* out_off, int32_t* out_len,
                           int32_t n, int op)
{
    const bool src_pageable = is_pageable(src), dst_pageable = is_pageable(dst);
    int32_t b0 = 0; int k = 0; int64_t written = 0;
    struct Pending { int32_t b0, b1; int32_t* h_out; int64_t* h_off; };
    Pending pend[NSLOT]; bool busy[NSLOT] = {false, false, false};
    struct Drain { lz4b200_ctx* c; ~Drain() { for (int i = 0; i < NSLOT; i++) cudaStreamSynchronize(c->slot[i].stream); } } drain{c};

    auto retire = [&](int s) -> int {
        if (!busy[s]) return LZ4B200_OK;
        Slot& sl = c->slot[s]; Pending& p = pend[s];
        CU(cudaStreamSynchronize(sl.stream));                        // lengths and local offsets are on the host now
        const int32_t m = p.b1 - p.b0;
        const int64_t total = p.h_off[m];
        if (written + total > dst_total_cap) return fail(LZ4B200_E_ARG, "packed destination too small");
        const bool stage = dst_pageable && total > 0;
        if (stage) CU(sl.hdst.reserve((size_t)total));
        if (total > 0) CU(cudaMemcpyAsync(stage ? sl.hdst.p : (void*)(dst + written), sl.packed.p, (size_t)total, cudaMemcpyDeviceToHost, sl.stream));
        std::memcpy(out_len + p.b0, p.h_out, sizeof(int32_t) * (size_t)m);
        for (int32_t i = 0; i < m; i++) out_off[p.b0 + i] = written + p.h_off[i];
        CU(cudaStreamSynchronize(sl.stream));
        if (stage) par_memcpy(dst + written, sl.hdst.p, (size_t)total);
        written += total;
        busy[s] = false;
        return LZ4B200_OK;
    };

    while (b0 < n) {
        int64_t bytes = 0; int32_t b1 = b0;
        while (b1 < n) {
            if (src_len[b1] < 0 || dst_cap[b1] < 0) return fail(LZ4B200_E_ARG, "negative block length");
            int64_t w = (int64_t)src_len[b1] + dst_cap[b1];
            if (b1 > b0 && bytes + w > (int64_t)c->host_chunk_bytes) break;
            bytes += w; b1++;
        }
        const int s = k % NSLOT; k++;
        // payloads must land in block order: retire every older chunk first (its D2H overlaps this chunk's H2D + kernel
        // only through the other slots' streams)
        int rc = retire(s); if (rc) return rc;
        Slot& sl = c->slot[s];
        const int32_t m = b1 - b0;
        int64_t slo = INT64_MAX, shi = INT64_MIN, dsum = 0;
        for (int32_t i = b0; i < b1; i++) { slo = std::min(slo, src_off[i]); shi = std::max(shi, src_off[i] + src_len[i]); dsum += dst_cap[i]; }
        const size_t sbytes = (size_t)(shi - slo);
        CU(sl.src.reserve(sbytes + 64)); CU(sl.dst.reserve((size_t)dsum + 64)); CU(sl.packed.reserve((size_t)dsum + 64));
        CU(sl.offs.reserve(sizeof(int64_t) * (size_t)(m + 1))); CU(sl.scan.reserve(compact_tmp_bytes(m)));
        const size_t meta_bytes = (size_t)m * 28 + sizeof(int64_t) * (size_t)(m + 1);
        CU(sl.meta.reserve((size_t)m * 28)); CU(sl.hmeta.reserve(meta_bytes + 64));
        int64_t* h_so = (int64_t*)sl.hmeta.p; int64_t* h_do = h_so + m;
        int32_t* h_sl = (int32_t*)(h_do + m); int32_t* h_dc = h_sl + m; int32_t* h_out = h_dc + m;
        int64_t* h_off = (int64_t*)(((uintptr_t)(h_out + m) + 7) & ~(uintptr_t)7);
        int64_t acc = 0;
        for (int32_t i = 0; i < m; i++) {
            h_so[i] = src_off[b0 + i] - slo; h_do[i] = acc; acc += dst_cap[b0 + i];
            h_sl[i] = src_len[b0 + i]; h_dc[i] = dst_cap[b0 + i];
        }
        uint8_t* d_meta = (uint8_t*)sl.meta.p;
        CU(cudaMemcpyAsync(d_meta, sl.hmeta.p, (size_t)m * 24, cudaMemcpyHostToDevice, sl.stream));
        if (sbytes) {
            const uint8_t* from = src + slo;
            if (src_pageable && m > 8) { CU(sl.hsrc.reserve(sbytes)); par_memcpy(sl.hsrc.p, from, sbytes); from = (const uint8_t*)sl.hsrc.p; }
            CU(cudaMemcpyAsync(sl.src.p, from, sbytes, cudaMemcpyHostToDevice, sl.stream));
        }
        BatchArgs a;
        a.src = (const uint8_t*)sl.src.p; a.dst = (uint8_t*)sl.dst.p;
        a.src_off = (const int64_t*)d_meta; a.dst_off = a.src_off + m;
        a.src_len = (const int32_t*)(a.dst_off + m); a.dst_cap = a.src_len + m;
        a.out_len = (int32_t*)(a.dst_cap + m); a.n_blocks = m;
        rc = run_device(c, a, op, sl.stream); if (rc) return rc;
        cudaError_t e = launch_compact(a.dst, a.dst_off, a.out_len, (uint8_t*)sl.packed.p, (int64_t*)sl.offs.p, m,
                                       sl.scan.p, sl.scan.cap, c->dev, sl.stream, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "compact launch");
        CU(cudaMemcpyAsync(h_out, a.out_len, sizeof(int32_t) * (size_t)m, cudaMemcpyDeviceToHost, sl.stream));
        CU(cudaMemcpyAsync(h_off, sl.offs.p, sizeof(int64_t) * (size_t)(m + 1), cudaMemcpyDeviceToHost, sl.stream));
        pend[s] = Pending{b0, b1, h_out, h_off}; busy[s] = true;
        b0 = b1;
    }
    for (int i = 0; i < NSLOT; i++) { int rc = retire((k + i) % NSLOT); if (rc) return rc; }
    out_off[n] = written;
    return LZ4B200_OK;
}

int batch(lz4b200_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, void* dst,
          const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n, int op, int mem, void* stream)
{
    if (!c) return fail(LZ4B200_E_ARG, "null context");
    if (n < 0) return fail(LZ4B200_E_ARG, "negative block count");
    if (n == 0) return LZ4B200_OK;
    if (!src_off || !src_len || !dst_off || !dst_cap || !out_len || !src || !dst) return fail(LZ4B200_E_ARG, "null argument");
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    if (mem == LZ4B200_MEM_DEVICE) {
        BatchArgs a{(const uint8_t*)src, src_off, src_len, (uint8_t*)dst, dst_off, dst_cap, out_len, n};
        return run_device(c, a, op, (cudaStream_t)stream);
    }
    if (mem != LZ4B200_MEM_HOST) return fail(LZ4B200_E_ARG, "mem must be LZ4B200_MEM_HOST or LZ4B200_MEM_DEVICE");
    return run_host(c, (const uint8_t*)src, src_off, src_len, (uint8_t*)dst, dst_off, dst_cap, out_len, n, op);
}

// ---- LZ4Stream framing on device memory (stream.cu) -------------------------------------------------------------------
// The same byte stream as framing.cpp, without the bytes leaving the GPU.  Every call runs on the caller's stream and
// waits for its own result there, so it is ordered after whatever the caller queued before it.

// groups of chunks bound the device scratch, like the host framing: 256 MiB of raw bytes, and at most 4 Mi chunks
// (44 bytes of metadata each) for tiny block sizes
constexpr int64_t STREAM_GROUP_BYTES = 256 << 20, STREAM_GROUP_CHUNKS = 1 << 22;

int64_t stream_encode_device(lz4b200_ctx* c, const uint8_t* src, int64_t n, int32_t bs, int hc, uint8_t* dst, cudaStream_t st)
{
    const int64_t chunks = (n + bs - 1) / bs;
    const int64_t group = std::min(std::max<int64_t>(1, STREAM_GROUP_BYTES / bs), STREAM_GROUP_CHUNKS);
    const int64_t gm = std::min(chunks, group);
    // work buffer: slots (capacity == raw length, LZ4Stream.cs:243-246) | int64 off[m] | int64 pos[2m+1] | int32 len[m] | out[m] | sizes[2m]
    const size_t slot_bytes = ((size_t)std::min<int64_t>(n, gm * bs) + 15) & ~(size_t)15;
    CU(c->stream_work.reserve(slot_bytes + (size_t)gm * 44 + 64));
    CU(c->stream_res.reserve(sizeof(StreamWalk)));
    CU(c->stream_host.reserve(sizeof(StreamWalk)));
    if (compact_tmp_bytes((int32_t)(2 * gm)) > c->compact_tmp.cap) { CU(cudaDeviceSynchronize()); CU(c->compact_tmp.reserve(compact_tmp_bytes((int32_t)(2 * gm)))); }
    uint8_t* slots = (uint8_t*)c->stream_work.p;
    int64_t* off = (int64_t*)(slots + slot_bytes);
    int64_t* pos = off + gm;
    int32_t* len = (int32_t*)(pos + 2 * gm + 1);
    int32_t* out = len + gm;
    int32_t* sizes = out + gm;
    int64_t* h_total = (int64_t*)c->stream_host.p;
    int64_t w = 0;
    for (int64_t c0 = 0; c0 < chunks; c0 += group) {
        const int32_t m = (int32_t)std::min(chunks - c0, group);
        const int64_t base = c0 * bs;
        cudaError_t e = launch_stream_layout(off, len, m, bs, n - base, st, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "stream layout launch");
        BatchArgs a{src + base, off, len, slots, off, len, out, m};
        int rc = run_device(c, a, hc ? 1 : 0, st); if (rc) return rc;
        e = launch_stream_frame_sizes(len, out, m, hc, sizes, st, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "stream frame sizes launch");
        CU(cudaStreamWaitEvent(st, c->compact_done, 0));            // the scan scratch is shared with lz4b200_compact
        e = launch_compact(nullptr, nullptr, sizes, nullptr, pos, 2 * m, c->compact_tmp.p, c->compact_tmp.cap, c->dev, st, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "stream scan launch");
        CU(cudaEventRecord(c->compact_done, st));
        e = launch_stream_frame_write(src + base, off, len, slots, out, pos, m, hc, dst + w, st, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "stream frame write launch");
        CU(cudaMemcpyAsync(h_total, pos + 2 * m, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));                              // the next group reuses the slots and needs w
        w += *h_total;
    }
    return w;
}

// one walk of the chunk headers into the context's table (cap entries per table; 0 = count only); result on the host
int stream_walk(lz4b200_ctx* c, const uint8_t* src, int64_t n, int64_t cap, cudaStream_t st, StreamWalk* out)
{
    CU(c->stream_res.reserve(sizeof(StreamWalk)));
    CU(c->stream_host.reserve(sizeof(StreamWalk)));
    if (cap) CU(c->stream_table.reserve(stream_table_bytes(cap)));
    const StreamTable t = stream_table_at(c->stream_table.p, cap);
    cudaError_t e = launch_stream_walk(src, n, cap, t, (StreamWalk*)c->stream_res.p, st, &c->launches);
    if (e != cudaSuccess) return cuda_fail(e, "stream walk launch");
    CU(cudaMemcpyAsync(c->stream_host.p, c->stream_res.p, sizeof(StreamWalk), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *out = *(const StreamWalk*)c->stream_host.p;
    return LZ4B200_OK;
}

int64_t stream_decode_device(lz4b200_ctx* c, const uint8_t* src, int64_t n, uint8_t* dst, int64_t dst_cap, cudaStream_t st)
{
    // every chunk has at least two header bytes; start from a guess for chunks of a few KiB and walk again if it was short
    int64_t cap = std::max<int64_t>((int64_t)(c->stream_table.cap / stream_table_bytes(1)), std::min(n / 2 + 1, n / 4096 + 1024));
    StreamWalk r;
    int rc = stream_walk(c, src, n, cap, st, &r); if (rc) return rc;
    if (r.status == 0 && std::max(r.n_stored, r.n_comp) > cap) {
        cap = std::max(r.n_stored, r.n_comp);
        rc = stream_walk(c, src, n, cap, st, &r); if (rc) return rc;
    }
    if (r.status < 0) return r.status;
    if (r.total > dst_cap || (r.total > 0 && !dst)) return fail(LZ4B200_E_ARG, "destination too small");
    if (std::max(r.n_stored, r.n_comp) > INT32_MAX) return fail(LZ4B200_E_ARG, "more than 2^31 chunks");
    const StreamTable t = stream_table_at(c->stream_table.p, cap);
    cudaError_t e = launch_scatter(src, t.st_src, t.st_len, dst, t.st_dst, (int32_t)r.n_stored, st, &c->launches);   // stored chunks (:295-299)
    if (e != cudaSuccess) return cuda_fail(e, "stream stored-chunk copy launch");
    if (r.n_comp > 0) {
        const int32_t m = (int32_t)r.n_comp;
        BatchArgs a{src, t.cp_src, t.cp_len, dst, t.cp_dst, t.cp_raw, t.cp_out, m};
        rc = run_device(c, a, 2, st); if (rc) return rc;
        // LZ4Codec.Decode(..., knownOutputLength: true) throws unless exactly compLen bytes were consumed
        // (src/LZ4ps/LZ4Codec.Safe.cs:539-542)
        StreamWalk* res = (StreamWalk*)c->stream_res.p;
        e = launch_stream_verdict(t.cp_out, t.cp_len, m, &res->bad, c->dev, st, &c->launches);
        if (e != cudaSuccess) return cuda_fail(e, "stream verdict launch");
        CU(cudaMemcpyAsync(c->stream_host.p, res, sizeof(StreamWalk), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    if (r.n_comp > 0 && ((const StreamWalk*)c->stream_host.p)->bad) return LZ4B200_E_FORMAT;
    return r.total;
}

// The single-block entry points are re-entrant like the reference's (SURVEY 8b "Threading"): every calling thread gets
// a context of its own (streams + staging buffers), created on first use and destroyed with the thread.
struct ThreadCtx {
    lz4b200_ctx* c = nullptr;
    ~ThreadCtx() { if (c) lz4b200_destroy(c); }
};
thread_local ThreadCtx g_thread_ctx;

lz4b200_ctx* default_ctx()
{
    if (!g_thread_ctx.c) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
        if (lz4b200_create(&g_thread_ctx.c, dev) != LZ4B200_OK) g_thread_ctx.c = nullptr;
    }
    return g_thread_ctx.c;
}

int single(const char* source, char* dest, int isize, int ocap, int op)
{
    lz4b200_ctx* c = default_ctx();
    if (!c) return op >= 2 ? -1 : 0;               // no device: encoders report failure (0), decoders an error (<0)
    if (!source || !dest || isize < 0 || ocap < 0) return op >= 2 ? -1 : 0;
    int64_t so = 0, dof = 0; int32_t sl = isize, dc = ocap, out = op >= 2 ? -1 : 0;
    // zero-length buffers still need valid pointers for the staging copies
    int rc = batch(c, source, &so, &sl, dest, &dof, &dc, &out, 1, op, LZ4B200_MEM_HOST, nullptr);
    if (rc != LZ4B200_OK) return op >= 2 ? -1 : 0;
    return out;
}

}  // namespace

extern "C" {

int lz4b200_version(void) { return LZ4B200_VERSION; }
const char* lz4b200_last_error(void) { return g_err.c_str(); }

int lz4b200_device_count(void)
{
    int n = 0, ok = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    for (int i = 0; i < n; i++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

int lz4b200_compress_bound(int n) { return n < 0 ? 0 : n + n / 255 + 16; }

int lz4b200_create(lz4b200_ctx** out, int device)
{
    if (!out) return fail(LZ4B200_E_ARG, "null out pointer");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return fail(LZ4B200_E_NODEVICE, "no CUDA device"); }
    if (device < 0 || device >= n) return fail(LZ4B200_E_ARG, "device index out of range");
    int major = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    if (major != 10) return fail(LZ4B200_E_NODEVICE, "device is not compute capability 10.x (this library holds sm_100a code only)");
    DeviceGuard g(device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    lz4b200_ctx* c = new lz4b200_ctx();
    c->device = device;
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device); c->dev.num_sms = v;
    cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device); c->dev.smem_per_sm = v;
    cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device); c->dev.smem_optin = v;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&c->counters, sizeof(uint32_t) * NCOUNTER);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->hc_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->compact_done, cudaEventDisableTiming);
    for (int i = 0; i < NSLOT && e == cudaSuccess; i++) {
        e = cudaStreamCreateWithFlags(&c->slot[i].stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->slot[i].done, cudaEventDisableTiming);
    }
    if (e != cudaSuccess) { int rc = cuda_fail(e, "context creation"); lz4b200_destroy(c); return rc; }
    *out = c;
    return LZ4B200_OK;
}

void lz4b200_destroy(lz4b200_ctx* c)
{
    if (!c) return;
    DeviceGuard g(c->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < NSLOT; i++) {
        Slot& s = c->slot[i];
        s.src.release(); s.dst.release(); s.meta.release(); s.hmeta.release(); s.packed.release(); s.offs.release(); s.scan.release(); s.bounce.release(); s.hsrc.release(); s.hdst.release();
        if (s.done) cudaEventDestroy(s.done);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    c->hc_arena.release(); c->compact_tmp.release();
    c->stream_work.release(); c->stream_table.release(); c->stream_res.release(); c->stream_host.release();
    if (c->hc_done) cudaEventDestroy(c->hc_done);
    if (c->compact_done) cudaEventDestroy(c->compact_done);
    if (c->counters) cudaFree(c->counters);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int lz4b200_synchronize(lz4b200_ctx* c)
{
    if (!c) return fail(LZ4B200_E_ARG, "null context");
    DeviceGuard g(c->device);
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < NSLOT; i++) CU(cudaStreamSynchronize(c->slot[i].stream));
    return LZ4B200_OK;
}

int lz4b200_encode_batch(lz4b200_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, void* dst,
                         const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n, int mode, int mem, void* stream)
{
    if (mode != LZ4B200_MODE_FAST && mode != LZ4B200_MODE_HC) return fail(LZ4B200_E_ARG, "unknown encoder mode");
    return batch(c, src, src_off, src_len, dst, dst_off, dst_cap, out_len, n, mode == LZ4B200_MODE_HC ? 1 : 0, mem, stream);
}

int lz4b200_encode_batch_packed(lz4b200_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len,
                                const int32_t* dst_cap, void* dst, int64_t dst_total_cap, int64_t* out_off, int32_t* out_len,
                                int32_t n, int mode)
{
    if (!c) return fail(LZ4B200_E_ARG, "null context");
    if (mode != LZ4B200_MODE_FAST && mode != LZ4B200_MODE_HC) return fail(LZ4B200_E_ARG, "unknown encoder mode");
    if (n < 0 || !out_off) return fail(LZ4B200_E_ARG, "bad argument");
    if (n == 0) { out_off[0] = 0; return LZ4B200_OK; }
    if (!src || !src_off || !src_len || !dst_cap || !dst || !out_len) return fail(LZ4B200_E_ARG, "null argument");
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    return run_host_encode_packed(c, (const uint8_t*)src, src_off, src_len, dst_cap, (uint8_t*)dst, dst_total_cap, out_off, out_len,
                                  n, mode == LZ4B200_MODE_HC ? 1 : 0);
}

int lz4b200_decode_batch(lz4b200_ctx* c, const void* src, const int64_t* src_off, const int32_t* src_len, void* dst,
                         const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n, int known_len, int mem, void* stream)
{
    return batch(c, src, src_off, src_len, dst, dst_off, dst_cap, out_len, n, known_len ? 2 : 3, mem, stream);
}

int lz4b200_compact(lz4b200_ctx* c, const void* slots, const int64_t* slot_off, const int32_t* len, void* packed,
                    int64_t* out_off, int32_t n, void* stream)
{
    if (!c || !slot_off || !len || !out_off || n < 0) return fail(LZ4B200_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) { CU(cudaMemsetAsync(out_off, 0, sizeof(int64_t), st)); return LZ4B200_OK; }     // out_off[0] = total = 0
    if (compact_tmp_bytes(n) > c->compact_tmp.cap) { CU(cudaDeviceSynchronize()); CU(c->compact_tmp.reserve(compact_tmp_bytes(n))); }
    // one scan scratch per context: compactions on different streams are serialised on it
    CU(cudaStreamWaitEvent(st, c->compact_done, 0));
    cudaError_t e = launch_compact((const uint8_t*)slots, slot_off, len, (uint8_t*)packed, out_off, n,
                                   c->compact_tmp.p, c->compact_tmp.cap, c->dev, st, &c->launches);
    if (e != cudaSuccess) return cuda_fail(e, "compact launch");
    CU(cudaEventRecord(c->compact_done, st));
    return LZ4B200_OK;
}

int lz4b200_synth_fill(lz4b200_ctx* c, void* dst, int64_t n_blocks, int32_t block_size, int cls, uint64_t seed,
                       int64_t first_block, void* stream)
{
    if (!c || !dst) return fail(LZ4B200_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    cudaError_t e = launch_synth((uint8_t*)dst, n_blocks, block_size, cls, seed, first_block, c->dev,
                                 (cudaStream_t)stream, &c->launches);
    if (e != cudaSuccess) return cuda_fail(e, "synth launch");
    return LZ4B200_OK;
}

int lz4b200_set_option(lz4b200_ctx* c, const char* key, int64_t value)
{
    if (!c || !key) return fail(LZ4B200_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(c->mu);
    std::string k(key);
    if (k == "decode_lanes") {
        const int64_t g = value % 100;                 // 100 + G = the output-staged variant of the G-lane decoder
        const bool lpb = value == 1;                   // one lane per block (lz4_decode_lpb.cuh)
        if (!lpb && ((g != 4 && g != 8 && g != 16 && g != 32) || (value != g && value != 100 + g))) return fail(LZ4B200_E_ARG, "decode_lanes must be 1, 4, 8, 16, 32 (or 100 + one of the last four)");
        c->decode_lanes = (int)value; c->decode_lanes_auto = false;
    }
    else if (k == "decode_lanes_auto") { c->decode_lanes_auto = value != 0; }
    else if (k == "encode_variant") { if (value != 1 && value != 2) return fail(LZ4B200_E_ARG, "encode_variant must be 1 or 2"); c->encode_variant = (int)value; }
    else if (k == "encode_prefetch") { if (value < -65536 || value > 65536) return fail(LZ4B200_E_ARG, "encode_prefetch out of range"); c->encode_tune[0] = (int)value; }
    else if (k == "encode_lane_copy_max" || k == "encode_probe_max" || k == "encode_wide_min") {
        if (value < 0 || value > 65536) return fail(LZ4B200_E_ARG, "encoder heuristic out of range");
        c->encode_tune[k == "encode_lane_copy_max" ? 1 : (k == "encode_probe_max" ? 2 : 3)] = (int)value;
    }
    else if (k == "encode_ctas_per_sm") { if (value < 0 || value > 32) return fail(LZ4B200_E_ARG, "encode_ctas_per_sm out of range"); c->encode_ctas_per_sm = (int)value; }
    else if (k == "hc_concurrency") {
        if (value < 32 || value > (1 << 20)) return fail(LZ4B200_E_ARG, "hc_concurrency out of range");
        DeviceGuard g(c->device);
        cudaDeviceSynchronize();
        c->hc_arena.release();
        c->hc_concurrency = (int)value;
    }
    else if (k == "hc_kernel") { if (value < -1 || value > 2) return fail(LZ4B200_E_ARG, "hc_kernel must be -1 (chosen per batch), 0 (thread per block), 1 or 2 (warp per block on a static index: block in shared memory / read through L1)"); c->hc_kernel = (int)value; }
    else if (k == "hc_warps_per_sm") { if (value < 0 || value > 32) return fail(LZ4B200_E_ARG, "hc_warps_per_sm must be 0..32"); c->hc_warps_per_sm = (int)value; }
    else if (k == "host_chunk_mb") { if (value < 1 || value > 4096) return fail(LZ4B200_E_ARG, "host_chunk_mb out of range"); c->host_chunk_bytes = (size_t)value << 20; }
    else return fail(LZ4B200_E_ARG, "unknown option");
    return LZ4B200_OK;
}

int lz4b200_get_option(lz4b200_ctx* c, const char* key, int64_t* value)
{
    if (!c || !key || !value) return fail(LZ4B200_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lock(c->mu);
    const std::string k(key);
    if (k == "hc_kernel") *value = c->hc_kernel;
    else if (k == "hc_warps_per_sm") *value = c->hc_warps_per_sm;
    else if (k == "hc_concurrency") *value = c->hc_concurrency;
    else if (k == "decode_lanes") *value = c->decode_lanes_auto ? 0 : c->decode_lanes;
    else if (k == "encode_variant") *value = c->encode_variant;
    else if (k == "encode_ctas_per_sm") *value = c->encode_ctas_per_sm;
    else return fail(LZ4B200_E_ARG, "unknown option");
    return LZ4B200_OK;
}

int64_t lz4b200_launch_count(lz4b200_ctx* c) { return c ? c->launches : 0; }

int lz4b200_host_register(void* ptr, int64_t bytes)
{
    if (!ptr || bytes <= 0) return fail(LZ4B200_E_ARG, "bad argument");
    CU(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
    return LZ4B200_OK;
}
int lz4b200_host_unregister(void* ptr)
{
    if (!ptr) return fail(LZ4B200_E_ARG, "bad argument");
    CU(cudaHostUnregister(ptr));
    return LZ4B200_OK;
}

int lz4b200_peer_copy(void* dst, const void* src, int64_t bytes, void* stream)
{
    if (bytes < 0 || (bytes && (!dst || !src))) return fail(LZ4B200_E_ARG, "bad argument");
    if (!bytes) return LZ4B200_OK;
    int cur = 0, dev[2];
    CU(cudaGetDevice(&cur));
    const void* ends[2] = {dst, src};
    for (int k = 0; k < 2; k++) {
        cudaPointerAttributes at{};
        CU(cudaPointerGetAttributes(&at, ends[k]));
        if (at.type != cudaMemoryTypeDevice) return fail(LZ4B200_E_ARG, "lz4b200_peer_copy: both buffers must be device memory");
        dev[k] = at.device;
    }
    for (int k = 0; k < 2; k++) {                                // both directions of the pair, once
        CU(cudaSetDevice(dev[k]));
        cudaError_t e = cudaDeviceEnablePeerAccess(dev[1 - k], 0);
        (void)cudaGetLastError();
        if (dev[0] != dev[1] && e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaSetDevice(cur); return cuda_fail(e, "cudaDeviceEnablePeerAccess"); }
    }
    CU(cudaSetDevice(cur));
    CU(cudaMemcpyPeerAsync(dst, dev[0], src, dev[1], (size_t)bytes, (cudaStream_t)stream));   // a copy-engine transfer
    return LZ4B200_OK;
}

int64_t lz4b200_stream_encode_device(lz4b200_ctx* c, const void* src, int64_t n, int32_t block_size, int high_compression,
                                     void* dst, int64_t dst_cap, void* stream)
{
    if (!c || n < 0 || block_size < 1 || (n > 0 && (!src || !dst))) return fail(LZ4B200_E_ARG, "bad argument");
    if (dst_cap < lz4b200_stream_bound(n, block_size)) return fail(LZ4B200_E_ARG, "dst_cap is below lz4b200_stream_bound");
    if (n == 0) return 0;
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    return stream_encode_device(c, (const uint8_t*)src, n, block_size, high_compression ? 1 : 0, (uint8_t*)dst, (cudaStream_t)stream);
}

int64_t lz4b200_stream_decoded_size_device(lz4b200_ctx* c, const void* src, int64_t n, void* stream)
{
    if (!c || n < 0 || (n > 0 && !src)) return fail(LZ4B200_E_ARG, "bad argument");
    if (n == 0) return 0;
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    StreamWalk r;
    const int rc = stream_walk(c, (const uint8_t*)src, n, 0, (cudaStream_t)stream, &r);
    if (rc) return rc;
    return r.status < 0 ? r.status : r.total;
}

int64_t lz4b200_stream_decode_device(lz4b200_ctx* c, const void* src, int64_t n, void* dst, int64_t dst_cap, void* stream)
{
    if (!c || n < 0 || (n > 0 && !src)) return fail(LZ4B200_E_ARG, "bad argument");
    if (n == 0) return dst_cap < 0 ? fail(LZ4B200_E_ARG, "destination too small") : 0;
    std::lock_guard<std::mutex> lock(c->mu);
    DeviceGuard g(c->device);
    if (!g.ok) return fail(LZ4B200_E_CUDA, "cudaSetDevice failed");
    return stream_decode_device(c, (const uint8_t*)src, n, (uint8_t*)dst, dst_cap, (cudaStream_t)stream);
}

int lz4b200_compress_limitedOutput(const char* s, char* d, int isize, int cap) { return single(s, d, isize, cap, 0); }
int lz4b200_compressHC_limitedOutput(const char* s, char* d, int isize, int cap) { return single(s, d, isize, cap, 1); }
int lz4b200_uncompress(const char* s, char* d, int isize, int osize) { return single(s, d, isize, osize, 2); }
int lz4b200_uncompress_unknownOutputSize(const char* s, char* d, int isize, int cap) { return single(s, d, isize, cap, 3); }

}  // extern "C"
