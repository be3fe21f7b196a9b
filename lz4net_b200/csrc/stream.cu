// stream.cu -- LZ4Stream framing on device memory: the kernels behind lz4b200_stream_{encode,decoded_size,decode}_device.
//
// Encode (per group of chunks, after the encode batch has filled one slot per chunk, capacity == raw length):
//   frame sizes  one thread per chunk: header size and payload size (the compressed bytes, or the raw chunk when the
//                encoder did not make it smaller), as two entries of one length array;
//   scan         the exclusive scan of util.cu (launch_compact without a gather) turns them into byte positions;
//   frame write  one warp per chunk: the header, then the payload with 128-bit funnel-shifted moves.
// Decode:
//   chunk walk   ONE thread walks the headers (a chunk's position depends on every header before it: the format is
//                serial) with the step of lz4_stream.cuh, and writes two chunk tables -- stored chunks (copied by
//                gather_blocks) and compressed chunks (one batched decode) -- plus the counts, the total and a status;
//   verdict      a chunk whose LZ4 payload is not consumed exactly is malformed (LZ4Codec.Safe.cs:539-542).
#include "kernels.h"
#include "simt.cuh"
#include "lz4_copy.cuh"
#include "lz4_stream.cuh"

namespace lz4b200 {

// chunk i of a group: bytes [i * bs, i * bs + len[i]) of the group's input, and the same range of its slot buffer
__global__ void __launch_bounds__(256) stream_chunk_layout(int64_t* off, int32_t* len, int32_t m, int32_t bs, int64_t rem)
{
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int64_t o = (int64_t)i * bs;
    off[i] = o;
    len[i] = (int32_t)(rem - o < bs ? rem - o : bs);
}

__global__ void __launch_bounds__(256) stream_frame_sizes(const int32_t* len, const int32_t* out_len, int32_t m, int hc,
                                                          int32_t* sizes)
{
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int32_t raw = len[i], clen = out_len[i];
    sizes[2 * i] = lz4s::header_size(raw, clen, hc != 0);
    sizes[2 * i + 1] = lz4s::chunk_compressed(raw, clen) ? clen : raw;
}

// byte-exact move of l bytes by one warp: byte-wise head up to a 16-byte aligned destination, then aligned 128-bit
// loads funnel-shifted into place (the loop of gather_blocks), byte-wise tail
__device__ __forceinline__ void warp_move(const uint8_t* s, uint8_t* d, int32_t l, int lane)
{
    int head = (int)((16 - ((uintptr_t)d & 15)) & 15); if (head > l) head = l;
    for (int i = lane; i < head; i += 32) d[i] = s[i];
    const int nvec = (l - head) >> 4;
    const uint32_t r = (uint32_t)((uintptr_t)(s + head) & 15);
    const uint8_t* sa = s + head - r;
    for (int v = lane; v < nvec; v += 32) {
        uint4 lo = simt::ldg_nc_v4(sa + 16 * (size_t)v), o = lo;
        if (r) o = shift16(lo, simt::ldg_nc_v4(sa + 16 * (size_t)v + 16), r);
        simt::stg_v4(d + head + 16 * (size_t)v, o);
    }
    for (int i = head + (nvec << 4) + lane; i < l; i += 32) d[i] = s[i];
}

__global__ void __launch_bounds__(256) stream_frame_write(const uint8_t* src, const int64_t* off, const int32_t* len,
                                                          const uint8_t* slots, const int32_t* out_len, const int64_t* pos,
                                                          int32_t m, int hc, uint8_t* dst)
{
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= m) return;
    const int32_t raw = len[i], clen = out_len[i];
    const bool comp = lz4s::chunk_compressed(raw, clen);
    if (lane == 0) {
        uint8_t* p = dst + pos[2 * i];
        p = lz4s::put_varint(p, lz4s::chunk_flags(comp, hc != 0));
        p = lz4s::put_varint(p, (uint64_t)raw);
        if (comp) lz4s::put_varint(p, (uint64_t)clen);
    }
    warp_move((comp ? slots : src) + off[i], dst + pos[2 * i + 1], comp ? clen : raw, lane);
}

__global__ void __launch_bounds__(1) stream_walk(const uint8_t* s, int64_t n, int64_t cap, StreamTable t, StreamWalk* res)
{
    int64_t pos = 0, total = 0, ns = 0, nc = 0, status = 0;
    for (;;) {
        lz4s::Chunk c;
        const int r = lz4s::walk_step(s, n, &pos, &c);
        if (r == 0) break;
        if (r < 0) { status = r; break; }
        if (c.compressed) {
            if (c.raw > 0) {                       // a compressed chunk of 0 bytes decodes to nothing (framing.cpp)
                if (nc < cap) {
                    t.cp_src[nc] = c.payload; t.cp_dst[nc] = total;
                    t.cp_len[nc] = c.stored; t.cp_raw[nc] = c.raw; t.cp_out[nc] = -1;
                }
                nc++;
            }
        } else if (c.raw > 0) {
            if (ns < cap) { t.st_src[ns] = c.payload; t.st_dst[ns] = total; t.st_len[ns] = c.raw; }
            ns++;
        }
        total += c.raw;
    }
    res->status = status; res->total = total; res->n_stored = ns; res->n_comp = nc; res->bad = 0;
}

__global__ void __launch_bounds__(256) stream_verdict(const int32_t* out_len, const int32_t* want, int32_t m, int32_t* bad)
{
    bool mismatch = false;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x)
        mismatch |= out_len[i] != want[i];
    if (__any_sync(0xFFFFFFFFu, mismatch) && (threadIdx.x & 31) == 0) atomicOr(bad, 1);
}

size_t stream_table_bytes(int64_t cap) { return (size_t)cap * (4 * sizeof(int64_t) + 4 * sizeof(int32_t)); }

StreamTable stream_table_at(void* p, int64_t cap)
{
    StreamTable t;
    int64_t* q = (int64_t*)p;
    t.st_src = q; t.st_dst = q + cap; t.cp_src = q + 2 * cap; t.cp_dst = q + 3 * cap;
    int32_t* r = (int32_t*)(q + 4 * cap);
    t.st_len = r; t.cp_len = r + cap; t.cp_raw = r + 2 * cap; t.cp_out = r + 3 * cap;
    return t;
}

static unsigned grid_for(int64_t threads) { return (unsigned)((threads + 255) / 256); }

cudaError_t launch_stream_layout(int64_t* off, int32_t* len, int32_t m, int32_t block_size, int64_t rem,
                                 cudaStream_t stream, int64_t* launches)
{
    stream_chunk_layout<<<grid_for(m), 256, 0, stream>>>(off, len, m, block_size, rem);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_stream_frame_sizes(const int32_t* len, const int32_t* out_len, int32_t m, int hc, int32_t* sizes,
                                      cudaStream_t stream, int64_t* launches)
{
    stream_frame_sizes<<<grid_for(m), 256, 0, stream>>>(len, out_len, m, hc, sizes);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_stream_frame_write(const uint8_t* src, const int64_t* off, const int32_t* len, const uint8_t* slots,
                                      const int32_t* out_len, const int64_t* pos, int32_t m, int hc, uint8_t* dst,
                                      cudaStream_t stream, int64_t* launches)
{
    stream_frame_write<<<(unsigned)(((int64_t)m + 7) / 8), 256, 0, stream>>>(src, off, len, slots, out_len, pos, m, hc, dst);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_stream_walk(const uint8_t* src, int64_t n, int64_t cap, const StreamTable& t, StreamWalk* res,
                               cudaStream_t stream, int64_t* launches)
{
    stream_walk<<<1, 1, 0, stream>>>(src, n, cap, t, res);
    if (launches) ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_stream_verdict(const int32_t* out_len, const int32_t* want, int32_t m, int32_t* bad,
                                  const DeviceInfo& dev, cudaStream_t stream, int64_t* launches)
{
    if (m <= 0) return cudaSuccess;
    const int64_t blocks = (m + 255) / 256;
    stream_verdict<<<(unsigned)(blocks < dev.num_sms * 4 ? blocks : dev.num_sms * 4), 256, 0, stream>>>(out_len, want, m, bad);
    if (launches) ++*launches;
    return cudaGetLastError();
}

}  // namespace lz4b200
