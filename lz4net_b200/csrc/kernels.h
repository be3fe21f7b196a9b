// kernels.h -- internal launcher interface between the C-ABI translation unit and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lz4b200 {

struct BatchArgs {
    const uint8_t* src; const int64_t* src_off; const int32_t* src_len;
    uint8_t* dst; const int64_t* dst_off; const int32_t* dst_cap;
    int32_t* out_len; int32_t n_blocks;
};

struct DeviceInfo { int num_sms; int smem_per_sm; int smem_optin; };

// All launchers are asynchronous on `stream`; `counter` is a device uint32 the launcher zeroes itself (dynamic
// block hand-out).  They return the launch error (cudaSuccess on success) and add to *launches.
// lanes_per_block: 32 | 16 | 8 | 4 (+100 = output-staged), 1 | 2 = the lane-per-block decoder, 0 = chosen on the device from
// the batch's compression ratio.  `counter` points at FOUR device words the launcher owns (block counter, pick, two more counters).
int         decode_lanes_for_ratio(double ratio);
cudaError_t launch_decode(const BatchArgs& a, bool known_len, int lanes_per_block, uint32_t* counter,
                          const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
cudaError_t launch_encode_fast(const BatchArgs& a, uint32_t* counter, int warps_per_sm, const int* tune4 /* prefetch, lane_copy_max, probe_max, wide_min */, int variant,
                               const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
size_t      hc_scratch_bytes(int concurrency);
cudaError_t launch_encode_hc(const BatchArgs& a, void* scratch, int concurrency, uint32_t* counter,
                             const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
// blocks <= 64 KiB: one warp per block on a static index, followed by the thread-per-block kernel over the blocks it handed back
// (variant 1: the block staged in shared memory, <= 3 warps per SM; 2: nothing in shared memory, <= 32 warps per SM)
size_t      hcw_scratch_bytes(int32_t n_blocks, int variant, int warps_per_sm, const DeviceInfo& dev);
cudaError_t launch_encode_hcw(const BatchArgs& a, void* scratch, int variant, int warps_per_sm, uint32_t* counter,
                              const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
// kernel chosen per batch: small batches -> the shared-memory warp kernel; large ones -> a sample of the batch decides on
// the device between the thread kernel and the warp kernel (`counter` = four words)
size_t      hc_auto_scratch_bytes(int32_t n_blocks, int concurrency, const DeviceInfo& dev);
cudaError_t launch_encode_hc_auto(const BatchArgs& a, void* scratch, int concurrency, uint32_t* counter,
                                  const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
cudaError_t launch_compact(const uint8_t* slots, const int64_t* slot_off, const int32_t* len, uint8_t* packed,
                           int64_t* out_off, int32_t n_blocks, void* scan_tmp, size_t scan_tmp_bytes,
                           const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);
size_t      compact_tmp_bytes(int32_t n_blocks);
// scatter copy (gather_blocks): len[i] bytes from src + src_off[i] to dst + dst_off[i], one warp per entry (len <= 0: none)
cudaError_t launch_scatter(const uint8_t* src, const int64_t* src_off, const int32_t* len, uint8_t* dst, const int64_t* dst_off,
                           int32_t n, cudaStream_t stream, int64_t* launches);
cudaError_t launch_synth(uint8_t* dst, int64_t n_blocks, int32_t block_size, int cls, uint64_t seed, int64_t first_block,
                         const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);

// LZ4Stream framing on device memory (stream.cu).  Encode, per group of m chunks of block_size bytes (rem = input bytes
// from the group's start): layout fills off[i] = i * block_size and len[i] (the chunk length, also its slot capacity);
// frame_sizes writes sizes[2i] = header bytes, sizes[2i+1] = payload bytes; frame_write writes chunk i's header at
// dst + pos[2i] and its payload at dst + pos[2i+1] (pos = exclusive scan of sizes).
cudaError_t launch_stream_layout(int64_t* off, int32_t* len, int32_t m, int32_t block_size, int64_t rem,
                                 cudaStream_t stream, int64_t* launches);
cudaError_t launch_stream_frame_sizes(const int32_t* len, const int32_t* out_len, int32_t m, int hc, int32_t* sizes,
                                      cudaStream_t stream, int64_t* launches);
cudaError_t launch_stream_frame_write(const uint8_t* src, const int64_t* off, const int32_t* len, const uint8_t* slots,
                                      const int32_t* out_len, const int64_t* pos, int32_t m, int hc, uint8_t* dst,
                                      cudaStream_t stream, int64_t* launches);
// Decode: one thread walks the chunk headers of src[0, n) and fills at most `cap` entries of each table (stored chunks:
// payload offset, output offset, length; compressed chunks: payload offset, output offset, compressed length, raw
// length, out_len = -1).  Chunks of 0 raw bytes are skipped.  *res gets the status (0 or LZ4B200_E_FORMAT), the total
// raw size and the full counts, whatever cap was: a count above cap means "grow the table and walk again".
struct StreamTable { int64_t *st_src, *st_dst, *cp_src, *cp_dst; int32_t *st_len, *cp_len, *cp_raw, *cp_out; };
struct StreamWalk { int64_t status, total, n_stored, n_comp; int32_t bad; };
size_t      stream_table_bytes(int64_t cap);
StreamTable stream_table_at(void* p, int64_t cap);
cudaError_t launch_stream_walk(const uint8_t* src, int64_t n, int64_t cap, const StreamTable& t, StreamWalk* res,
                               cudaStream_t stream, int64_t* launches);
// *bad |= 1 if out_len[i] != want[i] for any i < m
cudaError_t launch_stream_verdict(const int32_t* out_len, const int32_t* want, int32_t m, int32_t* bad,
                                  const DeviceInfo& dev, cudaStream_t stream, int64_t* launches);

}  // namespace lz4b200
