// util.cu -- compaction of encoder slots and the synthetic workload generator.
#include "kernels.h"
#include "simt.cuh"
#include "lz4_copy.cuh"

namespace lz4b200 {

// ---------------------------------------------------------------------------------------------------------------------
// Compaction (the batched form of LZ4Codec.Encode's trim copy, src/LZ4/LZ4Codec.cs:357-364, and of the LZ4Stream chunk
// writer's payload write, src/LZ4/LZ4Stream.cs:262-266): exclusive scan of the lengths, then one warp per block moves
// len[i] bytes from its slot to packed + out_off[i] with 128-bit accesses.
// The scan is three small kernels (per-tile sums, scan of the tile sums by one CTA, per-tile rescan + offset).
// ---------------------------------------------------------------------------------------------------------------------
constexpr int SCAN_TILE = 1024;      // elements per CTA (256 threads x 4)

__device__ __forceinline__ int64_t warp_incl_scan(int64_t v, int lane)
{
    for (int d = 1; d < 32; d <<= 1) {
        int64_t t = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// block-wide inclusive scan of one int64 per thread (256 threads); returns inclusive value, *total = sum over the CTA
__device__ int64_t block_incl_scan(int64_t v, int64_t* total)
{
    __shared__ int64_t wsum[8];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int64_t inc = warp_incl_scan(v, lane);
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    int64_t base = 0, tot = 0;
    for (int i = 0; i < 8; i++) { if (i < w) base += wsum[i]; tot += wsum[i]; }
    __syncthreads();
    *total = tot;
    return inc + base;
}

__global__ void __launch_bounds__(256) scan_tile_sums(const int32_t* len, int32_t n, int64_t* tile_sum)
{
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    int64_t s = 0;
    for (int k = 0; k < 4; k++) { int i = base + k; if (i < n) { int32_t l = len[i]; s += l > 0 ? l : 0; } }
    int64_t tot; block_incl_scan(s, &tot);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(256) scan_tile_offsets(int64_t* tile_sum, int32_t ntiles)
{
    // exclusive scan of tile sums in place, single CTA, chunks of 256 with a running carry
    __shared__ int64_t carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int c = 0; c < ntiles; c += 256) {
        int i = c + threadIdx.x;
        int64_t v = i < ntiles ? tile_sum[i] : 0, tot;
        int64_t inc = block_incl_scan(v, &tot);
        int64_t carry = carry_s;
        if (i < ntiles) tile_sum[i] = carry + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) scan_finish(const int32_t* len, int32_t n, const int64_t* tile_off, int64_t* out_off)
{
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * 4;
    int64_t l[4], s = 0;
    for (int k = 0; k < 4; k++) { int i = base + k; int32_t v = i < n ? len[i] : 0; l[k] = v > 0 ? v : 0; s += l[k]; }
    int64_t tot; int64_t inc = block_incl_scan(s, &tot);
    int64_t run = tile_off[blockIdx.x] + inc - s;
    for (int k = 0; k < 4; k++) { int i = base + k; if (i < n) out_off[i] = run; run += l[k]; }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 255) out_off[n] = tile_off[blockIdx.x] + tot;
}

// one warp per block: byte-exact move of len bytes, 16-byte vectors where src/dst alignment allows
__global__ void __launch_bounds__(256) gather_blocks(const uint8_t* slots, const int64_t* slot_off, const int32_t* len,
                                                     uint8_t* packed, const int64_t* out_off, int32_t n)
{
    const int lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= n) return;
    const int32_t l = len[w];
    if (l <= 0) return;
    const uint8_t* s = slots + slot_off[w];
    uint8_t* d = packed + out_off[w];
    int head = (int)((16 - ((uintptr_t)d & 15)) & 15); if (head > l) head = l;
    for (int i = lane; i < head; i += 32) d[i] = s[i];
    const int nvec = (l - head) >> 4;
    const uint32_t r = (uint32_t)((uintptr_t)(s + head) & 15);
    const uint8_t* sa = s + head - r;
    for (int v = lane; v < nvec; v += 32) {
        uint4 lo = __ldg((const uint4*)(sa + 16 * (size_t)v)), o = lo;
        if (r) {
            uint4 hi = __ldg((const uint4*)(sa + 16 * (size_t)v + 16));
            o = shift16(lo, hi, r);
        }
        *(uint4*)(d + head + 16 * (size_t)v) = o;
    }
    for (int i = head + (nvec << 4) + lane; i < l; i += 32) d[i] = s[i];
}

size_t compact_tmp_bytes(int32_t n_blocks)
{
    return sizeof(int64_t) * (size_t)((n_blocks + SCAN_TILE - 1) / SCAN_TILE + 1);
}

cudaError_t launch_compact(const uint8_t* slots, const int64_t* slot_off, const int32_t* len, uint8_t* packed,
                           int64_t* out_off, int32_t n, void* tmp, size_t tmp_bytes,
                           const DeviceInfo&, cudaStream_t stream, int64_t* launches)
{
    if (n <= 0) return cudaSuccess;
    if (tmp_bytes < compact_tmp_bytes(n)) return cudaErrorInvalidValue;
    const int ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    int64_t* tile = (int64_t*)tmp;
    scan_tile_sums<<<ntiles, 256, 0, stream>>>(len, n, tile);
    scan_tile_offsets<<<1, 256, 0, stream>>>(tile, ntiles);
    scan_finish<<<ntiles, 256, 0, stream>>>(len, n, tile, out_off);
    if (packed) gather_blocks<<<(n + 7) / 8, 256, 0, stream>>>(slots, slot_off, len, packed, out_off, n);
    if (launches) *launches += packed ? 4 : 3;
    return cudaGetLastError();
}

cudaError_t launch_scatter(const uint8_t* src, const int64_t* src_off, const int32_t* len, uint8_t* dst, const int64_t* dst_off,
                           int32_t n, cudaStream_t stream, int64_t* launches)
{
    if (n <= 0) return cudaSuccess;
    gather_blocks<<<(n + 7) / 8, 256, 0, stream>>>(src, src_off, len, dst, dst_off, n);
    if (launches) ++*launches;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// Synthetic entropy classes -- the CUDA twin of lz4net_b200/synth.py (same formulas, same bytes).
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
constexpr uint64_t GOLD = 0x9E3779B97F4A7C15ull;

// classes E0 / E50 / E100: every 8-byte word is a closed formula -> one thread per word, fully coalesced
__global__ void __launch_bounds__(256) synth_words(uint8_t* dst, int64_t n_blocks, int32_t block_size, int cls,
                                                   uint64_t seed, int64_t first_block)
{
    const int64_t words_per_block = (block_size + 7) / 8;
    const int64_t total = n_blocks * words_per_block;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = t / words_per_block, k = t - b * words_per_block;
        uint64_t w = 0;
        if (cls != 2) {
            const uint64_t sb = mix64((seed ^ (uint64_t)(first_block + b)) + GOLD);
            // E0: word k is stream word k.  E50: 64-byte groups of 4 stream words written twice.
            const uint64_t idx = cls == 0 ? (uint64_t)k : (uint64_t)((k >> 3) * 4 + (k & 3));
            w = mix64(sb + (idx + 1) * GOLD);
        }
        uint8_t* p = dst + b * (int64_t)block_size + k * 8;
        const int rem = block_size - (int)(k * 8);
        if (rem >= 8 && (((uintptr_t)p) & 7) == 0) *(uint64_t*)p = w;
        else for (int i = 0; i < 8 && i < rem; i++) p[i] = (uint8_t)(w >> (8 * i));
    }
}

// class ETEXT: dictionary words of different lengths laid out sequentially -> one thread walks one block (setup only)
__constant__ char ETEXT_DICT[8][10] = {"lz", "net", "code", "block", "stream", "encoder", "compress", "blackwell"};
__constant__ int  ETEXT_LEN[8] = {2, 3, 4, 5, 6, 7, 8, 9};

__global__ void __launch_bounds__(64) synth_text(uint8_t* dst, int64_t n_blocks, int32_t block_size, uint64_t seed, int64_t first_block)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const uint64_t sb = mix64((seed ^ (uint64_t)(first_block + b)) + GOLD);
    uint8_t* p = dst + b * (int64_t)block_size;
    int pos = 0;
    for (uint64_t k = 1; pos < block_size; k++) {
        const int w = (int)(mix64(sb + k * GOLD) >> 61);
        const int l = ETEXT_LEN[w];
        for (int i = 0; i <= l && pos < block_size; i++) p[pos++] = i < l ? (uint8_t)ETEXT_DICT[w][i] : (uint8_t)' ';
    }
}

cudaError_t launch_synth(uint8_t* dst, int64_t n_blocks, int32_t block_size, int cls, uint64_t seed, int64_t first_block,
                         const DeviceInfo& dev, cudaStream_t stream, int64_t* launches)
{
    if (n_blocks <= 0 || block_size <= 0) return cudaSuccess;
    if (cls < 0 || cls > 3) return cudaErrorInvalidValue;
    if (cls == 3) synth_text<<<(unsigned)((n_blocks + 63) / 64), 64, 0, stream>>>(dst, n_blocks, block_size, seed, first_block);
    else synth_words<<<dev.num_sms * 8, 256, 0, stream>>>(dst, n_blocks, block_size, cls, seed, first_block);
    if (launches) ++*launches;
    return cudaGetLastError();
}

}  // namespace lz4b200
