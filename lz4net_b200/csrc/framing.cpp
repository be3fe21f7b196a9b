// framing.cpp -- host-side framing on top of the batch ABI: the LZ4Stream chunk format and the Wrap/Unwrap packet.
//
// LZ4Stream (src/LZ4/LZ4Stream.cs) is the reference's block dispatcher: it buffers one block, calls
// LZ4Codec.Encode/EncodeHC with capacity == block length, and writes  varint(flags) varint(rawLen) [varint(compLen)]
// payload  per chunk (FlushCurrentChunk :239-269; reader AcquireNextChunk :274-312; varints :167-187,225-236).
// Here the same byte stream is produced / consumed with ONE batched GPU call for all chunks of a buffer.
// Pure host code: no kernels, no codec arithmetic -- that all lives behind lz4b200_{encode,decode}_batch.  The chunk
// header codec is lz4_stream.cuh, which the device framing of stream.cu / capi.cu uses as well.
#include "../../include/lz4b200.h"
#include "lz4_stream.cuh"

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

using namespace lz4b200::lz4s;

// walk the chunk headers of a whole stream; returns total raw size or a negative status
int64_t walk(const uint8_t* s, int64_t n, std::vector<Chunk>* out)
{
    int64_t pos = 0, total = 0;
    for (;;) {
        Chunk c;
        const int r = walk_step(s, n, &pos, &c);
        if (r == 0) return total;
        if (r < 0) return r;
        if (out) out->push_back(c);
        total += c.raw;
    }
}

}  // namespace

extern "C" {

int64_t lz4b200_stream_bound(int64_t n, int32_t block_size)
{
    if (n < 0 || block_size < 1) return LZ4B200_E_ARG;
    const int64_t chunks = (n + block_size - 1) / block_size;
    return n + chunks * (1 + 2 * varint_size((uint64_t)block_size));
}

int64_t lz4b200_stream_encode(lz4b200_ctx* ctx, const void* src, int64_t n, int32_t block_size, int hc, void* dst, int64_t dst_cap)
{
    if (!ctx || n < 0 || block_size < 1 || (n > 0 && (!src || !dst))) return LZ4B200_E_ARG;
    if (dst_cap < lz4b200_stream_bound(n, block_size)) return LZ4B200_E_ARG;
    const uint8_t* s = (const uint8_t*)src; uint8_t* d = (uint8_t*)dst;
    const int64_t chunks = (n + block_size - 1) / block_size;
    // groups of chunks bound the temporary slot buffer (capacity == raw length per chunk, LZ4Stream.cs:243-246)
    const int64_t group = std::max<int64_t>(1, (int64_t)(256u << 20) / block_size);
    std::vector<uint8_t> slots;
    std::vector<int64_t> so, dof; std::vector<int32_t> sl, dc, out;
    int64_t w = 0;
    for (int64_t c0 = 0; c0 < chunks; c0 += group) {
        const int64_t c1 = std::min(chunks, c0 + group), m = c1 - c0;
        so.resize(m); dof.resize(m); sl.resize(m); dc.resize(m); out.assign(m, 0);
        const int64_t base = c0 * block_size;
        for (int64_t i = 0; i < m; i++) {
            const int64_t off = (c0 + i) * block_size;
            so[i] = off; dof[i] = off - base;
            sl[i] = dc[i] = (int32_t)std::min<int64_t>(block_size, n - off);
        }
        slots.resize((size_t)(dof[m - 1] + dc[m - 1]));
        int rc = lz4b200_encode_batch(ctx, s, so.data(), sl.data(), slots.data(), dof.data(), dc.data(), out.data(),
                                      (int32_t)m, hc ? LZ4B200_MODE_HC : LZ4B200_MODE_FAST, LZ4B200_MEM_HOST, nullptr);
        if (rc != LZ4B200_OK) return rc;
        for (int64_t i = 0; i < m; i++) {
            const int32_t raw = sl[i], clen = out[i];
            const bool comp = chunk_compressed(raw, clen);                   // LZ4Stream.cs:248-255
            uint8_t* p = d + w;
            p = put_varint(p, chunk_flags(comp, hc != 0));
            p = put_varint(p, (uint64_t)raw);
            if (comp) p = put_varint(p, (uint64_t)clen);
            std::memcpy(p, comp ? slots.data() + dof[i] : s + so[i], (size_t)(comp ? clen : raw));
            w = (p - d) + (comp ? clen : raw);
        }
    }
    return w;
}

int64_t lz4b200_stream_decoded_size(const void* src, int64_t n)
{
    if (n < 0 || (n > 0 && !src)) return LZ4B200_E_ARG;
    return walk((const uint8_t*)src, n, nullptr);
}

int64_t lz4b200_stream_decode(lz4b200_ctx* ctx, const void* src, int64_t n, void* dst, int64_t dst_cap)
{
    if (!ctx || n < 0 || (n > 0 && !src)) return LZ4B200_E_ARG;
    std::vector<Chunk> chunks;
    const int64_t total = walk((const uint8_t*)src, n, &chunks);
    if (total < 0) return total;
    if (total > dst_cap || (total > 0 && !dst)) return LZ4B200_E_ARG;
    const uint8_t* s = (const uint8_t*)src; uint8_t* d = (uint8_t*)dst;
    std::vector<int64_t> so, dof; std::vector<int32_t> sl, dc, out;
    int64_t pos = 0;
    for (const Chunk& c : chunks) {
        if (!c.compressed) std::memcpy(d + pos, s + c.payload, (size_t)c.raw);           // stored chunk (:295-299)
        else if (c.raw > 0) { so.push_back(c.payload); sl.push_back(c.stored); dof.push_back(pos); dc.push_back(c.raw); }
        pos += c.raw;
    }
    if (!so.empty()) {
        out.assign(so.size(), -1);
        int rc = lz4b200_decode_batch(ctx, s, so.data(), sl.data(), d, dof.data(), dc.data(), out.data(),
                                      (int32_t)so.size(), 1, LZ4B200_MEM_HOST, nullptr);
        if (rc != LZ4B200_OK) return rc;
        // LZ4Codec.Decode(..., knownOutputLength: true) throws unless exactly compLen bytes were consumed
        // (src/LZ4ps/LZ4Codec.Safe.cs:539-542)
        for (size_t i = 0; i < so.size(); i++) if (out[i] != sl[i]) return LZ4B200_E_FORMAT;
    }
    return total;
}

int lz4b200_wrap(lz4b200_ctx* ctx, const void* src, int32_t n, int hc, void* dst, int32_t dst_cap)
{
    // src/LZ4/LZ4Codec.cs:510-543
    if (!ctx || n < 0 || !dst || (n > 0 && !src)) return LZ4B200_E_ARG;
    if ((int64_t)dst_cap < (int64_t)n + 8) return LZ4B200_E_ARG;
    uint8_t* d = (uint8_t*)dst;
    auto poke4 = [](uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); };
    if (n == 0) { std::memset(d, 0, 8); return 8; }
    int64_t so = 0, dof = 0; int32_t sl = n, dc = n, out = 0;
    int rc = lz4b200_encode_batch(ctx, src, &so, &sl, d + 8, &dof, &dc, &out, 1, hc ? LZ4B200_MODE_HC : LZ4B200_MODE_FAST,
                                  LZ4B200_MEM_HOST, nullptr);
    if (rc != LZ4B200_OK) return rc;
    poke4(d, (uint32_t)n);
    if (out >= n || out <= 0) { poke4(d + 4, (uint32_t)n); std::memcpy(d + 8, src, (size_t)n); return n + 8; }
    poke4(d + 4, (uint32_t)out);
    return out + 8;
}

int lz4b200_unwrap_size(const void* src, int32_t n)
{
    if (!src || n < 8) return LZ4B200_E_FORMAT;                                          // :577-578
    const uint8_t* s = (const uint8_t*)src;
    const int32_t raw = (int32_t)(s[0] | s[1] << 8 | s[2] << 16 | (uint32_t)s[3] << 24);
    const int32_t stored = (int32_t)(s[4] | s[5] << 8 | s[6] << 16 | (uint32_t)s[7] << 24);
    if (stored > n - 8 || stored < 0 || raw < 0) return LZ4B200_E_FORMAT;                // :582-583
    return stored >= raw ? stored : raw;                                                 // :587-596
}

int lz4b200_unwrap(lz4b200_ctx* ctx, const void* src, int32_t n, void* dst, int32_t dst_cap)
{
    const int size = lz4b200_unwrap_size(src, n);
    if (size < 0) return size;
    if (!ctx || size > dst_cap || (size > 0 && !dst)) return LZ4B200_E_ARG;
    const uint8_t* s = (const uint8_t*)src;
    const int32_t raw = (int32_t)(s[0] | s[1] << 8 | s[2] << 16 | (uint32_t)s[3] << 24);
    const int32_t stored = (int32_t)(s[4] | s[5] << 8 | s[6] << 16 | (uint32_t)s[7] << 24);
    if (stored >= raw) { std::memcpy(dst, s + 8, (size_t)stored); return stored; }
    int64_t so = 8, dof = 0; int32_t sl = stored, dc = raw, out = -1;
    int rc = lz4b200_decode_batch(ctx, s, &so, &sl, dst, &dof, &dc, &out, 1, 1, LZ4B200_MEM_HOST, nullptr);
    if (rc != LZ4B200_OK) return rc;
    return out == stored ? raw : LZ4B200_E_FORMAT;
}

// ---- batched Wrap / Unwrap (SURVEY.md 8f rank 2): n packets, ONE encode / decode batch ---------------------------------
// Packet i of the batch is exactly what lz4b200_wrap / LZ4Codec.Wrap (src/LZ4/LZ4Codec.cs:510-543) produces for input i:
// u32le rawLen, u32le storedLen, payload (the compressed bytes, or the input itself when compression does not shrink it).
// Inputs: src + src_off[i], src_len[i] bytes.  Packets: dst + dst_off[i], capacity dst_cap[i] >= src_len[i] + 8.
// out_len[i] = packet size (or a negative status for that packet).
int lz4b200_wrap_batch(lz4b200_ctx* ctx, const void* src, const int64_t* src_off, const int32_t* src_len, int high_compression,
                       void* dst, const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n)
{
    if (!ctx || n < 0) return LZ4B200_E_ARG;
    if (n == 0) return LZ4B200_OK;
    if (!src || !dst || !src_off || !src_len || !dst_off || !dst_cap || !out_len) return LZ4B200_E_ARG;
    const uint8_t* s = (const uint8_t*)src; uint8_t* d = (uint8_t*)dst;
    auto poke4 = [](uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); };
    std::vector<int64_t> po(n); std::vector<int32_t> pc(n), res(n, 0);
    for (int32_t i = 0; i < n; i++) {
        if (src_len[i] < 0 || (int64_t)dst_cap[i] < (int64_t)src_len[i] + 8) return LZ4B200_E_ARG;
        po[i] = dst_off[i] + 8; pc[i] = src_len[i];                  // payload capacity = the input length (:518-523)
    }
    int rc = lz4b200_encode_batch(ctx, s, src_off, src_len, d, po.data(), pc.data(), res.data(), n,
                                  high_compression ? LZ4B200_MODE_HC : LZ4B200_MODE_FAST, LZ4B200_MEM_HOST, nullptr);
    if (rc != LZ4B200_OK) return rc;
    for (int32_t i = 0; i < n; i++) {
        uint8_t* p = d + dst_off[i]; const int32_t len = src_len[i];
        poke4(p, (uint32_t)len);
        if (len == 0) { poke4(p + 4, 0); out_len[i] = 8; continue; }
        if (res[i] >= len || res[i] <= 0) { poke4(p + 4, (uint32_t)len); std::memcpy(p + 8, s + src_off[i], (size_t)len); out_len[i] = len + 8; }
        else { poke4(p + 4, (uint32_t)res[i]); out_len[i] = res[i] + 8; }
    }
    return LZ4B200_OK;
}

// Mirror image (src/LZ4/LZ4Codec.cs:574-599).  Packets: src + src_off[i], src_len[i] bytes.  Outputs: dst + dst_off[i],
// capacity dst_cap[i] >= lz4b200_unwrap_size(packet i).  out_len[i] = bytes restored, or LZ4B200_E_FORMAT / E_ARG.
int lz4b200_unwrap_batch(lz4b200_ctx* ctx, const void* src, const int64_t* src_off, const int32_t* src_len,
                         void* dst, const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n)
{
    if (!ctx || n < 0) return LZ4B200_E_ARG;
    if (n == 0) return LZ4B200_OK;
    if (!src || !dst || !src_off || !src_len || !dst_off || !dst_cap || !out_len) return LZ4B200_E_ARG;
    const uint8_t* s = (const uint8_t*)src; uint8_t* d = (uint8_t*)dst;
    std::vector<int64_t> so, dof; std::vector<int32_t> sl, dc, res, idx;
    for (int32_t i = 0; i < n; i++) {
        const uint8_t* p = s + src_off[i];
        const int size = lz4b200_unwrap_size(p, src_len[i]);
        if (size < 0) { out_len[i] = size; continue; }
        if (size > dst_cap[i]) { out_len[i] = LZ4B200_E_ARG; continue; }
        const int32_t raw = (int32_t)(p[0] | p[1] << 8 | p[2] << 16 | (uint32_t)p[3] << 24);
        const int32_t stored = (int32_t)(p[4] | p[5] << 8 | p[6] << 16 | (uint32_t)p[7] << 24);
        if (stored >= raw) { std::memcpy(d + dst_off[i], p + 8, (size_t)stored); out_len[i] = stored; continue; }
        so.push_back(src_off[i] + 8); sl.push_back(stored); dof.push_back(dst_off[i]); dc.push_back(raw); idx.push_back(i);
    }
    if (!so.empty()) {
        res.assign(so.size(), -1);
        int rc = lz4b200_decode_batch(ctx, s, so.data(), sl.data(), d, dof.data(), dc.data(), res.data(), (int32_t)so.size(), 1,
                                      LZ4B200_MEM_HOST, nullptr);
        if (rc != LZ4B200_OK) return rc;
        for (size_t j = 0; j < so.size(); j++) out_len[idx[j]] = res[j] == sl[j] ? dc[j] : LZ4B200_E_FORMAT;
    }
    return LZ4B200_OK;
}

}  // extern "C"
