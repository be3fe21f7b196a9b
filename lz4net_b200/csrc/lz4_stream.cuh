// lz4_stream.cuh -- the LZ4Stream chunk header codec, shared by the host framing (framing.cpp) and the device framing
// kernels (stream.cu), so that the two parsers cannot drift apart.
//
// Chunk:  varint(flags) varint(rawLen) [varint(compLen)] payload  (src/LZ4/LZ4Stream.cs:167-187,225-236,239-312).
// Compiles under nvcc (host + device), under a plain C++ compiler and in the g++ emulator build.
#pragma once
#include <stdint.h>

#include "../../include/lz4b200.h"

#if defined(__CUDACC__)
#define LZ4S_HD __host__ __device__ __forceinline__
#else
#define LZ4S_HD inline
#endif

namespace lz4b200 {
namespace lz4s {

enum : uint64_t { FLAG_COMPRESSED = 1, FLAG_HC = 2 };          // ChunkFlags, LZ4Stream.cs:43-58

LZ4S_HD int varint_size(uint64_t v) { int n = 1; while (v >>= 7) n++; return n; }

LZ4S_HD uint8_t* put_varint(uint8_t* p, uint64_t v)            // LZ4Stream.cs:225-236
{
    for (;;) {
        uint8_t b = (uint8_t)(v & 0x7F);
        v >>= 7;
        *p++ = (uint8_t)(b | (v ? 0x80 : 0));
        if (!v) return p;
    }
}

// LZ4Stream.cs:167-187.  Returns 1 = value read, 0 = clean end of data before the first byte, -1 = truncated.
// Never reads s[i] for i >= n.
LZ4S_HD int get_varint(const uint8_t* s, int64_t n, int64_t* pos, uint64_t* out)
{
    uint64_t r = 0; int count = 0;
    for (;;) {
        if (*pos >= n) return count == 0 ? 0 : -1;
        uint8_t b = s[(*pos)++];
        r += (uint64_t)(b & 0x7F) << count;
        count += 7;
        if (!(b & 0x80) || count >= 64) break;
    }
    *out = r;
    return 1;
}

// The chunk writer's choice (LZ4Stream.cs:248-255): a chunk is stored raw unless the encoder made it smaller.
LZ4S_HD bool chunk_compressed(int32_t raw, int32_t clen) { return clen > 0 && clen < raw; }
LZ4S_HD uint64_t chunk_flags(bool comp, bool hc) { return (comp ? FLAG_COMPRESSED : 0) | (hc ? FLAG_HC : 0); }
LZ4S_HD int header_size(int32_t raw, int32_t clen, bool hc)
{
    const bool comp = chunk_compressed(raw, clen);
    return varint_size(chunk_flags(comp, hc)) + varint_size((uint64_t)raw) + (comp ? varint_size((uint64_t)clen) : 0);
}

struct Chunk { int64_t payload; int32_t raw; int32_t stored; bool compressed; };

// One step of the chunk reader (LZ4Stream.cs:274-312): parses the header at *pos and skips its payload.
// Returns 1 = a chunk (*c filled, *pos behind its payload), 0 = clean end of the stream, LZ4B200_E_FORMAT = malformed.
LZ4S_HD int walk_step(const uint8_t* s, int64_t n, int64_t* pos, Chunk* c)
{
    uint64_t flags, raw, clen;
    const int r = get_varint(s, n, pos, &flags);
    if (r == 0) return 0;                                                   // legitimate end (LZ4Stream.cs:281)
    if (r < 0) return LZ4B200_E_FORMAT;
    if (get_varint(s, n, pos, &raw) != 1) return LZ4B200_E_FORMAT;
    const bool comp = (flags & FLAG_COMPRESSED) != 0;
    clen = raw;
    if (comp && get_varint(s, n, pos, &clen) != 1) return LZ4B200_E_FORMAT;
    const int32_t rawi = (int32_t)raw, cleni = (int32_t)clen;              // the reference casts to int (:286-287)
    if (rawi < 0 || cleni < 0 || cleni > rawi) return LZ4B200_E_FORMAT;    // :288 corrupted
    if (*pos + cleni > n) return LZ4B200_E_FORMAT;                          // :293 short read
    if (comp && (flags >> 2) != 0) return LZ4B200_E_FORMAT;                // :301-303 multi-pass chunks unsupported
    c->payload = *pos; c->raw = rawi; c->stored = cleni; c->compressed = comp;
    *pos += cleni;
    return 1;
}

}  // namespace lz4s
}  // namespace lz4b200
