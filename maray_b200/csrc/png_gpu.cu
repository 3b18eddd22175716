// PNG encoder on the GPU (png_gpu.hpp, DESIGN.md 3.8).
//
// Pipeline on one stream of the first GPU:
//   png_filter_kernel    one block per row: the filter (None/Sub/Up/Average/Paeth) with the least sum of |signed byte|
//                        (libpng's heuristic), written to the scanline stream (hgt * (3w + 1) bytes);
//   png_deflate_kernel   one block per segment of S bytes (segment_bytes: a function of the stream length only):
//                        hash-table match finding in parallel over positions, a greedy parse by one warp, a dynamic
//                        Huffman block (15-bit lit/len and distance codes, 7-bit code-length code) or stored blocks
//                        when those are smaller, bits packed after a scan of the token lengths; Adler-32 sums;
//   png_layout_kernel    scan of the segment sizes, Adler-32 combine, signature, IHDR, IDAT framing, IEND;
//   png_gather_kernel    every segment's bytes to their place in the file;
//   png_crc_kernel       CRC-32 of pieces of every IDAT, then png_crc_finish_kernel combines them per chunk.
// The CPU twin (maray_cuda_png_encode_host) runs the same functions serially over a frame and writes the same bytes.
#include "png_gpu.hpp"

#include <cub/block/block_scan.cuh>

#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "../../include/maray_cuda.h"

#define HD __host__ __device__ __forceinline__

namespace maray {
namespace {

constexpr uint32_t kThreads = 512;        // threads of a deflate block = positions per match-finding round
constexpr uint32_t kHashBits = 13;
constexpr uint32_t kWindow = 32768;       // deflate's largest distance
constexpr uint32_t kMaxMatch = 258;
constexpr uint32_t kProbe = 16;           // match bytes compared per position; the parse extends longer matches
constexpr uint32_t kStoredMax = 65535;
constexpr uint64_t kIdatBytes = uint64_t(1) << 30;   // IDAT payload (PNG allows up to 2^31 - 1)
constexpr uint32_t kCrcPiece = 65536;     // bytes of an IDAT's CRC computed by one block
constexpr uint32_t kCrcThreads = 256;
constexpr uint32_t kHeaderBytes = 33;     // signature + IHDR

// ---- sizes ----------------------------------------------------------------------------------------------------------

// Segment size from the stream length alone, so the file does not depend on the GPU: about 320 segments per frame
// (two or more per SM of a B200 from 4K up), 4 KiB granules, 16 KiB .. 128 KiB.
HD uint64_t segment_bytes(uint64_t L) {
    uint64_t s = ((L + 319) / 320 + 4095) & ~uint64_t(4095);
    return s < 16384 ? 16384 : (s > 131072 ? 131072 : s);
}
HD uint64_t stored_size(uint64_t n) { return n + 5 * ((n + kStoredMax - 1) / kStoredMax); }
// A segment's output never exceeds its stored form: that bounds every slot in advance.
HD uint64_t slot_bytes(uint64_t S) { return (stored_size(S) + 7) & ~uint64_t(7); }
HD uint64_t file_offset(uint64_t z, uint64_t chunk) { return kHeaderBytes + (z / chunk) * 12 + 8 + z; }
HD uint64_t file_bytes(uint64_t zlen, uint64_t chunk) { return kHeaderBytes + 12 * ((zlen + chunk - 1) / chunk) + zlen + 12; }

HD uint32_t msb(uint32_t v) {
#ifdef __CUDA_ARCH__
    return 31 - __clz(v);
#else
    return 31 - __builtin_clz(v);
#endif
}

// ---- filters --------------------------------------------------------------------------------------------------------

HD int paeth(int a, int b, int c) {
    int p = a + b - c, pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}
HD uint8_t filter_byte(uint32_t f, int x, int a, int b, int c) {
    switch (f) {
    case 1: return uint8_t(x - a);
    case 2: return uint8_t(x - b);
    case 3: return uint8_t(x - ((a + b) >> 1));
    case 4: return uint8_t(x - paeth(a, b, c));
    default: return uint8_t(x);
    }
}
// a, b, c of byte i of a row (left, up, up-left); prev is NULL on the first row
HD void neighbours(const uint8_t* row, const uint8_t* prev, uint64_t i, int* a, int* b, int* c) {
    *a = i >= 3 ? row[i - 3] : 0;
    *b = prev ? prev[i] : 0;
    *c = (prev && i >= 3) ? prev[i - 3] : 0;
}
HD uint32_t byte_cost(uint8_t v) { return v < 128 ? v : 256u - v; }
HD void add_costs(const uint8_t* row, const uint8_t* prev, uint64_t i, uint64_t cost[5]) {
    int a, b, c;
    neighbours(row, prev, i, &a, &b, &c);
    for (uint32_t f = 0; f < 5; f++) cost[f] += byte_cost(filter_byte(f, row[i], a, b, c));
}
HD uint32_t best_filter(const uint64_t cost[5]) {
    uint32_t f = 0;
    for (uint32_t k = 1; k < 5; k++) if (cost[k] < cost[f]) f = k;
    return f;
}

// ---- LZ77 -----------------------------------------------------------------------------------------------------------

HD uint32_t hash3(const uint8_t* p) {
    return ((uint32_t(p[0]) | uint32_t(p[1]) << 8 | uint32_t(p[2]) << 16) * 2654435761u) >> (32 - kHashBits);
}
HD uint32_t match_len(const uint8_t* s, uint64_t i, uint64_t j, uint32_t maxlen) {
    uint32_t n = 0;
    while (n < maxlen && s[i + n] == s[j + n]) n++;
    return n;
}
// The hash table holds positions relative to the window base of the segment, +1 (0 = empty).
HD int64_t window_base(uint64_t s0) { return int64_t(s0) - int64_t(kWindow); }
// The match found for position p: the longest (up to kProbe bytes) of the previous byte, the previous pixel and the
// hash table's candidate, the nearer on ties (runs then code as distance 1 or 3, without extra bits).  Returns the
// length (0 = none) and sets *dist.
HD uint32_t probe(const uint8_t* s, uint64_t p, uint64_t s1, int64_t base, int32_t cand, uint32_t* dist) {
    *dist = 0;
    const uint32_t maxlen = uint32_t(s1 - p < kMaxMatch ? s1 - p : kMaxMatch);
    if (maxlen < 3) return 0;
    const uint32_t cap = maxlen < kProbe ? maxlen : kProbe;
    uint32_t best = 0;
    for (int k = 0; k < 3; k++) {
        uint64_t d = k == 0 ? 1 : (k == 1 ? 3 : (cand ? p - uint64_t(base + cand - 1) : 0));
        if (d == 0 || d > p || d > kWindow) continue;
        const uint32_t l = match_len(s, p, p - d, cap);
        if (l > best) { best = l; *dist = uint32_t(d); }
    }
    if (best < 3) { *dist = 0; return 0; }
    return best;
}

// tokens: a literal is its byte; a match is bit 31 | (distance - 1) << 8 | (length - 3)
HD uint32_t tok_match(uint32_t len, uint32_t dist) { return 0x80000000u | ((dist - 1) << 8) | (len - 3); }
HD uint32_t len_sym(uint32_t len, uint32_t* nx, uint32_t* x) {
    if (len == 258) { *nx = 0; *x = 0; return 285; }
    const uint32_t l = len - 3;
    if (l < 8) { *nx = 0; *x = 0; return 257 + l; }
    const uint32_t nb = msb(l) - 2;
    *nx = nb; *x = l & ((1u << nb) - 1);
    return 257 + 4 * nb + (l >> nb);
}
HD uint32_t dist_sym(uint32_t dist, uint32_t* nx, uint32_t* x) {
    const uint32_t d = dist - 1;
    if (d < 4) { *nx = 0; *x = 0; return d; }
    const uint32_t m = msb(d), nb = m - 1;
    *nx = nb; *x = d & ((1u << nb) - 1);
    return 2 * m + ((d >> nb) & 1);
}
HD uint32_t len_extra(uint32_t sym) { return (sym >= 265 && sym <= 284) ? (sym - 261) / 4 : 0; }
HD uint32_t dist_extra(uint32_t sym) { return sym >= 4 ? sym / 2 - 1 : 0; }

// ---- Huffman codes --------------------------------------------------------------------------------------------------

// Position of symbol i among the used symbols ordered by (frequency, symbol).
HD uint32_t sym_rank(const uint32_t* f, uint32_t n, uint32_t i) {
    uint32_t r = 0;
    for (uint32_t j = 0; j < n; j++) r += (f[j] && (f[j] < f[i] || (f[j] == f[i] && j < i))) ? 1u : 0u;
    return r;
}
// Moffat & Katajainen, in place: A[0..m) ascending weights -> A[k] = code length of element k (m >= 2).
HD void moffat(uint32_t* A, int n) {
    int root, leaf, next, avbl, used, dpth;
    A[0] += A[1]; root = 0; leaf = 2;
    for (next = 1; next < n - 1; next++) {
        if (leaf >= n || A[root] < A[leaf]) { A[next] = A[root]; A[root++] = uint32_t(next); }
        else A[next] = A[leaf++];
        if (leaf >= n || (root < next && A[root] < A[leaf])) { A[next] += A[root]; A[root++] = uint32_t(next); }
        else A[next] += A[leaf++];
    }
    A[n - 2] = 0;
    for (next = n - 3; next >= 0; next--) A[next] = A[A[next]] + 1;
    avbl = 1; used = dpth = 0; root = n - 2; next = n - 1;
    while (avbl > 0) {
        while (root >= 0 && int(A[root]) == dpth) { used++; root--; }
        while (avbl > used) { A[next--] = uint32_t(dpth); avbl--; }
        avbl = 2 * used; dpth++; used = 0;
    }
}
// Lengths of at most `limit` bits for the m used symbols sorted[0..m), A[k] = frequency of sorted[k] (ascending).
// Lengths above the limit are folded into it and the Kraft sum restored by lengthening the deepest shorter codes
// (miniz's method); the longest codes then go to the least frequent symbols.  One used symbol gets length 1.
HD void lengths_from_sorted(const uint16_t* sorted, uint32_t* A, uint32_t m, uint32_t limit, uint8_t* lens) {
    if (m == 0) return;
    if (m == 1) { lens[sorted[0]] = 1; return; }
    moffat(A, int(m));
    uint32_t count[16] = {0};
    for (uint32_t k = 0; k < m; k++) count[A[k] < limit ? A[k] : limit]++;
    uint32_t total = 0;
    for (uint32_t i = 1; i <= limit; i++) total += count[i] << (limit - i);
    while (total != (1u << limit)) {
        count[limit]--;
        for (uint32_t i = limit - 1; i > 0; i--)
            if (count[i]) { count[i]--; count[i + 1] += 2; break; }
        total--;
    }
    uint32_t k = 0;
    for (uint32_t len = limit; len >= 1; len--)
        for (uint32_t c = count[len]; c > 0; c--) lens[sorted[k++]] = uint8_t(len);
}
HD void build_lengths(const uint32_t* f, uint32_t n, uint32_t limit, uint8_t* lens, uint16_t* sorted, uint32_t* A) {
    uint32_t m = 0;
    for (uint32_t i = 0; i < n; i++) {
        lens[i] = 0;
        if (f[i]) { sorted[sym_rank(f, n, i)] = uint16_t(i); m++; }
    }
    for (uint32_t k = 0; k < m; k++) A[k] = f[sorted[k]];
    lengths_from_sorted(sorted, A, m, limit, lens);
}
// Canonical codes (deflate 3.2.2), bit-reversed for LSB-first packing.
HD void canonical(const uint8_t* lens, uint32_t n, uint16_t* codes) {
    uint32_t count[16] = {0}, next[16] = {0};
    for (uint32_t i = 0; i < n; i++) if (lens[i]) count[lens[i]]++;
    uint32_t code = 0;
    for (uint32_t b = 1; b < 16; b++) { code = (code + count[b - 1]) << 1; next[b] = code; }
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t l = lens[i];
        if (!l) { codes[i] = 0; continue; }
        uint32_t c = next[l]++, r = 0;
        for (uint32_t k = 0; k < l; k++) { r = (r << 1) | (c & 1); c >>= 1; }
        codes[i] = uint16_t(r);
    }
}

struct BlockCode {
    uint32_t lit_freq[286], dist_freq[30], cl_freq[19];
    uint8_t lit_len[286], dist_len[30], cl_len[19];
    uint16_t lit_code[286], dist_code[30], cl_code[19];
    uint8_t rle_sym[316], rle_extra[316];
    uint32_t n_rle, hlit, hdist, hclen;
    uint64_t header_bits, data_bits;
};

HD uint32_t cl_order(uint32_t i) {
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    return order[i];
}
HD uint32_t cl_extra(uint32_t sym) { return sym == 16 ? 2 : (sym == 17 ? 3 : (sym == 18 ? 7 : 0)); }

// Everything after the lit/len and distance lengths: codes, the code-length RLE (16/17/18) and its 7-bit code,
// HLIT/HDIST/HCLEN, and the bit counts of the block header and of the data.
HD void finish_code(BlockCode& c, uint16_t* sorted, uint32_t* A) {
    bool any_dist = false;
    for (uint32_t i = 0; i < 30; i++) any_dist |= c.dist_len[i] != 0;
    if (!any_dist) c.dist_len[0] = 1;   // a block without matches still declares one distance code
    canonical(c.lit_len, 286, c.lit_code);
    canonical(c.dist_len, 30, c.dist_code);
    c.hlit = 286;
    while (c.hlit > 257 && !c.lit_len[c.hlit - 1]) c.hlit--;
    c.hdist = 30;
    while (c.hdist > 1 && !c.dist_len[c.hdist - 1]) c.hdist--;
    const uint32_t n = c.hlit + c.hdist;
    auto len_at = [&](uint32_t i) -> uint32_t { return i < c.hlit ? c.lit_len[i] : c.dist_len[i - c.hlit]; };
    c.n_rle = 0;
    for (uint32_t i = 0; i < 19; i++) c.cl_freq[i] = 0;
    auto emit = [&](uint32_t sym, uint32_t extra) {
        c.rle_sym[c.n_rle] = uint8_t(sym); c.rle_extra[c.n_rle] = uint8_t(extra); c.n_rle++; c.cl_freq[sym]++;
    };
    for (uint32_t i = 0; i < n;) {
        const uint32_t cur = len_at(i);
        uint32_t run = 1;
        while (i + run < n && len_at(i + run) == cur) run++;
        i += run;
        if (cur == 0) {
            while (run >= 11) { const uint32_t r = run < 138 ? run : 138; emit(18, r - 11); run -= r; }
            if (run >= 3) { emit(17, run - 3); run = 0; }
            while (run) { emit(0, 0); run--; }
        } else {
            emit(cur, 0); run--;
            while (run >= 3) { const uint32_t r = run < 6 ? run : 6; emit(16, r - 3); run -= r; }
            while (run) { emit(cur, 0); run--; }
        }
    }
    uint32_t used = 0;
    for (uint32_t i = 0; i < 19; i++) used += c.cl_freq[i] ? 1u : 0u;
    uint32_t cl_f[19];
    for (uint32_t i = 0; i < 19; i++) cl_f[i] = c.cl_freq[i];
    if (used == 1)   // the code-length code must be complete: give the single symbol a partner of length 1
        for (uint32_t i = 0; i < 19; i++) if (!cl_f[i]) { cl_f[i] = 1; break; }
    build_lengths(cl_f, 19, 7, c.cl_len, sorted, A);
    canonical(c.cl_len, 19, c.cl_code);
    c.hclen = 19;
    while (c.hclen > 4 && !c.cl_len[cl_order(c.hclen - 1)]) c.hclen--;
    uint64_t hb = 3 + 5 + 5 + 4 + 3 * uint64_t(c.hclen);
    for (uint32_t k = 0; k < c.n_rle; k++) hb += c.cl_len[c.rle_sym[k]] + cl_extra(c.rle_sym[k]);
    c.header_bits = hb;
    uint64_t db = 0;
    for (uint32_t s = 0; s < 286; s++) db += uint64_t(c.lit_freq[s]) * (c.lit_len[s] + len_extra(s));
    for (uint32_t s = 0; s < 30; s++) db += uint64_t(c.dist_freq[s]) * (c.dist_len[s] + dist_extra(s));
    c.data_bits = db;
}
// Bytes of the Huffman-coded segment: block, then (not last) an empty stored block, byte-aligned.
HD uint64_t coded_bytes(const BlockCode& c, bool last) {
    return (c.header_bits + c.data_bits + (last ? 0 : 3) + 7) / 8 + (last ? 0 : 4);
}

// ---- bit packing ----------------------------------------------------------------------------------------------------

HD void or_bits(uint64_t* w, uint64_t pos, uint64_t val) {   // val < 2^57; plain (one writer at a time)
    const uint32_t sh = uint32_t(pos & 63);
    w[pos >> 6] |= val << sh;
    if (sh && (val >> (64 - sh))) w[(pos >> 6) + 1] |= val >> (64 - sh);
}
HD uint64_t write_header(const BlockCode& c, bool last, uint64_t* w) {
    uint64_t pos = 0;
    auto put = [&](uint64_t v, uint32_t n) { or_bits(w, pos, v); pos += n; };
    put((last ? 1u : 0u) | (2u << 1), 3);
    put(c.hlit - 257, 5); put(c.hdist - 1, 5); put(c.hclen - 4, 4);
    for (uint32_t i = 0; i < c.hclen; i++) put(c.cl_len[cl_order(i)], 3);
    for (uint32_t k = 0; k < c.n_rle; k++) {
        const uint32_t s = c.rle_sym[k];
        put(c.cl_code[s], c.cl_len[s]);
        if (cl_extra(s)) put(c.rle_extra[k], cl_extra(s));
    }
    return pos;
}
HD uint32_t token_bits(const BlockCode& c, uint32_t tok, uint64_t* val) {
    if (!(tok >> 31)) { *val = c.lit_code[tok]; return c.lit_len[tok]; }
    uint32_t nx, x, dnx, dx;
    const uint32_t ls = len_sym((tok & 0xff) + 3, &nx, &x);
    const uint32_t ds = dist_sym(((tok >> 8) & 0x7fff) + 1, &dnx, &dx);
    uint64_t v = c.lit_code[ls];
    uint32_t n = c.lit_len[ls];
    v |= uint64_t(x) << n; n += nx;
    v |= uint64_t(c.dist_code[ds]) << n; n += c.dist_len[ds];
    v |= uint64_t(dx) << n; n += dnx;
    *val = v;
    return n;
}

// Stored block headers of a segment of n bytes: block b at out[b * 65540], data behind it.
HD void stored_header(uint8_t* out, uint64_t n, uint32_t b, bool last) {
    const uint64_t nblk = (n + kStoredMax - 1) / kStoredMax;
    const uint32_t len = uint32_t(b + 1 == nblk ? n - uint64_t(b) * kStoredMax : kStoredMax);
    uint8_t* p = out + uint64_t(b) * (kStoredMax + 5);
    p[0] = (last && b + 1 == nblk) ? 1 : 0;
    p[1] = uint8_t(len); p[2] = uint8_t(len >> 8); p[3] = uint8_t(~len); p[4] = uint8_t(~len >> 8);
}
HD uint64_t stored_pos(uint64_t q) { return q + 5 * (q / kStoredMax + 1); }

// ---- checksums ------------------------------------------------------------------------------------------------------

constexpr uint32_t kBase = 65521;
// Adler-32 of X then Y from the sums of each (A = sum of bytes, B = sum of (n - i) * byte_i, mod 65521): zlib's
// adler32_combine arithmetic, starting from (1, 0).
HD void adler_append(uint32_t* a, uint32_t* b, uint32_t ay, uint32_t by, uint64_t ny) {
    *b = uint32_t((uint64_t(*b) + (ny % kBase) * *a + by) % kBase);
    *a = (*a + ay) % kBase;
}
constexpr uint32_t kPoly = 0xedb88320u;
HD uint32_t crc32_bytes(uint32_t crc, const uint8_t* p, uint64_t n) {
    uint32_t c = ~crc;
    for (uint64_t i = 0; i < n; i++) {
        c ^= p[i];
        for (int k = 0; k < 8; k++) c = (c >> 1) ^ (kPoly & (0u - (c & 1)));
    }
    return ~c;
}
// zlib's crc32_combine: a(x) * b(x) modulo the CRC polynomial (reflected), and x^(8n).
HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ kPoly : b >> 1;
    }
    return p;
}
HD uint32_t x8nmodp(uint64_t n) {
    uint32_t p = 1u << 31, q = 1u << 30;   // x^0, x^1
    for (int k = 0; k < 3; k++) q = multmodp(q, q);
    while (n) {
        if (n & 1) p = multmodp(q, p);
        n >>= 1;
        if (n) q = multmodp(q, q);
    }
    return p;
}
HD uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, uint64_t len2) { return multmodp(x8nmodp(len2), crc1) ^ crc2; }

// ---- framing --------------------------------------------------------------------------------------------------------

HD void put_be32(uint8_t* p, uint32_t v) { p[0] = uint8_t(v >> 24); p[1] = uint8_t(v >> 16); p[2] = uint8_t(v >> 8); p[3] = uint8_t(v); }
// Everything in the file except the segments' bytes and the IDAT CRCs.
HD void write_framing(uint8_t* f, uint32_t w, uint32_t h, uint64_t zlen, uint64_t chunk, uint32_t adler) {
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    for (int i = 0; i < 8; i++) f[i] = sig[i];
    put_be32(f + 8, 13);
    f[12] = 'I'; f[13] = 'H'; f[14] = 'D'; f[15] = 'R';
    put_be32(f + 16, w); put_be32(f + 20, h);
    f[24] = 8; f[25] = 2; f[26] = 0; f[27] = 0; f[28] = 0;   // 8-bit RGB, deflate, adaptive filtering, no interlace
    put_be32(f + 29, crc32_bytes(0, f + 12, 17));
    const uint64_t nchunks = (zlen + chunk - 1) / chunk;
    for (uint64_t c = 0; c < nchunks; c++) {
        uint8_t* p = f + kHeaderBytes + c * (chunk + 12);
        put_be32(p, uint32_t(c + 1 < nchunks ? chunk : zlen - c * chunk));
        p[4] = 'I'; p[5] = 'D'; p[6] = 'A'; p[7] = 'T';
    }
    const uint32_t cmf = 0x78, flg0 = 0;   // deflate, 32 KiB window; FLEVEL 0 (fastest), no dictionary
    f[file_offset(0, chunk)] = uint8_t(cmf);
    f[file_offset(1, chunk)] = uint8_t(flg0 + 31 - (cmf * 256 + flg0) % 31);   // FCHECK
    for (int i = 0; i < 4; i++) f[file_offset(zlen - 4 + i, chunk)] = uint8_t(adler >> (24 - 8 * i));
    uint8_t* e = f + file_bytes(zlen, chunk) - 12;
    const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xae, 0x42, 0x60, 0x82};
    for (int i = 0; i < 12; i++) e[i] = iend[i];
}
// The CRC of IDAT chunk c covers its type and data: (4 + data) bytes from file offset chunk_crc_start.
HD uint64_t chunk_crc_start(uint64_t c, uint64_t chunk) { return kHeaderBytes + c * (chunk + 12) + 4; }
HD uint64_t chunk_crc_len(uint64_t c, uint64_t zlen, uint64_t chunk) {
    return 4 + (zlen - c * chunk < chunk ? zlen - c * chunk : chunk);
}
HD uint64_t pieces_per_chunk(uint64_t chunk) { return (chunk + 4 + kCrcPiece - 1) / kCrcPiece; }
HD void finish_chunk_crc(uint8_t* f, uint64_t c, uint64_t zlen, uint64_t chunk, const uint32_t* piece_crc) {
    const uint64_t len = chunk_crc_len(c, zlen, chunk), np = (len + kCrcPiece - 1) / kCrcPiece;
    uint32_t crc = 0;
    for (uint64_t k = 0; k < np; k++) {
        const uint64_t n = (k + 1 < np) ? kCrcPiece : len - k * kCrcPiece;
        crc = crc32_combine(crc, piece_crc[c * pieces_per_chunk(chunk) + k], n);
    }
    put_be32(f + chunk_crc_start(c, chunk) + len, crc);
}

// ---- kernels --------------------------------------------------------------------------------------------------------

__global__ void __launch_bounds__(256) png_filter_kernel(const uint8_t* __restrict__ rgb, uint32_t w,
                                                         uint8_t* __restrict__ scan) {
    __shared__ unsigned long long s_cost[5];
    __shared__ uint32_t s_f;
    const uint64_t y = blockIdx.x, stride = 3 * uint64_t(w);
    const uint8_t* row = rgb + y * stride;
    const uint8_t* prev = y ? row - stride : nullptr;
    if (threadIdx.x < 5) s_cost[threadIdx.x] = 0;
    __syncthreads();
    uint64_t cost[5] = {0, 0, 0, 0, 0};
    for (uint64_t i = threadIdx.x; i < stride; i += blockDim.x) add_costs(row, prev, i, cost);
    for (int f = 0; f < 5; f++) atomicAdd(&s_cost[f], (unsigned long long)cost[f]);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t c[5];
        for (int f = 0; f < 5; f++) c[f] = s_cost[f];
        s_f = best_filter(c);
    }
    __syncthreads();
    const uint32_t f = s_f;
    uint8_t* out = scan + y * (stride + 1);
    if (threadIdx.x == 0) out[0] = uint8_t(f);
    for (uint64_t i = threadIdx.x; i < stride; i += blockDim.x) {
        int a, b, c;
        neighbours(row, prev, i, &a, &b, &c);
        out[1 + i] = filter_byte(f, row[i], a, b, c);
    }
}

// or_bits for many writers: tokens of one block land in shared words concurrently
__device__ __forceinline__ void or_bits_atomic(uint64_t* w, uint64_t pos, uint64_t val) {
    const uint32_t sh = uint32_t(pos & 63);
    atomicOr(reinterpret_cast<unsigned long long*>(w + (pos >> 6)), (unsigned long long)(val << sh));
    if (sh && (val >> (64 - sh)))
        atomicOr(reinterpret_cast<unsigned long long*>(w + (pos >> 6) + 1), (unsigned long long)(val >> (64 - sh)));
}

struct DeflateShared {
    int32_t table[1u << kHashBits];
    uint16_t len[kThreads], dist[kThreads];
    BlockCode code;
    uint16_t sorted[286 + 30];
    uint32_t A[286];
    unsigned long long adler[2];
    uint64_t carry;
    uint32_t ntok, m_lit, m_dist, stored;
    uint64_t bytes, bits;
};

// seg[4k..4k+3] of segment k: output bytes, Adler-32 A, Adler-32 B, 1 when stored
__global__ void __launch_bounds__(kThreads) png_deflate_kernel(const uint8_t* __restrict__ scan, uint64_t L, uint64_t S,
                                                               uint32_t* __restrict__ tokens, uint8_t* __restrict__ slots,
                                                               uint32_t* __restrict__ seg) {
    __shared__ DeflateShared sh;
    using Scan = cub::BlockScan<uint32_t, kThreads>;
    __shared__ typename Scan::TempStorage scan_tmp;
    const uint32_t tid = threadIdx.x, k = blockIdx.x, lane = tid & 31;
    const uint64_t s0 = uint64_t(k) * S, s1 = (s0 + S < L) ? s0 + S : L, n = s1 - s0;
    const bool last = s1 == L;
    const int64_t base = window_base(s0);
    uint32_t* tok = tokens + s0;
    uint8_t* out = slots + uint64_t(k) * slot_bytes(S);

    for (uint32_t i = tid; i < (1u << kHashBits); i += kThreads) sh.table[i] = 0;
    for (uint32_t i = tid; i < 286; i += kThreads) sh.code.lit_freq[i] = 0;
    if (tid < 30) sh.code.dist_freq[tid] = 0;
    if (tid < 2) sh.adler[tid] = 0;
    if (tid == 0) { sh.carry = s0; sh.ntok = 0; }
    __syncthreads();
    // Adler-32 sums of the segment
    {
        unsigned long long a = 0, b = 0;
        for (uint64_t i = tid; i < n; i += kThreads) { a += scan[s0 + i]; b += (n - i) * scan[s0 + i]; }
        atomicAdd(&sh.adler[0], a % kBase);
        atomicAdd(&sh.adler[1], b % kBase);
    }
    // the window before the segment: matches may reach back into earlier segments
    for (uint64_t p = uint64_t(base > 0 ? base : 0) + tid; p < s0; p += kThreads)
        if (p + 2 < L) atomicMax(&sh.table[hash3(scan + p)], int32_t(int64_t(p) - base + 1));
    __syncthreads();

    for (uint64_t t0 = s0; t0 < s1; t0 += kThreads) {
        const uint64_t p = t0 + tid, te = (t0 + kThreads < s1) ? t0 + kThreads : s1;
        const bool hashable = p < te && p + 2 < L;
        uint32_t h = 0;
        int32_t cand = 0;
        if (hashable) { h = hash3(scan + p); cand = sh.table[h]; }
        __syncthreads();
        if (hashable) atomicMax(&sh.table[h], int32_t(int64_t(p) - base + 1));
        if (p < te) {
            uint32_t d;
            sh.len[tid] = uint16_t(probe(scan, p, s1, base, cand, &d));
            sh.dist[tid] = uint16_t(d);
        }
        __syncthreads();
        if (tid < 32) {   // greedy parse of the round's positions by one warp
            uint64_t q = sh.carry;
            uint32_t nt = sh.ntok;
            while (q < te) {
                uint32_t l = sh.len[q - t0], t;
                if (l >= 3) {
                    const uint32_t d = sh.dist[q - t0];
                    const uint32_t maxlen = uint32_t(s1 - q < kMaxMatch ? s1 - q : kMaxMatch);
                    if (l == kProbe && maxlen > kProbe) {   // extend: 8 bytes per lane covers up to 16 + 256
                        const uint32_t from = kProbe + lane * 8;
                        uint32_t first = 0xffffffffu;
                        for (uint32_t i = from; i < from + 8 && i < maxlen; i++)
                            if (scan[q + i] != scan[q - d + i]) { first = i; break; }
                        const uint32_t mask = __ballot_sync(0xffffffffu, first != 0xffffffffu);
                        l = mask ? __shfl_sync(0xffffffffu, first, __ffs(mask) - 1) : maxlen;
                    }
                    t = tok_match(l, d);
                    q += l;
                } else {
                    t = scan[q];
                    q++;
                }
                if (lane == 0) tok[nt] = t;
                nt++;
            }
            if (lane == 0) { sh.carry = q; sh.ntok = nt; }
        }
        __syncthreads();
    }

    const uint32_t ntok = sh.ntok;
    for (uint32_t i = tid; i < ntok; i += kThreads) {
        const uint32_t t = tok[i];
        if (!(t >> 31)) { atomicAdd(&sh.code.lit_freq[t], 1u); continue; }
        uint32_t nx, x;
        atomicAdd(&sh.code.lit_freq[len_sym((t & 0xff) + 3, &nx, &x)], 1u);
        atomicAdd(&sh.code.dist_freq[dist_sym(((t >> 8) & 0x7fff) + 1, &nx, &x)], 1u);
    }
    __syncthreads();
    if (tid == 0) sh.code.lit_freq[256] = 1;   // end of block
    __syncthreads();
    // sort the used symbols by (frequency, symbol): one thread per symbol
    if (tid < 286) {
        sh.code.lit_len[tid] = 0;
        if (sh.code.lit_freq[tid]) sh.sorted[sym_rank(sh.code.lit_freq, 286, tid)] = uint16_t(tid);
    } else if (tid < 316) {
        const uint32_t i = tid - 286;
        sh.code.dist_len[i] = 0;
        if (sh.code.dist_freq[i]) sh.sorted[286 + sym_rank(sh.code.dist_freq, 30, i)] = uint16_t(i);
    }
    __syncthreads();
    if (tid == 0) {
        BlockCode& c = sh.code;
        uint32_t m = 0;
        for (uint32_t i = 0; i < 286; i++) m += c.lit_freq[i] ? 1u : 0u;
        for (uint32_t i = 0; i < m; i++) sh.A[i] = c.lit_freq[sh.sorted[i]];
        lengths_from_sorted(sh.sorted, sh.A, m, 15, c.lit_len);
        m = 0;
        for (uint32_t i = 0; i < 30; i++) m += c.dist_freq[i] ? 1u : 0u;
        for (uint32_t i = 0; i < m; i++) sh.A[i] = c.dist_freq[sh.sorted[286 + i]];
        lengths_from_sorted(sh.sorted + 286, sh.A, m, 15, c.dist_len);
        finish_code(c, sh.sorted, sh.A);
        const uint64_t cb = coded_bytes(c, last), sb = stored_size(n);
        sh.stored = cb >= sb;
        sh.bytes = sh.stored ? sb : cb;
        seg[4 * k + 0] = uint32_t(sh.bytes);
        seg[4 * k + 1] = uint32_t(sh.adler[0] % kBase);
        seg[4 * k + 2] = uint32_t(sh.adler[1] % kBase);
        seg[4 * k + 3] = sh.stored;
    }
    __syncthreads();
    if (sh.stored) {
        const uint32_t nblk = uint32_t((n + kStoredMax - 1) / kStoredMax);
        if (tid < nblk) stored_header(out, n, tid, last);
        for (uint64_t q = tid; q < n; q += kThreads) out[stored_pos(q)] = scan[s0 + q];
        return;
    }
    uint64_t* words = reinterpret_cast<uint64_t*>(out);
    const uint64_t nwords = (sh.bytes + 7) / 8;
    for (uint64_t i = tid; i < nwords; i += kThreads) words[i] = 0;
    __syncthreads();
    if (tid == 0) sh.bits = write_header(sh.code, last, words);
    __syncthreads();
    uint64_t pos = sh.bits;
    for (uint32_t i0 = 0; i0 < ntok; i0 += kThreads) {
        uint64_t v = 0;
        const uint32_t nb = (i0 + tid < ntok) ? token_bits(sh.code, tok[i0 + tid], &v) : 0;
        uint32_t off, total;
        Scan(scan_tmp).ExclusiveSum(nb, off, total);
        if (nb) or_bits_atomic(words, pos + off, v);
        pos += total;
        __syncthreads();
    }
    if (tid == 0) {
        or_bits_atomic(words, pos, sh.code.lit_code[256]);   // end of block; the empty stored block's 3 bits are zeros
        if (!last) {
            uint8_t* tail = out + sh.bytes - 4;
            tail[0] = 0; tail[1] = 0; tail[2] = 0xff; tail[3] = 0xff;
        }
    }
}

// One thread: segment offsets in the zlib stream, the Adler-32 of the stream, the framing.  info = {file bytes, stored}
__global__ void png_layout_kernel(const uint32_t* __restrict__ seg, uint32_t nseg, uint64_t L, uint32_t w, uint32_t h,
                                  uint64_t chunk, uint64_t* __restrict__ zoff, uint8_t* __restrict__ file,
                                  uint64_t* __restrict__ info) {
    const uint64_t S = segment_bytes(L);
    uint64_t z = 2;
    uint32_t a = 1, b = 0, stored = 0;
    for (uint32_t k = 0; k < nseg; k++) {
        zoff[k] = z;
        z += seg[4 * k];
        const uint64_t s0 = uint64_t(k) * S;
        adler_append(&a, &b, seg[4 * k + 1], seg[4 * k + 2], (s0 + S < L ? s0 + S : L) - s0);
        stored += seg[4 * k + 3];
    }
    const uint64_t zlen = z + 4;
    write_framing(file, w, h, zlen, chunk, (b << 16) | a);
    info[0] = file_bytes(zlen, chunk);
    info[1] = stored;
    info[2] = zlen;
}

// One block per segment.  A segment's bytes cross at most one IDAT boundary (slot_bytes(S) <= chunk).
__global__ void __launch_bounds__(256) png_gather_kernel(const uint8_t* __restrict__ slots, uint64_t slot,
                                                         const uint32_t* __restrict__ seg, const uint64_t* __restrict__ zoff,
                                                         uint64_t chunk, uint8_t* __restrict__ file) {
    const uint32_t k = blockIdx.x;
    const uint64_t z0 = zoff[k], n = seg[4 * k], f0 = file_offset(z0, chunk);
    const uint64_t split = (z0 / chunk + 1) * chunk - z0;   // bytes before the next chunk boundary
    const uint8_t* src = slots + uint64_t(k) * slot;
    for (uint64_t q = threadIdx.x; q < n; q += blockDim.x) file[f0 + q + (q >= split ? 12 : 0)] = src[q];
}

// CRC-32 of piece blockIdx.x of the IDATs' checked bytes: kCrcThreads sub-pieces, combined in a tree.
__global__ void __launch_bounds__(kCrcThreads) png_crc_kernel(const uint8_t* __restrict__ file, const uint64_t* __restrict__ info,
                                                              uint64_t chunk, uint32_t* __restrict__ piece_crc) {
    __shared__ uint32_t table[256];
    __shared__ uint32_t crc[kCrcThreads];
    __shared__ uint32_t len[kCrcThreads];
    const uint64_t zlen = info[2], ppc = pieces_per_chunk(chunk);
    const uint64_t c = blockIdx.x / ppc, kp = blockIdx.x % ppc;
    if (c * chunk >= zlen) return;
    const uint64_t total = chunk_crc_len(c, zlen, chunk);
    if (kp * kCrcPiece >= total) return;
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t v = i;
        for (int b = 0; b < 8; b++) v = (v >> 1) ^ (kPoly & (0u - (v & 1)));
        table[i] = v;
    }
    __syncthreads();
    const uint64_t p0 = kp * kCrcPiece, pn = (total - p0 < kCrcPiece) ? total - p0 : kCrcPiece;
    constexpr uint32_t kSub = kCrcPiece / kCrcThreads;
    const uint64_t a = uint64_t(threadIdx.x) * kSub;
    const uint64_t e = (a + kSub < pn) ? a + kSub : pn;
    const uint8_t* p = file + chunk_crc_start(c, chunk) + p0;
    uint32_t v = 0xffffffffu;
    for (uint64_t i = a; i < e; i++) v = table[(v ^ p[i]) & 0xff] ^ (v >> 8);
    crc[threadIdx.x] = a < e ? ~v : 0;
    len[threadIdx.x] = a < e ? uint32_t(e - a) : 0;
    __syncthreads();
    for (uint32_t s = 1; s < kCrcThreads; s *= 2) {
        if ((threadIdx.x & (2 * s - 1)) == 0 && len[threadIdx.x + s]) {
            crc[threadIdx.x] = crc32_combine(crc[threadIdx.x], crc[threadIdx.x + s], len[threadIdx.x + s]);
            len[threadIdx.x] += len[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) piece_crc[blockIdx.x] = crc[0];
}

__global__ void png_crc_finish_kernel(uint8_t* __restrict__ file, const uint64_t* __restrict__ info, uint64_t chunk,
                                      uint64_t max_chunks, const uint32_t* __restrict__ piece_crc) {
    const uint64_t c = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x, zlen = info[2];
    if (c >= max_chunks || c * chunk >= zlen) return;
    finish_chunk_crc(file, c, zlen, chunk, piece_crc);
}

template <typename T>
cudaError_t grow(T** p, size_t* cap, size_t need) {
    if (*cap >= need) return cudaSuccess;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    cudaError_t e = cudaMalloc(p, need * sizeof(T));
    if (e == cudaSuccess) *cap = need;
    return e;
}

// ---- the CPU twin ---------------------------------------------------------------------------------------------------

struct HostSegment { std::vector<uint8_t> bytes; uint32_t adler_a = 0, adler_b = 0; bool stored = false; };

// Segment [s0, s1) of the scanline stream, as png_deflate_kernel encodes it, one position and one token at a time.
void encode_segment_host(const uint8_t* scan, uint64_t L, uint64_t s0, uint64_t s1, HostSegment* out) {
    const uint64_t n = s1 - s0;
    const bool last = s1 == L;
    const int64_t base = window_base(s0);
    uint64_t a = 0, b = 0;
    for (uint64_t i = 0; i < n; i++) { a += scan[s0 + i]; b += (n - i) * scan[s0 + i]; }
    out->adler_a = uint32_t(a % kBase); out->adler_b = uint32_t(b % kBase);
    std::vector<int32_t> table(1u << kHashBits, 0);
    for (uint64_t p = uint64_t(base > 0 ? base : 0); p < s0; p++)
        if (p + 2 < L) { int32_t& t = table[hash3(scan + p)]; t = std::max(t, int32_t(int64_t(p) - base + 1)); }
    std::vector<uint32_t> tok;
    uint32_t len[kThreads], dist[kThreads];
    int32_t cand[kThreads];
    uint64_t carry = s0;
    for (uint64_t t0 = s0; t0 < s1; t0 += kThreads) {
        const uint64_t te = std::min(t0 + kThreads, s1);
        for (uint64_t p = t0; p < te; p++) cand[p - t0] = p + 2 < L ? table[hash3(scan + p)] : 0;
        for (uint64_t p = t0; p < te; p++)
            if (p + 2 < L) { int32_t& t = table[hash3(scan + p)]; t = std::max(t, int32_t(int64_t(p) - base + 1)); }
        for (uint64_t p = t0; p < te; p++) len[p - t0] = probe(scan, p, s1, base, cand[p - t0], &dist[p - t0]);
        uint64_t q = carry;
        while (q < te) {
            uint32_t l = len[q - t0];
            if (l >= 3) {
                const uint32_t d = dist[q - t0];
                const uint32_t maxlen = uint32_t(std::min<uint64_t>(s1 - q, kMaxMatch));
                if (l == kProbe && maxlen > kProbe) l = match_len(scan, q, q - d, maxlen);
                tok.push_back(tok_match(l, d));
                q += l;
            } else {
                tok.push_back(scan[q]);
                q++;
            }
        }
        carry = q;
    }
    BlockCode c{};
    for (uint32_t t : tok) {
        if (!(t >> 31)) { c.lit_freq[t]++; continue; }
        uint32_t nx, x;
        c.lit_freq[len_sym((t & 0xff) + 3, &nx, &x)]++;
        c.dist_freq[dist_sym(((t >> 8) & 0x7fff) + 1, &nx, &x)]++;
    }
    c.lit_freq[256] = 1;
    uint16_t sorted[286];
    uint32_t A[286];
    build_lengths(c.lit_freq, 286, 15, c.lit_len, sorted, A);
    build_lengths(c.dist_freq, 30, 15, c.dist_len, sorted, A);
    finish_code(c, sorted, A);
    const uint64_t cb = coded_bytes(c, last), sb = stored_size(n);
    out->stored = cb >= sb;
    if (out->stored) {
        out->bytes.assign(sb, 0);
        for (uint32_t k = 0; k < (n + kStoredMax - 1) / kStoredMax; k++) stored_header(out->bytes.data(), n, k, last);
        for (uint64_t q = 0; q < n; q++) out->bytes[stored_pos(q)] = scan[s0 + q];
        return;
    }
    std::vector<uint64_t> words((cb + 7) / 8 + 1, 0);
    uint64_t pos = write_header(c, last, words.data());
    for (uint32_t t : tok) {
        uint64_t v;
        const uint32_t nb = token_bits(c, t, &v);
        or_bits(words.data(), pos, v);
        pos += nb;
    }
    or_bits(words.data(), pos, c.lit_code[256]);
    out->bytes.assign(reinterpret_cast<uint8_t*>(words.data()), reinterpret_cast<uint8_t*>(words.data()) + cb);
    if (!last) { out->bytes[cb - 2] = 0xff; out->bytes[cb - 1] = 0xff; }
}

std::vector<uint8_t> encode_host(const uint8_t* rgb, uint32_t w, uint32_t h, uint64_t chunk, uint32_t* segments,
                                 uint32_t* stored) {
    const uint64_t stride = 3 * uint64_t(w), L = uint64_t(h) * (stride + 1);
    std::vector<uint8_t> scan(L);
    for (uint64_t y = 0; y < h; y++) {
        const uint8_t* row = rgb + y * stride;
        const uint8_t* prev = y ? row - stride : nullptr;
        uint64_t cost[5] = {0, 0, 0, 0, 0};
        for (uint64_t i = 0; i < stride; i++) add_costs(row, prev, i, cost);
        const uint32_t f = best_filter(cost);
        uint8_t* o = &scan[y * (stride + 1)];
        o[0] = uint8_t(f);
        for (uint64_t i = 0; i < stride; i++) {
            int a, b, c;
            neighbours(row, prev, i, &a, &b, &c);
            o[1 + i] = filter_byte(f, row[i], a, b, c);
        }
    }
    const uint64_t S = segment_bytes(L), nseg = (L + S - 1) / S;
    std::vector<HostSegment> segs(nseg);
    uint64_t z = 2;
    uint32_t a = 1, b = 0;
    *stored = 0;
    for (uint64_t k = 0; k < nseg; k++) {
        const uint64_t s0 = k * S, s1 = std::min(L, s0 + S);
        encode_segment_host(scan.data(), L, s0, s1, &segs[k]);
        adler_append(&a, &b, segs[k].adler_a, segs[k].adler_b, s1 - s0);
        z += segs[k].bytes.size();
        *stored += segs[k].stored ? 1 : 0;
    }
    *segments = uint32_t(nseg);
    const uint64_t zlen = z + 4;
    std::vector<uint8_t> file(file_bytes(zlen, chunk), 0);
    write_framing(file.data(), w, h, zlen, chunk, (b << 16) | a);
    z = 2;
    for (const HostSegment& s : segs)
        for (uint8_t v : s.bytes) file[file_offset(z++, chunk)] = v;
    const uint64_t nchunks = (zlen + chunk - 1) / chunk, ppc = pieces_per_chunk(chunk);
    std::vector<uint32_t> piece_crc(nchunks * ppc, 0);
    for (uint64_t c = 0; c < nchunks; c++) {
        const uint64_t len = chunk_crc_len(c, zlen, chunk);
        for (uint64_t k = 0; k * kCrcPiece < len; k++)
            piece_crc[c * ppc + k] = crc32_bytes(0, &file[chunk_crc_start(c, chunk) + k * kCrcPiece],
                                                 std::min<uint64_t>(kCrcPiece, len - k * kCrcPiece));
        finish_chunk_crc(file.data(), c, zlen, chunk, piece_crc.data());
    }
    return file;
}

double now_ms() {
    using namespace std::chrono;
    return duration<double, std::milli>(steady_clock::now().time_since_epoch()).count();
}

}  // namespace

cudaError_t png_encode_device(PngScratch& sc, const uint8_t* d_rgb, uint32_t w, uint32_t hgt, cudaStream_t stream,
                              PngResult* res, std::string* err) {
#define PNG_TRY(expr)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess) { *err = std::string(#expr) + ": " + cudaGetErrorString(e_); return e_; } \
    } while (0)
    const uint64_t L = uint64_t(hgt) * (3 * uint64_t(w) + 1);
    const uint64_t S = segment_bytes(L), nseg = (L + S - 1) / S, slot = slot_bytes(S);
    const uint64_t zbound = 2 + nseg * slot + 4, max_chunks = (zbound + kIdatBytes - 1) / kIdatBytes;
    const uint64_t fbound = file_bytes(zbound, kIdatBytes), ppc = pieces_per_chunk(kIdatBytes);
    const uint64_t npieces = max_chunks == 1 ? (zbound + 4 + kCrcPiece - 1) / kCrcPiece : max_chunks * ppc;
    PNG_TRY(grow(&sc.d_scan, &sc.scan_cap, L));
    PNG_TRY(grow(&sc.d_tokens, &sc.tokens_cap, L));
    PNG_TRY(grow(&sc.d_slots, &sc.slots_cap, nseg * slot));
    PNG_TRY(grow(&sc.d_seg, &sc.seg_cap, 4 * nseg));
    PNG_TRY(grow(&sc.d_zoff, &sc.zoff_cap, nseg));
    PNG_TRY(grow(&sc.d_file, &sc.file_cap, fbound));
    PNG_TRY(grow(&sc.d_crc, &sc.crc_cap, npieces));
    if (!sc.d_info) PNG_TRY(cudaMalloc(&sc.d_info, 4 * sizeof(uint64_t)));
    if (!sc.ev0) { PNG_TRY(cudaEventCreate(&sc.ev0)); PNG_TRY(cudaEventCreate(&sc.ev1)); }

    PNG_TRY(cudaEventRecord(sc.ev0, stream));
    png_filter_kernel<<<hgt, 256, 0, stream>>>(d_rgb, w, sc.d_scan);
    png_deflate_kernel<<<uint32_t(nseg), kThreads, 0, stream>>>(sc.d_scan, L, S, sc.d_tokens, sc.d_slots, sc.d_seg);
    png_layout_kernel<<<1, 1, 0, stream>>>(sc.d_seg, uint32_t(nseg), L, w, hgt, kIdatBytes, sc.d_zoff, sc.d_file, sc.d_info);
    png_gather_kernel<<<uint32_t(nseg), 256, 0, stream>>>(sc.d_slots, slot, sc.d_seg, sc.d_zoff, kIdatBytes, sc.d_file);
    png_crc_kernel<<<uint32_t(npieces), kCrcThreads, 0, stream>>>(sc.d_file, sc.d_info, kIdatBytes, sc.d_crc);
    png_crc_finish_kernel<<<uint32_t((max_chunks + 127) / 128), 128, 0, stream>>>(sc.d_file, sc.d_info, kIdatBytes,
                                                                                 max_chunks, sc.d_crc);
    PNG_TRY(cudaGetLastError());
    PNG_TRY(cudaEventRecord(sc.ev1, stream));
    uint64_t info[4];
    PNG_TRY(cudaMemcpyAsync(info, sc.d_info, sizeof info, cudaMemcpyDeviceToHost, stream));
    PNG_TRY(cudaStreamSynchronize(stream));
    float ms = 0.f;
    PNG_TRY(cudaEventElapsedTime(&ms, sc.ev0, sc.ev1));
    const double t0 = now_ms();
    if (sc.h_cap < info[0]) {
        if (sc.h_file) cudaFreeHost(sc.h_file);
        sc.h_file = nullptr; sc.h_cap = 0;
        PNG_TRY(cudaMallocHost(&sc.h_file, info[0]));
        sc.h_cap = info[0];
    }
    PNG_TRY(cudaMemcpyAsync(sc.h_file, sc.d_file, info[0], cudaMemcpyDeviceToHost, stream));
    PNG_TRY(cudaStreamSynchronize(stream));
    res->file = sc.h_file;
    res->file_bytes = info[0];
    res->scanline_bytes = L;
    res->segments = uint32_t(nseg);
    res->stored_segments = uint32_t(info[1]);
    res->encode_ms = ms;
    res->d2h_ms = now_ms() - t0;
    return cudaSuccess;
#undef PNG_TRY
}

void png_release(PngScratch& sc) {
    cudaFree(sc.d_scan); cudaFree(sc.d_tokens); cudaFree(sc.d_slots); cudaFree(sc.d_seg); cudaFree(sc.d_zoff);
    cudaFree(sc.d_file); cudaFree(sc.d_crc); cudaFree(sc.d_info);
    if (sc.h_file) cudaFreeHost(sc.h_file);
    if (sc.ev0) cudaEventDestroy(sc.ev0);
    if (sc.ev1) cudaEventDestroy(sc.ev1);
    sc = PngScratch{};
}

}  // namespace maray

// The encoder's CPU twin, for tests: the same file png_encode_device writes for this frame, built serially on the
// host.  `idat_bytes` is the IDAT payload size (the library uses 2^30; tests pass small values to get many chunks).
// Writes at most `cap` bytes to `out`; *len receives the file size (MARAY_E_INVALID when it exceeds cap).
extern "C" __attribute__((visibility("default"))) int maray_cuda_png_encode_host(
    const uint8_t* rgb, uint32_t w, uint32_t hgt, uint64_t idat_bytes, uint8_t* out, size_t cap, size_t* len,
    uint32_t* segments, uint32_t* stored) {
    if (!rgb || !len || !segments || !stored || !w || !hgt || w > 0x7fffffffu || hgt > 0x7fffffffu ||
        idat_bytes == 0 || idat_bytes > 0x7fffffffu)
        return MARAY_E_INVALID;
    std::vector<uint8_t> f = maray::encode_host(rgb, w, hgt, idat_bytes, segments, stored);
    *len = f.size();
    if (f.size() > cap || !out) return MARAY_E_INVALID;
    std::memcpy(out, f.data(), f.size());
    return MARAY_OK;
}
