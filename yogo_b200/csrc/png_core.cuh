// Per-stream pieces of the PNG decoder (png.cu): CRC-32, Adler-32, the DEFLATE bit reader, Huffman table build and
// symbol decode, and the scanline unfilter.  Everything here is __host__ __device__ and free of CUDA intrinsics, so
// the same code can be compiled for the host and checked against zlib on a CPU.
#pragma once
#include <stdint.h>
#include "../../include/yogo_b200.h"
#ifndef __CUDACC__
#define __host__
#define __device__
#define __forceinline__ inline
#endif

namespace yg {
namespace png {

#define PNG_HD __host__ __device__ __forceinline__

// ---- CRC-32 (ISO-HDLC, reflected polynomial 0xedb88320) -------------------------------------------------------------
struct CrcTables {
  uint32_t byte[256];   // one-byte update
  uint32_t x2n[32];     // x^(2^k) mod p, for combining the CRCs of concatenated pieces (zlib's crc32_combine)
};
constexpr uint32_t CRC_POLY = 0xedb88320u;

// a(x) * b(x) mod p(x), reflected (zlib's multmodp)
PNG_HD constexpr uint32_t multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ CRC_POLY : b >> 1;
  }
  return p;
}

constexpr CrcTables make_crc_tables() {
  CrcTables t{};
  for (uint32_t n = 0; n < 256; ++n) {
    uint32_t c = n;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
    t.byte[n] = c;
  }
  uint32_t p = 1u << 30;   // x^1
  t.x2n[0] = p;
  for (int n = 1; n < 32; ++n) t.x2n[n] = p = multmodp(p, p);
  return t;
}

// x^(n * 2^k) mod p
PNG_HD uint32_t x2nmodp(const CrcTables& t, unsigned long long n, unsigned k) {
  uint32_t p = 1u << 31;   // x^0
  while (n) {
    if (n & 1) p = multmodp(t.x2n[k & 31], p);
    n >>= 1;
    ++k;
  }
  return p;
}

// crc32(A || B) from crc32(A), crc32(B) and len(B)
PNG_HD uint32_t crc32_combine(const CrcTables& t, uint32_t crc_a, uint32_t crc_b, unsigned long long len_b) {
  return multmodp(x2nmodp(t, len_b, 3), crc_a) ^ crc_b;
}

// ---- Adler-32 -----------------------------------------------------------------------------------------------------
// Over bytes b_0..b_{n-1}: A = 1 + sum b_i, B = n + sum (n - i) b_i (mod 65521); both sums split over any partition.
constexpr uint32_t ADLER_MOD = 65521u;

// ---- DEFLATE (RFC 1951) -------------------------------------------------------------------------------------------
enum { LIT_BITS = 10, DIST_BITS = 8, CL_BITS = 7 };   // primary-table index widths; longer codes take the slow path
enum { MAX_LIT = 288, MAX_DIST = 32 };

// canonical Huffman code: codes per length and the symbols in code order (puff.c's representation)
struct Huff {
  uint16_t count[16];
  uint16_t sym[MAX_LIT];
};

// primary-table entry: symbol in bits 0..11, code length in bits 12..15; 0 = slow path (longer code or unused code)
PNG_HD uint16_t tab_entry(int sym, int len) { return (uint16_t)(sym | (len << 12)); }

PNG_HD uint32_t bit_reverse(uint32_t code, int len) {
  uint32_t r = 0;
  for (int i = 0; i < len; ++i) {
    r = (r << 1) | (code & 1);
    code >>= 1;
  }
  return r;
}

// Fills h from the code lengths; returns the number of unused codes at length 15 scaled as zlib's `left`
// (0 = complete), or -1 when over-subscribed or a length exceeds 15.
PNG_HD int huff_counts(Huff& h, const uint16_t* lens, int n) {
  for (int l = 0; l < 16; ++l) h.count[l] = 0;
  for (int s = 0; s < n; ++s) {
    if (lens[s] > 15) return -1;
    h.count[lens[s]]++;
  }
  int left = 1;
  for (int l = 1; l < 16; ++l) {
    left <<= 1;
    left -= h.count[l];
    if (left < 0) return -1;
  }
  uint16_t offs[16];
  offs[1] = 0;
  for (int l = 1; l < 15; ++l) offs[l + 1] = (uint16_t)(offs[l] + h.count[l]);
  for (int s = 0; s < n; ++s)
    if (lens[s]) h.sym[offs[lens[s]]++] = (uint16_t)s;
  return left;
}

// Primary table of `bits` index bits from h (after huff_counts).  The caller clears the table to 0 first; entries are
// written by lanes lane, lane + nlanes, ... over the coded symbols, so a warp can fill it in parallel (nlanes = 1 on the
// host).  Every index written is < 1 << bits by construction (code length <= bits).
PNG_HD void huff_fill(const Huff& h, const uint16_t* lens, uint16_t* tab, int bits, int lane, int nlanes) {
  int ncoded = 0;
  for (int l = 1; l < 16; ++l) ncoded += h.count[l];
  for (int i = lane; i < ncoded; i += nlanes) {
    const int s = h.sym[i];
    const int len = lens[s];
    if (len > bits) continue;
    // canonical code of the i-th symbol in code order: first code of its length + rank within the length
    int code = 0, start = 0;
    for (int l = 1; l < len; ++l) {
      code = (code + h.count[l]) << 1;
      start += h.count[l];
    }
    code += i - start;
    const uint32_t rev = bit_reverse((uint32_t)code, len);
    for (uint32_t k = rev; k < (1u << bits); k += 1u << len) tab[k] = tab_entry(s, len);
  }
}

// Decodes one symbol from the low bits of `bits` (at least 15 valid).  Returns the symbol and sets len, or returns -1
// when the bits are not a code of this table (an incomplete distance code).
PNG_HD int huff_decode(const uint16_t* tab, int tbits, const Huff& h, uint64_t bits, int& len) {
  const uint16_t e = tab[bits & ((1u << tbits) - 1)];
  if (e >> 12) {
    len = e >> 12;
    return e & 0xfff;
  }
  int code = 0, first = 0, index = 0;
  for (int l = 1; l < 16; ++l) {
    code |= (int)((bits >> (l - 1)) & 1);
    const int count = h.count[l];
    if (code < first + count) {
      len = l;
      return h.sym[index + code - first];
    }
    index += count;
    first = (first + count) << 1;
    code <<= 1;
  }
  len = 0;
  return -1;
}

// Validity of a code built by huff_counts, as zlib's inflate_table: the literal/length and code-length codes must be
// complete; a distance code may also be empty or a single code of length 1.
PNG_HD bool code_ok(int left, const Huff& h, bool is_dist) {
  if (left < 0) return false;
  if (left == 0) return true;
  if (!is_dist) return false;
  int ncoded = 0;
  for (int l = 1; l < 16; ++l) ncoded += h.count[l];
  return ncoded == 0 || (ncoded == 1 && h.count[1] == 1);
}

// length / distance base values and extra bits (RFC 1951 3.2.5)
// (i = symbol - 257 / distance symbol), in closed form so that no table is needed
PNG_HD int len_extra(int i) { return (i < 8 || i == 28) ? 0 : (i - 4) >> 2; }
PNG_HD int len_base(int i) { return i < 8 ? 3 + i : i == 28 ? 258 : ((4 + ((i - 4) & 3)) << len_extra(i)) + 3; }
PNG_HD int dist_extra(int i) { return i < 4 ? 0 : (i - 2) >> 1; }
PNG_HD int dist_base(int i) { return i < 4 ? 1 + i : ((2 + (i & 1)) << dist_extra(i)) + 1; }

// order of the code-length code lengths in a dynamic block header
PNG_HD int clen_order(int i) {
  constexpr uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
  return order[i];
}

// LSB-first bit reader over one zlib stream of `len` bytes.  Bytes in [wbase, wbase + wlen) come from `win` (a
// shared-memory copy on the device), others from `src`; positions at or past `len` read as zero.  Whether the stream
// really ended early is decided from consumed() > len, since the reader runs up to 4 bytes ahead.
struct BitReader {
  const uint8_t* src;
  long long len;
  const uint8_t* win;
  long long wbase;
  int wlen;
  long long pos;   // next byte to load
  uint64_t buf;
  int cnt;         // valid bits in buf

  PNG_HD uint32_t byte(long long p) const {
    if (p >= len) return 0;
    const long long w = p - wbase;
    return (w >= 0 && w < wlen) ? win[w] : src[p];
  }
  // at least 32 valid bits afterwards
  PNG_HD void refill() {
    if (cnt < 32) {
      const uint32_t w = byte(pos) | byte(pos + 1) << 8 | byte(pos + 2) << 16 | byte(pos + 3) << 24;
      buf |= (uint64_t)w << cnt;
      cnt += 32;
      pos += 4;
    }
  }
  PNG_HD uint32_t peek(int n) const { return (uint32_t)(buf & ((1ull << n) - 1)); }
  PNG_HD void drop(int n) {
    buf >>= n;
    cnt -= n;
  }
  // n <= 32 bits; refills first
  PNG_HD uint32_t bits(int n) {
    refill();
    const uint32_t v = peek(n);
    drop(n);
    return v;
  }
  // byte position of the next unconsumed bit, rounded up
  PNG_HD long long byte_pos() const { return pos - (cnt >> 3); }
  PNG_HD long long consumed_bits() const { return pos * 8 - cnt; }
  PNG_HD void align() { drop(cnt & 7); }
  // continue reading whole bytes at p (after align())
  PNG_HD void seek(long long p) {
    pos = p;
    buf = 0;
    cnt = 0;
  }
};

// ---- inflate stages, run by one thread (lane 0 of the decoding warp on the device) ---------------------------------
struct InflateTables {
  uint16_t lit[1 << LIT_BITS];
  uint16_t dist[1 << DIST_BITS];   // also the code-length code's table while a dynamic header is read
  Huff hl, hd;
  uint16_t lens[MAX_LIT + MAX_DIST];
};

// zlib header (RFC 1950): CM 8, CINFO <= 7, FCHECK, no preset dictionary.  Sets the window size.
PNG_HD int zlib_header(BitReader& br, int& window) {
  const uint32_t cmf = br.bits(8), flg = br.bits(8);
  if ((cmf & 15) != 8 || (cmf >> 4) > 7 || (cmf * 256 + flg) % 31 != 0 || (flg & 32)) return YG_PNG_BAD_ZLIB_HEADER;
  window = 1 << ((cmf >> 4) + 8);
  return YG_PNG_OK;
}

// Code lengths of the fixed block (RFC 1951 3.2.6): all 288 / 32 symbols, so that 286, 287, 30 and 31 decode and are
// then rejected as invalid symbols, as zlib does.
PNG_HD void fixed_lengths(InflateTables& t) {
  for (int s = 0; s < MAX_LIT; ++s) t.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
  for (int s = 0; s < MAX_DIST; ++s) t.lens[MAX_LIT + s] = 5;
  huff_counts(t.hl, t.lens, MAX_LIT);
  huff_counts(t.hd, t.lens + MAX_LIT, MAX_DIST);
}

// Dynamic block header: reads the code-length code and the literal/length and distance code lengths into t.lens (the
// distance lengths at MAX_LIT), and counts both codes into t.hl / t.hd.  The caller fills the primary tables.
PNG_HD int dynamic_lengths(BitReader& br, InflateTables& t) {
  const int nlen = (int)br.bits(5) + 257, ndist = (int)br.bits(5) + 1, ncode = (int)br.bits(4) + 4;
  if (nlen > 286 || ndist > 30) return YG_PNG_BAD_CODE_LENGTHS;
  uint16_t cl[19];
  for (int i = 0; i < 19; ++i) cl[clen_order(i)] = i < ncode ? (uint16_t)br.bits(3) : 0;
  if (huff_counts(t.hd, cl, 19) != 0) return YG_PNG_BAD_CODE_LENGTHS;   // must be complete
  for (int i = 0; i < (1 << CL_BITS); ++i) t.dist[i] = 0;
  huff_fill(t.hd, cl, t.dist, CL_BITS, 0, 1);
  for (int s = 0; s < MAX_LIT + MAX_DIST; ++s) t.lens[s] = 0;
  int i = 0;
  while (i < nlen + ndist) {
    br.refill();
    int len;
    const int sym = huff_decode(t.dist, CL_BITS, t.hd, br.buf, len);   // complete code of <= 7 bits: always found
    br.drop(len);
    if (sym < 16) {
      t.lens[i < nlen ? i : MAX_LIT + i - nlen] = (uint16_t)sym;
      ++i;
      continue;
    }
    int rep, val = 0;
    if (sym == 16) {
      if (i == 0) return YG_PNG_BAD_CODE_LENGTHS;
      val = t.lens[i - 1 < nlen ? i - 1 : MAX_LIT + i - 1 - nlen];
      rep = 3 + (int)br.bits(2);
    } else if (sym == 17) {
      rep = 3 + (int)br.bits(3);
    } else {
      rep = 11 + (int)br.bits(7);
    }
    if (i + rep > nlen + ndist) return YG_PNG_BAD_CODE_LENGTHS;
    for (; rep > 0; --rep, ++i) t.lens[i < nlen ? i : MAX_LIT + i - nlen] = (uint16_t)val;
  }
  if (t.lens[256] == 0) return YG_PNG_BAD_CODE_LENGTHS;   // no end-of-block code
  if (!code_ok(huff_counts(t.hl, t.lens, MAX_LIT), t.hl, false)) return YG_PNG_BAD_CODE_LENGTHS;
  if (!code_ok(huff_counts(t.hd, t.lens + MAX_LIT, MAX_DIST), t.hd, true)) return YG_PNG_BAD_CODE_LENGTHS;
  return YG_PNG_OK;
}

// queue entry: a literal byte (< 256), or MATCH | length << 16 | (distance - 1)
constexpr uint32_t Q_MATCH = 1u << 31;
PNG_HD int q_len(uint32_t e) { return (e & Q_MATCH) ? (int)((e >> 16) & 0x1ff) : 1; }
PNG_HD int q_dist(uint32_t e) { return (int)(e & 0xffff) + 1; }

// Decodes up to qcap symbols of a Huffman block into q.  `out` counts the bytes produced by the stream so far (the
// queued entries included); every distance is checked against it and against the window, every entry against the
// output capacity.  Sets eob at the end-of-block symbol.  Each symbol consumes at least one bit and each queued entry
// produces at least one byte below `cap`, so the decode ends on every input.
PNG_HD int decode_symbols(BitReader& br, const InflateTables& t, uint32_t* q, int qcap, long long& out, long long cap,
                          int window, int& n, bool& eob) {
  n = 0;
  eob = false;
  while (n < qcap) {
    br.refill();
    int len;
    const int sym = huff_decode(t.lit, LIT_BITS, t.hl, br.buf, len);
    br.drop(len);
    if (sym < 256) {
      if (out >= cap) return YG_PNG_OUTPUT_OVERFLOW;
      q[n++] = (uint32_t)sym;
      ++out;
      continue;
    }
    if (sym == 256) {
      eob = true;
      return YG_PNG_OK;
    }
    if (sym > 285) return YG_PNG_BAD_SYMBOL;
    const int li = sym - 257;
    br.refill();
    const int length = len_base(li) + (int)br.peek(len_extra(li));
    br.drop(len_extra(li));
    const int dsym = huff_decode(t.dist, DIST_BITS, t.hd, br.buf, len);
    if (dsym < 0 || dsym > 29) return YG_PNG_BAD_SYMBOL;
    br.drop(len);
    const int dist = dist_base(dsym) + (int)br.bits(dist_extra(dsym));
    if (dist > out || dist > window) return YG_PNG_BAD_DISTANCE;
    if (length > cap - out) return YG_PNG_OUTPUT_OVERFLOW;
    q[n++] = Q_MATCH | (uint32_t)length << 16 | (uint32_t)(dist - 1);
    out += length;
  }
  return YG_PNG_OK;
}

// ---- PNG scanline filters (bpp 1) ---------------------------------------------------------------------------------
// raw: the filtered byte; a: reconstructed left, b: up, c: upper-left (0 outside the image)
PNG_HD uint8_t unfilter_byte(int ft, uint32_t raw, uint32_t a, uint32_t b, uint32_t c) {
  uint32_t pred;
  if (ft == 1) {
    pred = a;
  } else if (ft == 2) {
    pred = b;
  } else if (ft == 3) {
    pred = (a + b) >> 1;
  } else if (ft == 4) {
    const int p = (int)a + (int)b - (int)c;
    const int pa = p > (int)a ? p - (int)a : (int)a - p;
    const int pb = p > (int)b ? p - (int)b : (int)b - p;
    const int pc = p > (int)c ? p - (int)c : (int)c - p;
    pred = (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
  } else {
    pred = 0;
  }
  return (uint8_t)(raw + pred);
}

}  // namespace png
}  // namespace yg
