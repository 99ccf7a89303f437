// PNG files -> decoded images and label maps on the device (the dataset feed: LoadImageFromFile / LoadAnnotations).
//
// Supported: bit depth 8, colour types 0 / 2 / 3 / 4 / 6, and bit depth 16 grey in the grey16 mode; no interlace (the
// caller read the IHDR and rejected the rest).
// Colour mode writes [3, h, w] uint8 BGR, what cv2.imdecode(buf, IMREAD_COLOR) returns transposed to CHW: grey
// replicated, palette expanded through PLTE (indices past its end read black, as libpng's zero-filled palette does),
// alpha dropped, tRNS / gAMA and every other ancillary chunk ignored.  Label mode (colour types 0 and 3) writes [1, h, w]
// uint8: the grey value or the palette index through a 256-entry lookup table.  Grey16 mode (bit depth 16, colour type 0
// only: Cityscapes' instanceIds maps) writes [1, h, w] int32, the big-endian samples as np.array(Image.open(f)) reads them.
//
//  * png_inflate_kernel  : one warp per file.  Lane 0 walks the chunks (order and lengths; ChunkWalk), the warp checks
//      the CRC of every critical chunk (per-lane CRCs merged with crc_combine) and gathers the IDAT payloads into one
//      contiguous zlib stream in the workspace.  Lane 0 then decodes symbols (64-bit bit buffer, canonical Huffman
//      tables with a 10-bit first-level lookup in shared memory, rebuilt per block) into a buffer of up to kTok tokens;
//      the warp writes the literals of 32 tokens at once and copies every match / stored run with all lanes, in token
//      order (out[p + i] = out[p - d + (i mod d)], so overlapping matches read only finished bytes).  Last, the
//      Adler-32 of the output, split over the lanes.
//  * png_unfilter_kernel : one block of 256 threads per file: thread t owns row r0 + t and reconstructs it tile by tile
//      (16 pixels), one tile behind the row above (Sub / Avg / Paeth read the byte bpp to the left and the row above:
//      a wavefront), writing each finished tile straight into the output layout.
//
// Everything that decides validity (the IHDR check, the chunk walk, inflate, unfilter, the pixel layout) is
// __host__ __device__, and ledb200_png_decode_host runs it on the CPU: a corrupt or hostile file gets the same status
// there as on the device.  No input makes a kernel read outside its file or write outside its workspace slot and its
// output: every length is checked before it is used.
#include <cstring>
#include <string>
#include <vector>

#include "kernels.h"
#include "png_common.cuh"

namespace ledb {
namespace {

#define HD __host__ __device__ inline

constexpr int kDecMax = 64;       // files per launch (descriptors in a __grid_constant__ block)
constexpr int kTok = 512;         // tokens per decode round
constexpr int kFastBits = 10;
constexpr int kTile = 16;         // pixels per unfilter step
constexpr int kUnfilterThreads = 256;

HD uint32_t be32(const uint8_t* p) {
  return (uint32_t)p[0] << 24 | (uint32_t)p[1] << 16 | (uint32_t)p[2] << 8 | (uint32_t)p[3];
}
HD int bytes_per_pixel(int ct, int mode) {
  return mode == LEDB200_PNG_GREY16 ? 2 : ct == 2 ? 3 : ct == 4 ? 2 : ct == 6 ? 4 : 1;
}
HD int bit_depth(int mode) { return mode == LEDB200_PNG_GREY16 ? 16 : 8; }

// ---- signature and IHDR against the descriptor ----------------------------------------------------------------------
HD int check_header(const uint8_t* f, int64_t size, int h, int w, int ct, int depth) {
  const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
  if (size < 33) return LEDB200_PNG_EHEADER;
  for (int k = 0; k < 8; ++k)
    if (f[k] != sig[k]) return LEDB200_PNG_EHEADER;
  const uint8_t* c = f + 8;
  if (be32(c) != 13 || be32(c + 4) != 0x49484452u) return LEDB200_PNG_EHEADER;   // "IHDR"
  if (be32(c + 8) != (uint32_t)w || be32(c + 12) != (uint32_t)h || c[16] != depth || c[17] != (uint8_t)ct || c[18] || c[19] ||
      c[20])
    return LEDB200_PNG_EHEADER;
  return LEDB200_PNG_OK;
}

// ---- chunk walk -----------------------------------------------------------------------------------------------------
enum { kChunkSkip = 0, kChunkIdat, kChunkPlte, kChunkEnd };
struct ChunkWalk {
  int64_t pos = 33;                 // after the signature and IHDR
  int plte = 0, idat = 0, idat_closed = 0;
};
struct Chunk {
  int kind;
  int critical;                     // its CRC is checked
  int64_t data, len;                // payload offset and length
};

HD bool is_letter(uint8_t c) { return (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z'); }

// The chunk at w.pos: bounds, name, order.  Advances w.pos past it.
HD int chunk_next(const uint8_t* f, int64_t size, int ct, ChunkWalk& w, Chunk& c) {
  if (size - w.pos < 12) return LEDB200_PNG_ECHUNK;                 // IEND missing or a header cut short
  const int64_t len = be32(f + w.pos);
  if (len > 0x7fffffff || len > size - w.pos - 12) return LEDB200_PNG_ECHUNK;
  const uint8_t* t = f + w.pos + 4;
  for (int k = 0; k < 4; ++k)
    if (!is_letter(t[k])) return LEDB200_PNG_ECHUNK;
  const uint32_t type = be32(t);
  c.data = w.pos + 8; c.len = len; c.kind = kChunkSkip;
  c.critical = !(t[0] & 0x20);
  w.pos += 12 + len;
  if (type == 0x49444154u) {                                         // IDAT: one unbroken run
    if (w.idat_closed) return LEDB200_PNG_ECHUNK;
    w.idat = 1;
    c.kind = kChunkIdat;
    return LEDB200_PNG_OK;
  }
  if (w.idat) w.idat_closed = 1;
  if (type == 0x504c5445u) {                                         // PLTE
    if (w.idat || w.plte) return LEDB200_PNG_ECHUNK;
    w.plte = 1;
    if (ct == 3) {
      if (len % 3 || len < 3 || len > 768) return LEDB200_PNG_EPLTE;
      c.kind = kChunkPlte;
    }
    return LEDB200_PNG_OK;                                           // a suggested palette of a truecolour / grey file
  }
  if (type == 0x49454e44u) {                                         // IEND
    if (len) return LEDB200_PNG_ECHUNK;
    if (!w.idat) return LEDB200_PNG_ECHUNK;
    if (ct == 3 && !w.plte) return LEDB200_PNG_EPLTE;
    c.kind = kChunkEnd;
    return LEDB200_PNG_OK;
  }
  if (type == 0x65584966u) return LEDB200_PNG_EUNSUPPORTED;          // eXIf: cv2 would rotate by its orientation
  if (c.critical) return LEDB200_PNG_ECHUNK;                        // a second IHDR or an unknown critical chunk
  return LEDB200_PNG_OK;
}

// ---- inflate (RFC 1950 / 1951) ---------------------------------------------------------------------------------------
// Canonical Huffman code: count / symbol in code order (puff.c's form) and a first-level table of kFastBits bits,
// entries len << 9 | sym, 0 where the code is longer.
struct Huff {
  uint16_t count[16];
  uint16_t symbol[288];
  uint16_t fast[1 << kFastBits];
};
struct Tables {
  Huff lit, dist, cl;
  uint8_t lens[320];
};

// zlib's rules (inftrees.c): an over-subscribed code is invalid; an incomplete one is valid only for literal / length
// and distance codes whose single code has length 1; a code without symbols builds and fails at its first use.
HD int huff_build(Huff& h, const uint8_t* len, int n, bool code_lengths) {
  for (int l = 0; l < 16; ++l) h.count[l] = 0;
  for (int s = 0; s < n; ++s) ++h.count[len[s]];
  h.count[0] = 0;
  for (int i = 0; i < (1 << kFastBits); ++i) h.fast[i] = 0;
  int max = 15;
  while (max > 0 && !h.count[max]) --max;
  if (max == 0) return LEDB200_PNG_OK;
  int left = 1;
  for (int l = 1; l < 16; ++l) {
    left = 2 * left - h.count[l];
    if (left < 0) return LEDB200_PNG_EDEFLATE;
  }
  if (left > 0 && (code_lengths || max != 1)) return LEDB200_PNG_EDEFLATE;
  uint16_t offs[16];
  offs[1] = 0;
  for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + h.count[l];
  for (int s = 0; s < n; ++s)
    if (len[s]) h.symbol[offs[len[s]]++] = (uint16_t)s;
  int code = 0, idx = 0;
  for (int l = 1; l <= kFastBits; ++l) {
    for (int k = 0; k < h.count[l]; ++k, ++code, ++idx) {
      int rev = 0;
      for (int b = 0; b < l; ++b) rev |= ((code >> b) & 1) << (l - 1 - b);
      for (int r = rev; r < (1 << kFastBits); r += 1 << l) h.fast[r] = (uint16_t)(l << 9 | h.symbol[idx]);
    }
    code <<= 1;
  }
  return LEDB200_PNG_OK;
}

enum { kTokLit = 0, kTokMatch = 1, kTokStored = 2 };
struct Tok {
  uint32_t a;                       // length (<= 65535) | kind << 16
  uint32_t b;                       // literal byte, distance, or source offset in the zlib stream
};
HD Tok make_tok(int kind, uint32_t len, uint32_t b) { return Tok{len | (uint32_t)kind << 16, b}; }

enum { kStZlib = 0, kStHeader, kStHuff, kStDone };
struct Inflate {
  const uint8_t* in;
  int64_t n, pos;                   // stream bytes, next byte to load
  uint64_t buf;
  int cnt;                          // bits in buf
  int64_t out, cap;                 // bytes produced, bytes expected
  int state, last, status;
  uint32_t adler;                   // the stream's Adler-32 trailer
};

HD void refill(Inflate& s) {
  while (s.cnt <= 56) {
    const uint64_t b = s.pos < s.n ? s.in[s.pos] : 0;
    ++s.pos;
    s.buf |= b << s.cnt;
    s.cnt += 8;
  }
}
HD uint32_t take(Inflate& s, int k) {
  const uint32_t v = (uint32_t)(s.buf & ((1ull << k) - 1));
  s.buf >>= k;
  s.cnt -= k;
  return v;
}
HD bool overrun(const Inflate& s) { return s.pos * 8 - s.cnt > s.n * 8; }

// one symbol of h (at least 15 bits buffered), -1 on an unused code
HD int decode(Inflate& s, const Huff& h) {
  const uint16_t e = h.fast[s.buf & ((1u << kFastBits) - 1)];
  if (e) { take(s, e >> 9); return e & 511; }
  int code = 0, first = 0, index = 0;
  for (int l = 1; l < 16; ++l) {
    code |= (int)((s.buf >> (l - 1)) & 1);
    const int count = h.count[l];
    if (code - count < first) { take(s, l); return h.symbol[index + (code - first)]; }
    index += count; first += count;
    first <<= 1; code <<= 1;
  }
  return -1;
}

HD void fixed_tables(Tables& t) {
  for (int s = 0; s < 288; ++s) t.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
  huff_build(t.lit, t.lens, 288, false);
  for (int s = 0; s < 32; ++s) t.lens[s] = 5;                       // codes 30 and 31 exist and are invalid
  huff_build(t.dist, t.lens, 32, false);
}

HD int dynamic_tables(Inflate& s, Tables& t) {
  const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
  refill(s);
  const int nlen = (int)take(s, 5) + 257, ndist = (int)take(s, 5) + 1, ncode = (int)take(s, 4) + 4;
  if (nlen > 286 || ndist > 30) return LEDB200_PNG_EDEFLATE;
  uint8_t cl[19];
  for (int k = 0; k < 19; ++k) cl[k] = 0;
  refill(s);
  for (int k = 0; k < ncode; ++k) cl[order[k]] = (uint8_t)take(s, 3);
  if (overrun(s)) return LEDB200_PNG_ETRUNC;
  if (huff_build(t.cl, cl, 19, true)) return LEDB200_PNG_EDEFLATE;
  for (int k = 0; k < nlen + ndist;) {
    refill(s);
    const int sym = decode(s, t.cl);
    if (sym < 0) return overrun(s) ? LEDB200_PNG_ETRUNC : LEDB200_PNG_EDEFLATE;
    if (sym < 16) { t.lens[k++] = (uint8_t)sym; continue; }
    int v = 0, rep;
    if (sym == 16) {
      if (k == 0) return LEDB200_PNG_EDEFLATE;
      v = t.lens[k - 1]; rep = 3 + (int)take(s, 2);
    } else if (sym == 17) {
      rep = 3 + (int)take(s, 3);
    } else {
      rep = 11 + (int)take(s, 7);
    }
    if (k + rep > nlen + ndist) return LEDB200_PNG_EDEFLATE;
    while (rep--) t.lens[k++] = (uint8_t)v;
  }
  if (overrun(s)) return LEDB200_PNG_ETRUNC;
  if (t.lens[256] == 0) return LEDB200_PNG_EDEFLATE;                  // no end-of-block code
  if (huff_build(t.lit, t.lens, nlen, false)) return LEDB200_PNG_EDEFLATE;
  if (huff_build(t.dist, t.lens + nlen, ndist, false)) return LEDB200_PNG_EDEFLATE;
  return LEDB200_PNG_OK;
}

HD void inflate_init(Inflate& s, const uint8_t* in, int64_t n, int64_t cap) {
  s.in = in; s.n = n; s.pos = 0; s.buf = 0; s.cnt = 0;
  s.out = 0; s.cap = cap; s.state = kStZlib; s.last = 0; s.status = LEDB200_PNG_OK; s.adler = 0;
}

HD int inflate_fail(Inflate& s, int status) {
  s.status = status;
  s.state = kStDone;
  return status;
}

// Decodes until `cap` tokens are buffered or the stream ends (state kStDone; status says how).  Every token stays
// inside [0, s.cap) of the output and inside the stream.  Returns the number of tokens.
HD int inflate_run(Inflate& s, Tables& t, Tok* toks, int cap) {
  int nt = 0;
  while (nt < cap && s.state != kStDone) {
    if (s.state == kStZlib) {
      if (s.n < 2) { inflate_fail(s, LEDB200_PNG_ETRUNC); break; }
      const int cmf = s.in[0], flg = s.in[1];
      if ((cmf & 15) != 8 || (cmf >> 4) > 7 || (cmf * 256 + flg) % 31 || (flg & 0x20)) {
        inflate_fail(s, LEDB200_PNG_EZLIB);
        break;
      }
      s.pos = 2;
      s.state = kStHeader;
      continue;
    }
    if (s.state == kStHeader) {
      if (s.last) {                                                  // the Adler-32 trailer, byte-aligned
        take(s, s.cnt & 7);
        refill(s);
        uint32_t a = 0;
        for (int k = 0; k < 4; ++k) a = a << 8 | take(s, 8);
        if (overrun(s)) { inflate_fail(s, LEDB200_PNG_ETRUNC); break; }
        if (s.pos - s.cnt / 8 != s.n) { inflate_fail(s, LEDB200_PNG_EZLIB); break; }     // data after the stream
        if (s.out != s.cap) { inflate_fail(s, LEDB200_PNG_ESIZE); break; }
        s.adler = a;
        s.state = kStDone;
        break;
      }
      refill(s);
      s.last = (int)take(s, 1);
      const int type = (int)take(s, 2);
      if (type == 0) {
        take(s, s.cnt & 7);
        const uint32_t len = take(s, 16), nlen = take(s, 16);
        if (overrun(s)) { inflate_fail(s, LEDB200_PNG_ETRUNC); break; }
        if (len != (~nlen & 0xffffu)) { inflate_fail(s, LEDB200_PNG_EDEFLATE); break; }
        const int64_t src = s.pos - s.cnt / 8;
        if ((int64_t)len > s.n - src) { inflate_fail(s, LEDB200_PNG_ETRUNC); break; }
        if ((int64_t)len > s.cap - s.out) { inflate_fail(s, LEDB200_PNG_ESIZE); break; }
        if (len) toks[nt++] = make_tok(kTokStored, len, (uint32_t)src);
        s.out += len;
        s.pos = src + len; s.buf = 0; s.cnt = 0;
      } else if (type == 1) {
        fixed_tables(t);
        s.state = kStHuff;
      } else if (type == 2) {
        const int st = dynamic_tables(s, t);
        if (st) { inflate_fail(s, st); break; }
        s.state = kStHuff;
      } else {
        inflate_fail(s, LEDB200_PNG_EDEFLATE);
        break;
      }
      continue;
    }
    // kStHuff: 57 buffered bits cover a length / distance pair (15 + 5 + 15 + 13)
    refill(s);
    const int sym = decode(s, t.lit);
    if (sym < 0) { inflate_fail(s, overrun(s) ? LEDB200_PNG_ETRUNC : LEDB200_PNG_EDEFLATE); break; }
    if (sym < 256) {
      if (s.out >= s.cap) { inflate_fail(s, LEDB200_PNG_ESIZE); break; }
      toks[nt++] = make_tok(kTokLit, 1, (uint32_t)sym);
      ++s.out;
    } else if (sym == 256) {
      s.state = kStHeader;
    } else {
      const int c = sym - 257;
      if (c >= 29) { inflate_fail(s, LEDB200_PNG_EDEFLATE); break; }
      int len;
      if (c < 8) len = c + 3;
      else if (c == 28) len = 258;
      else { const int eb = (c >> 2) - 1; len = ((4 + (c & 3)) << eb) + 3 + (int)take(s, eb); }
      const int dc = decode(s, t.dist);
      if (dc < 0 || dc >= 30) { inflate_fail(s, overrun(s) ? LEDB200_PNG_ETRUNC : LEDB200_PNG_EDEFLATE); break; }
      int64_t dist;
      if (dc < 4) dist = dc + 1;
      else { const int eb = (dc >> 1) - 1; dist = ((int64_t)(2 + (dc & 1)) << eb) + 1 + take(s, eb); }
      if (dist > s.out) { inflate_fail(s, LEDB200_PNG_EDEFLATE); break; }           // before the start of the stream
      if (len > s.cap - s.out) { inflate_fail(s, LEDB200_PNG_ESIZE); break; }
      toks[nt++] = make_tok(kTokMatch, (uint32_t)len, (uint32_t)dist);
      s.out += len;
    }
    if (overrun(s)) { inflate_fail(s, LEDB200_PNG_ETRUNC); break; }
  }
  return nt;
}

// ---- unfilter and output layout -------------------------------------------------------------------------------------
HD int paeth(int a, int b, int c) {
  const int p = a + b - c;
  const int pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
  return (pa <= pb && pa <= pc) ? a : pb <= pc ? b : c;
}

// Reconstructs bytes [j0, j1) of a row in place (cur: after the filter byte; prev: the reconstructed row above, or
// null on the first row).  Bytes before j0 and the row above must be final.
HD void unfilter_span(uint8_t* cur, const uint8_t* prev, int ft, int bpp, int64_t j0, int64_t j1) {
  for (int64_t j = j0; j < j1; ++j) {
    const int a = j >= bpp ? cur[j - bpp] : 0, b = prev ? prev[j] : 0, c = (prev && j >= bpp) ? prev[j - bpp] : 0;
    const int x = cur[j];
    const int v = ft == 1 ? x + a : ft == 2 ? x + b : ft == 3 ? x + ((a + b) >> 1) : ft == 4 ? x + paeth(a, b, c) : x;
    cur[j] = (uint8_t)v;
  }
}

// pixels [x0, x1) of reconstructed row y into the output: colour [3, h, w] BGR, label [1, h, w] through lut, grey16
// [1, h, w] int32
HD void emit_pixels(const uint8_t* d, int ct, int mode, const uint8_t* plte, const uint8_t* lut, uint8_t* out,
                    int64_t plane, int64_t y, int64_t w, int64_t x0, int64_t x1) {
  if (mode == LEDB200_PNG_GREY16) {
    int32_t* o = reinterpret_cast<int32_t*>(out) + y * w;
    for (int64_t x = x0; x < x1; ++x) o[x] = (int32_t)d[2 * x] << 8 | d[2 * x + 1];
    return;
  }
  uint8_t* o = out + y * w;
  for (int64_t x = x0; x < x1; ++x) {
    if (mode == LEDB200_PNG_LABEL) { o[x] = lut[d[x]]; continue; }
    int r, g, b;
    if (ct == 0) { r = g = b = d[x]; }
    else if (ct == 4) { r = g = b = d[2 * x]; }
    else if (ct == 3) { const uint8_t* p = plte + 3 * d[x]; r = p[0]; g = p[1]; b = p[2]; }
    else { const int64_t k = x * (ct == 2 ? 3 : 4); r = d[k]; g = d[k + 1]; b = d[k + 2]; }
    o[x] = (uint8_t)b; o[plane + x] = (uint8_t)g; o[2 * plane + x] = (uint8_t)r;
  }
}

// ---- device kernels -------------------------------------------------------------------------------------------------
struct DecFile {
  const uint8_t* data;
  int64_t size;
  uint8_t* out;
  uint8_t* zbuf;                    // workspace: the gathered IDAT payloads (<= size bytes)
  uint8_t* raw;                     // workspace: the inflated scanlines, h * (1 + w * bpp) bytes
  uint8_t* plte;                    // workspace: 768 bytes, zero past the file's palette
  int32_t h, w, ct, bpp;
};
struct DecArgs {
  DecFile f[kDecMax];
  uint8_t lut[256];
  int32_t* status;
  int32_t n, mode;
};

HD int64_t raw_bytes(const DecFile& f) { return (int64_t)f.h * (1 + (int64_t)f.w * f.bpp); }

// CRC-32 of p[0, n) by the warp: a contiguous segment per lane, merged pairwise in lane order
__device__ uint32_t warp_crc(const uint32_t* tab, const uint32_t* x2n, const uint8_t* p, int64_t n, int lane) {
  const int64_t per = (n + 31) / 32, a = min(n, lane * per), e = min(n, a + per);
  uint32_t c = ~crc_update(tab, 0xffffffffu, p + a, e - a);
  int64_t len = e - a;
  for (int s = 1; s < 32; s <<= 1) {
    const uint32_t c2 = __shfl_down_sync(0xffffffffu, c, s);
    const int64_t l2 = __shfl_down_sync(0xffffffffu, len, s);
    if ((lane & (2 * s - 1)) == 0) { c = crc_combine(c, c2, l2, x2n); len += l2; }
  }
  return __shfl_sync(0xffffffffu, c, 0);
}

// the warp writes tokens [0, nt) whose output starts at `base`
__device__ void apply_tokens(const Tok* toks, int nt, int64_t base, uint8_t* out, const uint8_t* zbuf, int lane) {
  for (int t0 = 0; t0 < nt; t0 += 32) {
    const int t = t0 + lane;
    const Tok k = t < nt ? toks[t] : Tok{0, 0};
    const int len = (int)(k.a & 0xffff), kind = (int)(k.a >> 16);
    int64_t incl = len;
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const int64_t p = base + incl - len;
    if (t < nt && kind == kTokLit) out[p] = (uint8_t)k.b;
    uint32_t todo = __ballot_sync(0xffffffffu, t < nt && kind != kTokLit);
    __syncwarp();
    while (todo) {
      const int j = __ffs(todo) - 1;
      todo &= todo - 1;
      const int lj = __shfl_sync(0xffffffffu, len, j), kj = __shfl_sync(0xffffffffu, kind, j);
      const uint32_t bj = __shfl_sync(0xffffffffu, k.b, j);
      const int64_t pj = __shfl_sync(0xffffffffu, p, j);
      if (kj == kTokMatch) {
        for (int i = lane; i < lj; i += 32) out[pj + i] = out[pj - bj + (uint32_t)i % bj];
      } else {
        for (int i = lane; i < lj; i += 32) out[pj + i] = zbuf[bj + i];
      }
      __syncwarp();
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
}

__global__ void __launch_bounds__(32) png_inflate_kernel(const __grid_constant__ DecArgs a) {
  __shared__ Tables T;
  __shared__ Tok toks[kTok];
  __shared__ uint32_t tab[256], x2n[32];
  const int lane = threadIdx.x;
  const DecFile& f = a.f[blockIdx.x];
  for (int i = lane; i < 256; i += 32) tab[i] = crc_table_entry((uint32_t)i);
  for (int i = lane; i < 768; i += 32) f.plte[i] = 0;
  if (lane == 0) crc_x2n_table(x2n);
  __syncwarp();
  int st = lane == 0 ? check_header(f.data, f.size, f.h, f.w, f.ct, bit_depth(a.mode)) : 0;
  st = __shfl_sync(0xffffffffu, st, 0);

  // chunks: lane 0 walks, the warp checks CRCs and gathers the IDAT payloads
  ChunkWalk w;
  int64_t zlen = 0;
  while (st == LEDB200_PNG_OK) {
    Chunk c{kChunkSkip, 0, 0, 0};
    if (lane == 0) st = chunk_next(f.data, f.size, f.ct, w, c);
    st = __shfl_sync(0xffffffffu, st, 0);
    if (st) break;
    const int kind = __shfl_sync(0xffffffffu, c.kind, 0), critical = __shfl_sync(0xffffffffu, c.critical, 0);
    const int64_t off = __shfl_sync(0xffffffffu, c.data, 0), len = __shfl_sync(0xffffffffu, c.len, 0);
    if (critical) {
      if (warp_crc(tab, x2n, f.data + off - 4, len + 4, lane) != be32(f.data + off + len)) { st = LEDB200_PNG_ECRC; break; }
      if (kind == kChunkIdat) {
        for (int64_t i = lane; i < len; i += 32) f.zbuf[zlen + i] = f.data[off + i];
        zlen += len;
      } else if (kind == kChunkPlte) {
        for (int64_t i = lane; i < len; i += 32) f.plte[i] = f.data[off + i];
      }
    }
    if (kind == kChunkEnd) break;
  }
  __syncwarp();

  // inflate: lane 0 decodes a round of tokens, the warp writes them
  const int64_t cap = raw_bytes(f);
  Inflate s;
  inflate_init(s, f.zbuf, zlen, cap);
  while (st == LEDB200_PNG_OK) {
    int nt = 0, done = 0, sst = 0;
    int64_t base = 0;
    if (lane == 0) {
      base = s.out;
      nt = inflate_run(s, T, toks, kTok);
      done = s.state == kStDone;
      sst = s.status;
    }
    nt = __shfl_sync(0xffffffffu, nt, 0);
    done = __shfl_sync(0xffffffffu, done, 0);
    base = __shfl_sync(0xffffffffu, base, 0);
    st = __shfl_sync(0xffffffffu, sst, 0);
    __syncwarp();
    apply_tokens(toks, nt, base, f.raw, f.zbuf, lane);
    __syncwarp();
    if (done) break;
  }

  if (st == LEDB200_PNG_OK) {                                        // Adler-32 of the output
    const int64_t per = (cap + 31) / 32, a0 = min(cap, lane * per), e0 = min(cap, a0 + per);
    uint64_t s1, s2;
    adler_sums(f.raw + a0, e0 - a0, s1, s2);
    s2 = adler_shift(s1, s2, cap - e0);
    for (int o = 16; o; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    const uint32_t want = __shfl_sync(0xffffffffu, s.adler, 0);
    if (adler_final(s1 % kAdlerMod, s2 % kAdlerMod, cap) != want) st = LEDB200_PNG_EADLER;
  }
  if (lane == 0) a.status[blockIdx.x] = st;
}

__global__ void __launch_bounds__(kUnfilterThreads) png_unfilter_kernel(const __grid_constant__ DecArgs a) {
  __shared__ uint8_t plte[768];
  __shared__ int bad;
  const DecFile& f = a.f[blockIdx.x];
  if (a.status[blockIdx.x] != LEDB200_PNG_OK) return;
  const int t = threadIdx.x;
  for (int i = t; i < 768; i += kUnfilterThreads) plte[i] = f.plte[i];
  if (t == 0) bad = 0;
  __syncthreads();
  const int64_t S = 1 + (int64_t)f.w * f.bpp, plane = (int64_t)f.h * f.w;
  const int tiles = (f.w + kTile - 1) / kTile;
  for (int64_t r0 = 0; r0 < f.h; r0 += kUnfilterThreads) {
    const int64_t r = r0 + t;
    uint8_t* row = f.raw + r * S;
    const int ft = r < f.h ? row[0] : 0;
    if (ft > 4) bad = 1;
    for (int step = 0; step < tiles + kUnfilterThreads - 1; ++step) {
      const int k = step - t;
      if (r < f.h && ft <= 4 && k >= 0 && k < tiles) {
        const int64_t x0 = (int64_t)k * kTile, x1 = min((int64_t)f.w, x0 + kTile);
        unfilter_span(row + 1, r ? row + 1 - S : nullptr, ft, f.bpp, x0 * f.bpp, x1 * f.bpp);
        emit_pixels(row + 1, f.ct, a.mode, plte, a.lut, f.out, plane, r, f.w, x0, x1);
      }
      __syncthreads();
    }
  }
  if (t == 0 && bad) a.status[blockIdx.x] = LEDB200_PNG_EFILTER;
}

// ---- host side ------------------------------------------------------------------------------------------------------
struct Slot { int64_t zbuf, raw, plte; };

int64_t align16(int64_t v) { return (v + 15) / 16 * 16; }

int check_files(const ledb200_png_file* files, int n, int mode, const char* who) {
  const std::string w(who);
  if (!files) return fail(LEDB200_EINVAL, w + ": null file descriptors");
  if (n < 1) return fail(LEDB200_EINVAL, w + ": at least one file");
  if (mode != LEDB200_PNG_COLOR && mode != LEDB200_PNG_LABEL && mode != LEDB200_PNG_GREY16)
    return fail(LEDB200_EINVAL, w + ": mode must be colour, label or grey16");
  for (int i = 0; i < n; ++i) {
    const ledb200_png_file& d = files[i];
    const std::string at = w + ": file " + std::to_string(i) + ": ";
    if (!d.data || !d.out) return fail(LEDB200_EINVAL, at + "null data or output");
    if (d.size < 33 || d.size > 0x7fffffff) return fail(LEDB200_EINVAL, at + "size must be in [33, 2^31)");
    if (d.h < 1 || d.w < 1 || (int64_t)d.h * d.w > (int64_t)1 << 30)
      return fail(LEDB200_EINVAL, at + "h and w must be at least 1 and h * w at most 2^30");
    if (d.color_type != 0 && d.color_type != 2 && d.color_type != 3 && d.color_type != 4 && d.color_type != 6)
      return fail(LEDB200_EINVAL, at + "colour type must be 0, 2, 3, 4 or 6");
    if (mode == LEDB200_PNG_LABEL && d.color_type != 0 && d.color_type != 3)
      return fail(LEDB200_EINVAL, at + "label maps must be grey or palette images");
    if (mode == LEDB200_PNG_GREY16 && d.color_type != 0) return fail(LEDB200_EINVAL, at + "grey16 files must be grey images");
  }
  return LEDB200_OK;
}

Slot slot_of(const ledb200_png_file& d, int mode, int64_t& at) {
  Slot s;
  s.zbuf = at; at += align16(d.size);
  s.raw = at; at += align16((int64_t)d.h * (1 + (int64_t)d.w * bytes_per_pixel(d.color_type, mode)));
  s.plte = at; at += 768;
  return s;
}

// the device pipeline on the CPU, for one file whose buffers are all host memory
int decode_host(DecFile f, int mode, const uint8_t* lut) {
  std::vector<uint32_t> tab(256), x2n(32);
  for (uint32_t i = 0; i < 256; ++i) tab[i] = crc_table_entry(i);
  crc_x2n_table(x2n.data());
  std::memset(f.plte, 0, 768);
  int st = check_header(f.data, f.size, f.h, f.w, f.ct, bit_depth(mode));
  ChunkWalk w;
  int64_t zlen = 0;
  while (st == LEDB200_PNG_OK) {
    Chunk c{kChunkSkip, 0, 0, 0};
    st = chunk_next(f.data, f.size, f.ct, w, c);
    if (st) break;
    if (c.critical) {
      if (~crc_update(tab.data(), 0xffffffffu, f.data + c.data - 4, c.len + 4) != be32(f.data + c.data + c.len)) {
        st = LEDB200_PNG_ECRC;
        break;
      }
      if (c.kind == kChunkIdat) { std::memcpy(f.zbuf + zlen, f.data + c.data, c.len); zlen += c.len; }
      else if (c.kind == kChunkPlte) std::memcpy(f.plte, f.data + c.data, c.len);
    }
    if (c.kind == kChunkEnd) break;
  }
  if (st) return st;
  const int64_t cap = raw_bytes(f);
  std::vector<Tok> toks(kTok);
  std::vector<Tables> T(1);
  Inflate s;
  inflate_init(s, f.zbuf, zlen, cap);
  while (s.state != kStDone) {
    int64_t p = s.out;
    const int nt = inflate_run(s, T[0], toks.data(), kTok);
    for (int i = 0; i < nt; ++i) {
      const int len = (int)(toks[i].a & 0xffff), kind = (int)(toks[i].a >> 16);
      const uint32_t b = toks[i].b;
      if (kind == kTokLit) f.raw[p] = (uint8_t)b;
      else if (kind == kTokMatch) for (int j = 0; j < len; ++j) f.raw[p + j] = f.raw[p + j - b];
      else std::memcpy(f.raw + p, f.zbuf + b, len);
      p += len;
    }
  }
  if (s.status) return s.status;
  uint64_t s1, s2;
  adler_sums(f.raw, cap, s1, s2);
  if (adler_final(s1, s2, cap) != s.adler) return LEDB200_PNG_EADLER;
  const int64_t S = 1 + (int64_t)f.w * f.bpp, plane = (int64_t)f.h * f.w;
  for (int64_t r = 0; r < f.h; ++r) {
    uint8_t* row = f.raw + r * S;
    if (row[0] > 4) return LEDB200_PNG_EFILTER;
    unfilter_span(row + 1, r ? row + 1 - S : nullptr, row[0], f.bpp, 0, S - 1);
    emit_pixels(row + 1, f.ct, mode, f.plte, lut, f.out, plane, r, f.w, 0, f.w);
  }
  return LEDB200_PNG_OK;
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int64_t ledb200_png_decode_mode_workspace_bytes(const ledb200_png_file* files, int32_t n, int32_t mode) {
  if (!files || n < 1) return fail(LEDB200_EINVAL, "png_decode_workspace_bytes: need at least one file descriptor");
  int64_t at = 0;
  for (int i = 0; i < n; ++i) slot_of(files[i], mode, at);
  return at;
}

int64_t ledb200_png_decode_workspace_bytes(const ledb200_png_file* files, int32_t n) {
  return ledb200_png_decode_mode_workspace_bytes(files, n, LEDB200_PNG_COLOR);
}

int ledb200_png_decode(const ledb200_png_file* files, int32_t n, int32_t mode, const uint8_t* lut, void* workspace,
                       int32_t* status, void* stream) {
  if (int rc = check_files(files, n, mode, "png_decode")) return rc;
  if (!workspace || !status) return fail(LEDB200_EINVAL, "png_decode: null workspace or status");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  int64_t at = 0;
  for (int i0 = 0; i0 < n; i0 += kDecMax) {
    DecArgs a;
    a.n = n - i0 < kDecMax ? n - i0 : kDecMax;
    a.mode = mode;
    a.status = status + i0;
    for (int k = 0; k < 256; ++k) a.lut[k] = lut ? lut[k] : (uint8_t)k;
    for (int i = 0; i < a.n; ++i) {
      const ledb200_png_file& d = files[i0 + i];
      const Slot s = slot_of(d, mode, at);
      DecFile& f = a.f[i];
      f.data = d.data; f.size = d.size; f.out = d.out;
      f.zbuf = ws + s.zbuf; f.raw = ws + s.raw; f.plte = ws + s.plte;
      f.h = d.h; f.w = d.w; f.ct = d.color_type; f.bpp = bytes_per_pixel(d.color_type, mode);
    }
    png_inflate_kernel<<<a.n, 32, 0, st>>>(a);
    LEDB_LAUNCH_OK("png_inflate_kernel");
    png_unfilter_kernel<<<a.n, kUnfilterThreads, 0, st>>>(a);
    LEDB_LAUNCH_OK("png_unfilter_kernel");
  }
  return LEDB200_OK;
}

int ledb200_png_decode_host(const ledb200_png_file* files, int32_t n, int32_t mode, const uint8_t* lut, int32_t* status) {
  if (int rc = check_files(files, n, mode, "png_decode_host")) return rc;
  if (!status) return fail(LEDB200_EINVAL, "png_decode_host: null status");
  uint8_t ident[256];
  for (int k = 0; k < 256; ++k) ident[k] = (uint8_t)k;
  for (int i = 0; i < n; ++i) {
    const ledb200_png_file& d = files[i];
    int64_t at = 0;
    const Slot s = slot_of(d, mode, at);
    std::vector<uint8_t> ws((size_t)at);
    DecFile f;
    f.data = d.data; f.size = d.size; f.out = d.out;
    f.zbuf = ws.data() + s.zbuf; f.raw = ws.data() + s.raw; f.plte = ws.data() + s.plte;
    f.h = d.h; f.w = d.w; f.ct = d.color_type; f.bpp = bytes_per_pixel(d.color_type, mode);
    status[i] = decode_host(f, mode, lut ? lut : ident);
  }
  return LEDB200_OK;
}

}  // extern "C"
