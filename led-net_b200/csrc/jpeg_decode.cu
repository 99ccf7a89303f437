// Baseline JPEG files -> decoded images on the device (the dataset feed: LoadImageFromFile on JPEG datasets).
//
// Output: [3, h, w] uint8 BGR, bit-identical to cv2.imdecode(buf, IMREAD_COLOR) transposed to CHW (libjpeg-turbo with
// JDCT_ISLOW, fancy upsampling, JCS_EXT_BGR).  Supported: SOF0 / SOF1, 8-bit, Huffman, one interleaved scan with every
// component; grey, or YCbCr with luma sampling {1, 2} x {1, 2} and chroma 1 x 1; any restart interval.
//
//  * jpeg_header_kernel  : one warp per file; lane 0 walks the markers (parse_header) and builds the Huffman tables
//      (jdhuff's validity rules, a 9-bit first-level lookup) and the MCU layout.
//  * jpeg_scan_kernel    : one block per file.  Finds the end of the entropy-coded segment and every RSTn (a flag per
//      byte, tile by tile), checks the restart numbers, and removes the FF 00 stuffing and the markers with a block
//      prefix sum: one contiguous, byte-aligned bit stream per restart interval.  Zeroes the coefficients.
//  * jpeg_huffman_kernel : one block per file: self-synchronising Huffman decoding (Weissenberger and Schmidt, ICPP
//      2018).  Every interval is cut into subsequences of kChunkBits bits; thread t owns a contiguous run of them.
//      A decoder state at a symbol boundary is (bit position, block within the MCU, zig-zag index).  Each thread
//      decodes its run from a guessed entry (its first subsequence's start, block 0, DC), recording every
//      subsequence's exit state (the first symbol boundary past its end) and completed blocks; then, round after
//      round, a thread whose predecessor's exit differs from its entry re-decodes from it until its states stop
//      changing.  Every decode is bounded by its interval, so the rounds end on any input (at worst one per thread).
//      A block scan of the block counts gives each subsequence's output block; a last pass decodes each once more
//      from its synchronised entry and writes int16 coefficients (libjpeg's JCOEF).  Only this pass reports errors.
//      DC values are then a segmented prefix sum (per component, reset at every interval) of the differences.
//  * jpeg_idct_kernel    : 8 threads per block: jidctint.c's jpeg_idct_islow in the 16-bit lanes of libjpeg-turbo's
//      SIMD kernels (see the IDCT section), one uint8 plane per component.
//  * jpeg_color_kernel   : a thread per pixel: jdsample.c's fancy upsampling (h2v1, h1v2, h2v2; box for components
//      at most 2 samples wide, as jinit_upsampler does) and jdcolor.c's YCbCr -> RGB, stored as BGR planes.
//
// Everything that decides validity is __host__ __device__, and ledb200_jpeg_decode_host runs it on the CPU (the sync
// rounds serially over the same 1024 "threads"): a corrupt or hostile file gets the same status there.  No input makes
// a kernel read outside its file or write outside its workspace slot and its output: every length is checked first.
#include <cstring>
#include <string>
#include <vector>

#include "kernels.h"

namespace ledb {
namespace {

#define HD __host__ __device__ inline

constexpr int kDecMax = 64;           // files per launch (descriptors in a __grid_constant__ block)
constexpr int kThreads = 1024;        // threads of the per-file blocks (scan, Huffman)
constexpr int kChunkBits = 1024;      // subsequence length
constexpr int kLook = 9;              // first-level Huffman lookup bits
constexpr int64_t kMaxSize = 1 << 28; // file bytes (bit positions stay in int32)

#define LEDB_NATURAL_ORDER                                                                                  \
  {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,   \
    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,   \
    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63}
__constant__ uint8_t kNaturalDev[64] = LEDB_NATURAL_ORDER;           // zig-zag index -> natural (row-major) index
#ifndef __CUDA_ARCH__
const uint8_t kNaturalHost[64] = LEDB_NATURAL_ORDER;
#endif
HD int natural(int k) {
#ifdef __CUDA_ARCH__
  return kNaturalDev[k];
#else
  return kNaturalHost[k];
#endif
}

struct HuffTab {
  uint16_t look[1 << kLook];          // len << 8 | symbol, 0 when the code is longer than kLook
  int32_t maxcode[18];                // largest code of each length, -1 if none (jdhuff's d_derived_tbl)
  int32_t valoff[18];
  uint8_t val[256];
};

struct Hdr {
  int32_t status;
  int32_t nc, h0, v0;                 // components; luma sampling (1 x 1 for grey)
  int32_t mcux, mcuy, nmcu, bpm, ri;  // MCUs per row / column / total, blocks per MCU, restart interval (0 = none)
  int32_t scan0;                      // first byte of the entropy-coded segment
  int32_t blk_comp[6];                // component of each block of an MCU
  int32_t dc[3], ac[3];               // Huffman table of each component (DC 0..3, AC 4..7)
  uint16_t q[3][64];                  // quantisation table of each component, natural order
  HuffTab tabs[8];
  int32_t nint, nchunks;              // filled by the scan stage
};

struct Raw {                          // the tables as the markers define them
  uint16_t q[4][64];
  uint8_t bits[8][17];
  uint8_t val[8][256];
  uint8_t qdef[4], hdef[8];
};

HD int be16(const uint8_t* p) { return p[0] << 8 | p[1]; }

// ---- tables ----------------------------------------------------------------------------------------------------------
// jdhuff.c's jpeg_make_d_derived_tbl: canonical codes, none all ones (code < 2^len after every length), DC symbols <= 15
HD int build_tab(HuffTab& t, const uint8_t* bits, const uint8_t* val, bool dc) {
  int code = 0, p = 0;
  for (int l = 1; l <= 16; ++l) {
    if (bits[l]) {
      t.valoff[l] = p - code;
      p += bits[l];
      code += bits[l];
      t.maxcode[l] = code - 1;
    } else {
      t.maxcode[l] = -1;
    }
    if (code >= (1 << l)) return LEDB200_JPEG_ETABLE;
    code <<= 1;
  }
  t.maxcode[0] = -1;
  t.maxcode[17] = 0x7fffffff;
  if (dc)
    for (int i = 0; i < p; ++i)
      if (val[i] > 15) return LEDB200_JPEG_ETABLE;
  for (int i = 0; i < 256; ++i) t.val[i] = i < p ? val[i] : 0;
  for (int i = 0; i < (1 << kLook); ++i) t.look[i] = 0;
  code = 0; p = 0;
  for (int l = 1; l <= kLook; ++l, code <<= 1)
    for (int k = 0; k < bits[l]; ++k, ++p, ++code)
      for (int j = 0; j < (1 << (kLook - l)); ++j) t.look[(code << (kLook - l)) | j] = (uint16_t)(l << 8 | val[p]);
  return LEDB200_JPEG_OK;
}

// ---- markers ---------------------------------------------------------------------------------------------------------
// the Exif orientation of an APP1 payload, 0 when there is none (or the TIFF structure does not reach it)
HD int exif_orientation(const uint8_t* s, int n) {
  const uint8_t id[6] = {'E', 'x', 'i', 'f', 0, 0};
  if (n < 14) return 0;
  for (int k = 0; k < 6; ++k)
    if (s[k] != id[k]) return 0;
  const uint8_t* t = s + 6;
  const int64_t tn = n - 6;
  bool le;
  if (t[0] == 'I' && t[1] == 'I') le = true;
  else if (t[0] == 'M' && t[1] == 'M') le = false;
  else return 0;
  auto u16 = [&](int64_t o) { return le ? (t[o] | t[o + 1] << 8) : (t[o] << 8 | t[o + 1]); };
  auto u32 = [&](int64_t o) { return (int64_t)(le ? (uint32_t)(u16(o) | u16(o + 2) << 16) : (uint32_t)(u16(o) << 16 | u16(o + 2))); };
  if (u16(2) != 42) return 0;
  const int64_t ifd = u32(4);
  if (ifd > tn - 2) return 0;
  const int cnt = u16(ifd);
  for (int i = 0; i < cnt; ++i) {
    const int64_t e = ifd + 2 + 12 * (int64_t)i;
    if (e + 12 > tn) break;
    if (u16(e) == 0x0112) return u16(e + 8);
  }
  return 0;
}

// Walks SOI .. SOS: tables, frame, scan header against the descriptor (h, w, nc); fills H up to scan0.
HD int parse_header(const uint8_t* f, int64_t size, int h, int w, int nc, Raw& R, Hdr& H) {
  if (size < 4 || f[0] != 0xFF || f[1] != 0xD8) return LEDB200_JPEG_EHEADER;
  for (int i = 0; i < 4; ++i) R.qdef[i] = 0;
  for (int i = 0; i < 8; ++i) R.hdef[i] = 0;
  int64_t p = 2;
  bool sof = false, jfif = false, adobe = false;
  int transform = 0, orient = 0, ri = 0, nf = 0;
  int id[3] = {0, 0, 0}, hs[3] = {1, 1, 1}, vs[3] = {1, 1, 1}, tq[3] = {0, 0, 0};
  for (;;) {
    if (p >= size || f[p] != 0xFF) return LEDB200_JPEG_ESEGMENT;
    while (p < size && f[p] == 0xFF) ++p;                            // fill bytes
    if (p >= size) return LEDB200_JPEG_ESEGMENT;
    const int m = f[p++];
    if (size - p < 2) return LEDB200_JPEG_ESEGMENT;
    const int len = be16(f + p);
    if (len < 2 || len > size - p) return LEDB200_JPEG_ESEGMENT;
    const uint8_t* s = f + p + 2;
    int n = len - 2;
    p += len;
    if (m == 0xC0 || m == 0xC1) {                                     // SOF0 / SOF1
      if (sof) return LEDB200_JPEG_ESEGMENT;
      sof = true;
      if (n < 6) return LEDB200_JPEG_ESEGMENT;
      nf = s[5];
      if (n != 6 + 3 * nf) return LEDB200_JPEG_ESEGMENT;
      if (s[0] != 8 || be16(s + 1) == 0 || (nf != 1 && nf != 3)) return LEDB200_JPEG_EUNSUPPORTED;
      if (be16(s + 3) == 0) return LEDB200_JPEG_ESEGMENT;
      for (int c = 0; c < nf; ++c) {
        id[c] = s[6 + 3 * c];
        hs[c] = s[7 + 3 * c] >> 4;
        vs[c] = s[7 + 3 * c] & 15;
        tq[c] = s[8 + 3 * c];
        if (hs[c] < 1 || hs[c] > 4 || vs[c] < 1 || vs[c] > 4) return LEDB200_JPEG_ESEGMENT;
        if (tq[c] > 3) return LEDB200_JPEG_ETABLE;
      }
      if (nf == 3 && (hs[0] > 2 || vs[0] > 2 || hs[1] != 1 || vs[1] != 1 || hs[2] != 1 || vs[2] != 1))
        return LEDB200_JPEG_EUNSUPPORTED;
      if (be16(s + 1) != h || be16(s + 3) != w || nf != nc) return LEDB200_JPEG_EHEADER;
    } else if (m == 0xC4) {                                           // DHT
      while (n > 0) {
        if (n < 17) return LEDB200_JPEG_ETABLE;
        const int tc = s[0] >> 4, th = s[0] & 15;
        if (tc > 1 || th > 3) return LEDB200_JPEG_ETABLE;
        int total = 0;
        for (int l = 1; l <= 16; ++l) total += s[l];
        if (total > 256 || total > n - 17) return LEDB200_JPEG_ETABLE;
        const int k = tc * 4 + th;
        R.bits[k][0] = 0;
        for (int l = 1; l <= 16; ++l) R.bits[k][l] = s[l];
        for (int i = 0; i < total; ++i) R.val[k][i] = s[17 + i];
        R.hdef[k] = 1;
        s += 17 + total;
        n -= 17 + total;
      }
    } else if (m == 0xDB) {                                           // DQT
      while (n > 0) {
        const int pq = s[0] >> 4, t = s[0] & 15;
        if (pq > 1 || t > 3) return LEDB200_JPEG_ETABLE;
        if (n < 1 + 64 * (pq + 1)) return LEDB200_JPEG_ETABLE;
        for (int k = 0; k < 64; ++k) R.q[t][natural(k)] = (uint16_t)(pq ? be16(s + 1 + 2 * k) : s[1 + k]);
        R.qdef[t] = 1;
        s += 1 + 64 * (pq + 1);
        n -= 1 + 64 * (pq + 1);
      }
    } else if (m == 0xDD) {                                           // DRI
      if (n != 2) return LEDB200_JPEG_ESEGMENT;
      ri = be16(s);
    } else if (m == 0xE0) {
      if (n >= 14 && s[0] == 'J' && s[1] == 'F' && s[2] == 'I' && s[3] == 'F' && s[4] == 0) jfif = true;
    } else if (m == 0xE1) {
      if (!orient) orient = exif_orientation(s, n);
    } else if (m == 0xEE) {
      if (n >= 12 && s[0] == 'A' && s[1] == 'd' && s[2] == 'o' && s[3] == 'b' && s[4] == 'e') {
        adobe = true;
        transform = s[11];
      }
    } else if ((m >= 0xE2 && m <= 0xEF) || m == 0xFE) {             // other APPn, COM
    } else if (m == 0xDA) {                                           // SOS
      if (!sof) return LEDB200_JPEG_ESEGMENT;
      const int ns = n >= 1 ? s[0] : 0;
      if (n < 1 || n != 4 + 2 * ns) return LEDB200_JPEG_ESEGMENT;
      if (ns != nf) return LEDB200_JPEG_EUNSUPPORTED;                 // a non-interleaved (multi-scan) file
      int td[3], ta[3];
      for (int c = 0; c < ns; ++c) {
        if (s[1 + 2 * c] != id[c]) return LEDB200_JPEG_EUNSUPPORTED;
        td[c] = s[2 + 2 * c] >> 4;
        ta[c] = s[2 + 2 * c] & 15;
        if (td[c] > 3 || ta[c] > 3) return LEDB200_JPEG_ETABLE;
      }
      const uint8_t* e = s + 1 + 2 * ns;
      if (e[0] != 0 || e[1] != 63 || e[2] != 0) return LEDB200_JPEG_EUNSUPPORTED;
      if (nf == 3 && (jfif ? false : adobe ? transform == 0 : (id[0] == 'R' && id[1] == 'G' && id[2] == 'B')))
        return LEDB200_JPEG_EUNSUPPORTED;                             // RGB colour space
      if (orient >= 2 && orient <= 8) return LEDB200_JPEG_EUNSUPPORTED;   // cv2 would rotate
      for (int c = 0; c < nf; ++c) {
        if (!R.qdef[tq[c]] || !R.hdef[td[c]] || !R.hdef[4 + ta[c]]) return LEDB200_JPEG_ETABLE;
        for (int k = 0; k < 64; ++k) H.q[c][k] = R.q[tq[c]][k];
        H.dc[c] = td[c];
        H.ac[c] = 4 + ta[c];
      }
      for (int k = 0; k < 8; ++k) {
        bool used = false;
        for (int c = 0; c < nf; ++c) used |= H.dc[c] == k || H.ac[c] == k;
        if (used && build_tab(H.tabs[k], R.bits[k], R.val[k], k < 4)) return LEDB200_JPEG_ETABLE;
      }
      H.nc = nf;
      H.h0 = nf == 3 ? hs[0] : 1;                                     // one component: non-interleaved, 1 x 1 MCUs
      H.v0 = nf == 3 ? vs[0] : 1;
      H.mcux = (w + 8 * H.h0 - 1) / (8 * H.h0);
      H.mcuy = (h + 8 * H.v0 - 1) / (8 * H.v0);
      H.nmcu = H.mcux * H.mcuy;
      H.bpm = H.h0 * H.v0 + (nf == 3 ? 2 : 0);
      for (int b = 0; b < 6; ++b) H.blk_comp[b] = b < H.h0 * H.v0 ? 0 : b - H.h0 * H.v0 + 1;
      H.ri = ri;
      H.scan0 = (int32_t)p;
      return LEDB200_JPEG_OK;
    } else if ((m >= 0xC2 && m <= 0xCF) && m != 0xC4 && m != 0xC8) {  // progressive, lossless, hierarchical, arithmetic
      return LEDB200_JPEG_EUNSUPPORTED;
    } else {                                                          // SOI, EOI, RSTn, DNL, JPG, reserved
      return LEDB200_JPEG_ESEGMENT;
    }
  }
}

// ---- entropy-coded segment -------------------------------------------------------------------------------------------
// Byte i of [scan0, size) ends the scan when it starts a marker other than RSTn (FF then not 00 / FF / D0..D7)
HD bool is_end(const uint8_t* d, int64_t i, int64_t size) {
  if (d[i] != 0xFF || i + 1 >= size) return false;
  const int v = d[i + 1];
  return v != 0x00 && v != 0xFF && (v < 0xD0 || v > 0xD7);
}
// Inside [scan0, end): byte i is data (keep), the FF of an RSTn (rst), or stuffing / fill / a marker's second byte.
HD void classify(const uint8_t* d, int64_t i, int64_t scan0, bool& keep, bool& rst) {
  const int v = d[i];
  rst = false;
  if (v == 0xFF) {
    const int nx = d[i + 1];                                           // i + 1 <= end < size
    keep = nx == 0x00;
    rst = nx >= 0xD0 && nx <= 0xD7;
    return;
  }
  keep = !(i > scan0 && d[i - 1] == 0xFF && (v == 0x00 || (v >= 0xD0 && v <= 0xD7)));
}

HD int expected_intervals(const Hdr& H) { return H.ri ? (H.nmcu + H.ri - 1) / H.ri : 1; }

// ---- Huffman decoding ------------------------------------------------------------------------------------------------
struct Reader {                        // MSB-first bits of cs[0, end) (zeros past it)
  const uint8_t* p;
  int32_t end, byte, cnt;
  uint64_t buf;
  HD void init(const uint8_t* cs, int32_t bit, int32_t endbyte) {
    p = cs; end = endbyte; byte = bit >> 3; cnt = 0; buf = 0;
    refill();
    skip(bit & 7);
  }
  HD void refill() {
    while (cnt <= 56) {
      const uint64_t b = byte < end ? p[byte] : 0;
      ++byte;
      buf |= b << (56 - cnt);
      cnt += 8;
    }
  }
  HD int32_t pos() const { return byte * 8 - cnt; }
  HD void skip(int k) { buf <<= k; cnt -= k; }
  HD uint32_t get(int k) {
    if (!k) return 0;
    const uint32_t v = (uint32_t)(buf >> (64 - k));
    skip(k);
    return v;
  }
};

// one symbol, -1 on a code no table entry has (jdhuff's "l > 16")
HD int huff_decode(Reader& r, const HuffTab& t) {
  const uint16_t e = t.look[r.buf >> (64 - kLook)];
  if (e) { r.skip(e >> 8); return e & 255; }
  for (int l = kLook + 1; l <= 16; ++l) {
    const int32_t code = (int32_t)(r.buf >> (64 - l));
    if (code <= t.maxcode[l]) { r.skip(l); return t.val[t.valoff[l] + code]; }
  }
  return -1;
}

HD int extend(uint32_t v, int s) { return s && v < (1u << (s - 1)) ? (int)v - (1 << s) + 1 : (int)v; }

// Decodes from state (pos, st = block << 8 | zig-zag index) while pos < cend, inside the interval ending at bit iend.
// kWrite: stops after `limit` completed blocks too and writes the coefficients (DC differences) from `coef` on.
// Returns a status; (pos, st) is the exit state, nblk the completed blocks.
template <bool kWrite>
HD int run_chunk(const Hdr& H, const HuffTab* T, const uint8_t* cs, int32_t cend, int32_t iend, int32_t& pos,
                 int32_t& st, int32_t& nblk, int32_t limit, int16_t* coef) {
  Reader r;
  r.init(cs, pos, (iend + 7) >> 3);
  int blk = st >> 8, zz = st & 255;
  nblk = 0;
  int status = LEDB200_JPEG_OK;
  while (r.pos() < cend && !(kWrite && nblk >= limit)) {
    r.refill();
    const int c = H.blk_comp[blk];
    int16_t* b = kWrite ? coef + (int64_t)nblk * 64 : nullptr;
    bool done = false;
    if (zz == 0) {
      const int s = huff_decode(r, T[H.dc[c]]);
      if (s < 0) { status = LEDB200_JPEG_EHUFF; break; }
      const int v = extend(r.get(s), s);
      if (kWrite) b[0] = (int16_t)v;
      zz = 1;
    } else {
      const int sym = huff_decode(r, T[H.ac[c]]);
      if (sym < 0) { status = LEDB200_JPEG_EHUFF; break; }
      const int run = sym >> 4, s = sym & 15;
      if (s) {
        zz += run;
        if (zz > 63) { status = LEDB200_JPEG_EZZ; break; }
        const int v = extend(r.get(s), s);
        if (kWrite) b[natural(zz)] = (int16_t)v;
        done = ++zz == 64;
      } else if (run == 15) {
        zz += 16;
        if (zz > 64) { status = LEDB200_JPEG_EZZ; break; }
        done = zz == 64;
      } else {
        done = true;                                                   // EOB
      }
    }
    if (r.pos() > iend) { status = LEDB200_JPEG_ETRUNC; break; }
    if (done) {
      ++nblk;
      zz = 0;
      blk = blk + 1 == H.bpm ? 0 : blk + 1;
    }
  }
  pos = r.pos();
  st = blk << 8 | zz;
  return status;
}

// Per-file views of the workspace of the Huffman stage
struct Chunks {
  const int32_t* ivl_bit;             // [nint + 1] first bit of each interval, then the stream's end
  const int32_t* ivl_chunk0;          // [nint + 1] first subsequence of each interval, then nchunks
  int32_t *ent_pos, *ent_st, *ex_pos, *ex_st, *nblk, *pref;   // [nchunks] each
};

struct ChunkGeo { int k; int32_t c0, c1, iend; bool first, last; };

HD ChunkGeo chunk_geo(const Chunks& X, int nint, int c) {
  int lo = 0, hi = nint;                                              // last k with ivl_chunk0[k] <= c
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (X.ivl_chunk0[mid] <= c) lo = mid; else hi = mid;
  }
  ChunkGeo g;
  g.k = lo;
  const int j = c - X.ivl_chunk0[lo];
  g.c0 = X.ivl_bit[lo] + j * kChunkBits;
  g.iend = X.ivl_bit[lo + 1];
  g.c1 = g.c0 + kChunkBits < g.iend ? g.c0 + kChunkBits : g.iend;
  g.first = j == 0;
  g.last = c + 1 == X.ivl_chunk0[lo + 1];
  return g;
}

// Speculative decodes of subsequences [a, b) from entry (pos, st) of a, each next entry the exit before it.  early:
// stop at the first subsequence (after a) whose entry is unchanged, since everything after it is too.
HD void sync_run(const Hdr& H, const HuffTab* T, const uint8_t* cs, const Chunks& X, int a, int b, int32_t pos,
                 int32_t st, bool early) {
  for (int c = a; c < b; ++c) {
    const ChunkGeo g = chunk_geo(X, H.nint, c);
    if (c > a) {
      if (g.first || X.ex_pos[c - 1] < 0) { pos = g.c0; st = 0; }
      else { pos = X.ex_pos[c - 1]; st = X.ex_st[c - 1]; }
      if (early && pos == X.ent_pos[c] && st == X.ent_st[c]) return;
    }
    X.ent_pos[c] = pos;
    X.ent_st[c] = st;
    int32_t p = pos, s = st, nb = 0;
    const int e = run_chunk<false>(H, T, cs, g.c1, g.iend, p, s, nb, 0, nullptr);
    X.ex_pos[c] = e ? -1 : p;
    X.ex_st[c] = s;
    X.nblk[c] = nb;
  }
}

// the entry of subsequence a as its predecessor's exit gives it (the interval's start for a first one)
HD void entry_of(const Hdr& H, const Chunks& X, int a, int32_t& pos, int32_t& st) {
  const ChunkGeo g = chunk_geo(X, H.nint, a);
  if (g.first || X.ex_pos[a - 1] < 0) { pos = g.c0; st = 0; }
  else { pos = X.ex_pos[a - 1]; st = X.ex_st[a - 1]; }
}

// interval k's blocks: [k * ri * bpm, + blocks)
HD int32_t interval_blocks(const Hdr& H, int k) {
  if (!H.ri) return H.nmcu * H.bpm;
  const int32_t m0 = k * H.ri, m1 = m0 + H.ri < H.nmcu ? m0 + H.ri : H.nmcu;
  return (m1 - m0) * H.bpm;
}

// The synchronised pass over subsequence c: writes its coefficients, returns its status (ETRUNC when the interval's
// last subsequence ends before the interval's blocks do).  pref: completed blocks before c (exclusive scan).
HD int final_chunk(const Hdr& H, const HuffTab* T, const uint8_t* cs, const Chunks& X, int c, int16_t* coef) {
  const ChunkGeo g = chunk_geo(X, H.nint, c);
  const int32_t rel = X.pref[c] - X.pref[X.ivl_chunk0[g.k]], target = interval_blocks(H, g.k);
  if (rel >= target) return LEDB200_JPEG_OK;                         // data after the interval's last MCU
  int32_t pos = X.ent_pos[c], st = X.ent_st[c], nb = 0;
  const int64_t blk0 = (int64_t)g.k * H.ri * H.bpm + rel;
  const int e = run_chunk<true>(H, T, cs, g.c1, g.iend, pos, st, nb, target - rel, coef + blk0 * 64);
  if (e) return e;
  if (g.last && nb < target - rel) return LEDB200_JPEG_ETRUNC;
  return LEDB200_JPEG_OK;
}

// DC differences -> values over MCUs [m0, m1): per component, reset at each interval's first MCU (wrapping int16 sums,
// libjpeg's (JCOEF) of its int predictor).  apply = false: only the local (reset seen, sums) of the range.
HD void dc_range(const Hdr& H, int16_t* coef, int32_t m0, int32_t m1, bool apply, bool& reset, uint16_t* sum) {
  for (int32_t m = m0; m < m1; ++m) {
    if (m == 0 || (H.ri && m % H.ri == 0)) { reset = true; sum[0] = sum[1] = sum[2] = 0; }
    for (int b = 0; b < H.bpm; ++b) {
      int16_t* d = coef + ((int64_t)m * H.bpm + b) * 64;
      const int c = H.blk_comp[b];
      sum[c] = (uint16_t)(sum[c] + (uint16_t)d[0]);
      if (apply) d[0] = (int16_t)sum[c];
    }
  }
}

// ---- IDCT (jidctint.c's jpeg_idct_islow, as libjpeg-turbo's SIMD kernels compute it) -------------------------------
// cv2's libjpeg-turbo runs the SIMD islow IDCT (jidctint-sse2 / -avx2 / -neon).  It is jidctint.c's arithmetic on
// 16-bit lanes: dequantisation keeps the low 16 bits (pmullw), the sums in0 +- in4 and tmp0 + tmp2 / tmp1 + tmp3 are
// 16-bit, products and the rest are 32-bit (pmaddwd), pass 1's outputs saturate to int16 and pass 2's to the sample
// range (packssdw / packsswb), where jidctint.c keeps 64-bit sums and wraps with & RANGE_MASK.  The two agree whenever
// nothing leaves those ranges, which holds for every file an encoder writes; on corrupt coefficients this restatement
// gives cv2's pixels.  Pass 1's DC-only shortcut (a shift, 16-bit) applies when the whole block has no AC term.
HD int16_t s16(int32_t v) { return (int16_t)(uint16_t)(uint32_t)v; }
HD int16_t sat16(int32_t v) { return (int16_t)(v < -32768 ? -32768 : v > 32767 ? 32767 : v); }
HD int32_t w32(int64_t v) { return (int32_t)(uint32_t)(uint64_t)v; }          // a 32-bit lane

// one 1-D pass on x[0..7] (16-bit lanes) -> 32-bit results before descaling, jidctint.c's output order
HD void idct_1d(const int16_t* x, int32_t* o) {
  const int64_t z2 = x[2], z3 = x[6];
  const int32_t tmp2 = w32(z2 * 4433 + z3 * (4433 - 15137)), tmp3 = w32(z2 * (4433 + 6270) + z3 * 4433);
  const int32_t tmp0 = w32((int64_t)s16(x[0] + x[4]) * 8192), tmp1 = w32((int64_t)s16(x[0] - x[4]) * 8192);
  const int32_t tmp10 = w32((int64_t)tmp0 + tmp3), tmp13 = w32((int64_t)tmp0 - tmp3);
  const int32_t tmp11 = w32((int64_t)tmp1 + tmp2), tmp12 = w32((int64_t)tmp1 - tmp2);
  const int64_t t0 = x[7], t1 = x[5], t2 = x[3], t3 = x[1];
  const int64_t z3o = s16(x[7] + x[3]), z4o = s16(x[5] + x[1]);
  const int64_t z3v = w32(z3o * (9633 - 16069) + z4o * 9633), z4v = w32(z3o * 9633 + z4o * (9633 - 3196));
  const int32_t o0 = w32(w32(t0 * (2446 - 7373) + t3 * -7373) + z3v);
  const int32_t o3 = w32(w32(t0 * -7373 + t3 * (12299 - 7373)) + z4v);
  const int32_t o1 = w32(w32(t1 * (16819 - 20995) + t2 * -20995) + z4v);
  const int32_t o2 = w32(w32(t1 * -20995 + t2 * (25172 - 20995)) + z3v);
  o[0] = w32((int64_t)tmp10 + o3); o[7] = w32((int64_t)tmp10 - o3);
  o[1] = w32((int64_t)tmp11 + o2); o[6] = w32((int64_t)tmp11 - o2);
  o[2] = w32((int64_t)tmp12 + o1); o[5] = w32((int64_t)tmp12 - o1);
  o[3] = w32((int64_t)tmp13 + o0); o[4] = w32((int64_t)tmp13 - o0);
}

HD bool block_has_ac(const int16_t* in) {
  int v = 0;
  for (int k = 8; k < 64; ++k) v |= in[k];
  return v != 0;
}

// pass 1 on column j: ws[8 * r + j]
HD void idct_col(const int16_t* in, const uint16_t* q, int j, bool ac, int16_t* ws) {
  int16_t x[8];
  for (int r = 0; r < 8; ++r) x[r] = s16((int32_t)in[8 * r + j] * (int32_t)q[8 * r + j]);
  if (!ac) {
    for (int r = 0; r < 8; ++r) ws[8 * r + j] = s16(x[0] * 4);
    return;
  }
  int32_t o[8];
  idct_1d(x, o);
  for (int r = 0; r < 8; ++r) ws[8 * r + j] = sat16(w32((int64_t)o[r] + 1024) >> 11);
}

// pass 2 on row r of ws into out[0..7]
HD void idct_row(const int16_t* ws, int r, uint8_t* out) {
  int32_t o[8];
  idct_1d(ws + 8 * r, o);
  for (int k = 0; k < 8; ++k) {
    const int32_t v = w32((int64_t)o[k] + (1 << 17)) >> 18;
    out[k] = (uint8_t)(v < -128 ? 0 : v > 127 ? 255 : v + 128);
  }
}

// component c's plane geometry: stride (= padded width) and the block (bx, by) of block b of MCU m
HD int32_t plane_stride(const Hdr& H, int c) { return H.mcux * 8 * (c ? 1 : H.h0); }
HD void block_xy(const Hdr& H, int32_t m, int b, int& c, int32_t& bx, int32_t& by) {
  const int32_t mx = m % H.mcux, my = m / H.mcux;
  c = H.blk_comp[b];
  if (c == 0) { bx = mx * H.h0 + b % H.h0; by = my * H.v0 + b / H.h0; }
  else { bx = mx; by = my; }
}

// ---- upsampling and colour (jdsample.c, jdcolor.c) -------------------------------------------------------------------
// chroma sample of output pixel (x, y) from plane p (stride ps) of dw x dh real samples
HD int chroma_at(const Hdr& H, const uint8_t* p, int32_t ps, int32_t dw, int32_t dh, int32_t x, int32_t y) {
  if (H.h0 == 1 && H.v0 == 1) return p[(int64_t)y * ps + x];
  if (H.h0 == 1) {                                                    // h1v2_fancy_upsample
    const int32_t j = y >> 1, jn = (y & 1) ? (j + 1 < dh ? j + 1 : j) : (j ? j - 1 : 0);
    return (3 * p[(int64_t)j * ps + x] + p[(int64_t)jn * ps + x] + ((y & 1) ? 2 : 1)) >> 2;
  }
  const int32_t i = x >> 1, in = (x & 1) ? (i + 1 < dw ? i + 1 : i) : (i ? i - 1 : 0);
  if (dw <= 2) return p[(int64_t)(H.v0 == 2 ? y >> 1 : y) * ps + i];  // h2v1_upsample / h2v2_upsample
  if (H.v0 == 1) {                                                    // h2v1_fancy_upsample
    const uint8_t* r = p + (int64_t)y * ps;
    return (3 * r[i] + r[in] + ((x & 1) ? 2 : 1)) >> 2;
  }
  const int32_t j = y >> 1, jn = (y & 1) ? (j + 1 < dh ? j + 1 : j) : (j ? j - 1 : 0);   // h2v2_fancy_upsample
  const uint8_t *r0 = p + (int64_t)j * ps, *r1 = p + (int64_t)jn * ps;
  const int cur = 3 * r0[i] + r1[i], nb = 3 * r0[in] + r1[in];
  return (3 * cur + nb + ((x & 1) ? 7 : 8)) >> 4;
}

HD uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

HD void color_pixel(const Hdr& H, uint8_t* const* planes, int32_t h, int32_t w, uint8_t* out, int32_t x, int32_t y) {
  const int64_t plane = (int64_t)h * w, o = (int64_t)y * w + x;
  const int yv = planes[0][(int64_t)y * plane_stride(H, 0) + x];
  if (H.nc == 1) { out[o] = out[plane + o] = out[2 * plane + o] = (uint8_t)yv; return; }
  const int32_t ps = plane_stride(H, 1), dw = (w + H.h0 - 1) / H.h0, dh = (h + H.v0 - 1) / H.v0;
  const int64_t cb = chroma_at(H, planes[1], ps, dw, dh, x, y) - 128, cr = chroma_at(H, planes[2], ps, dw, dh, x, y) - 128;
  // build_ycc_rgb_table: FIX(x) = x * 2^16 + 0.5; ONE_HALF = 2^15
  const int crr = (int)((91881 * cr + 32768) >> 16), cbb = (int)((116130 * cb + 32768) >> 16);
  const int g = (int)((-22554 * cb + 32768 + -46802 * cr) >> 16);
  out[o] = clamp255(yv + cbb);
  out[plane + o] = clamp255(yv + g);
  out[2 * plane + o] = clamp255(yv + crr);
}

// ---- device kernels --------------------------------------------------------------------------------------------------
struct DecFile {
  const uint8_t* data;
  int64_t size;
  uint8_t* out;
  Hdr* hdr;
  uint8_t* cs;                        // the de-stuffed stream (<= size bytes)
  int32_t* ivl;                       // ivl_bit [maxint + 1], ivl_chunk0 [maxint + 1]
  int32_t* ch;                        // 6 arrays of maxch
  int16_t* coef;                      // blocks bound x 64
  uint8_t* planes;                    // 3 planes of plane_bytes
  int64_t plane_bytes;
  int32_t h, w, nc, maxint, maxch;
};
struct DecArgs {
  DecFile f[kDecMax];
  int32_t* status;
  int32_t n;
};

HD Chunks chunks_of(const DecFile& f) {
  Chunks X;
  X.ivl_bit = f.ivl;
  X.ivl_chunk0 = f.ivl + f.maxint + 1;
  int32_t* c = f.ch;
  X.ent_pos = c; X.ent_st = c + f.maxch; X.ex_pos = c + 2 * f.maxch; X.ex_st = c + 3 * f.maxch;
  X.nblk = c + 4 * f.maxch; X.pref = c + 5 * f.maxch;
  return X;
}

// exclusive block-wide sum (blockDim.x a multiple of 32); total of every thread's v
__device__ int64_t block_excl_sum(int64_t v, int64_t* sh, int64_t& total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int64_t x = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[wid] = x;
  __syncthreads();
  if (wid == 0) {
    int64_t s = lane < nw ? sh[lane] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    sh[lane] = s;
  }
  __syncthreads();
  const int64_t r = x - v + (wid ? sh[wid - 1] : 0);
  total = sh[nw - 1];
  __syncthreads();
  return r;
}

__global__ void __launch_bounds__(32) jpeg_header_kernel(const __grid_constant__ DecArgs a) {
  __shared__ Raw R;
  const DecFile& f = a.f[blockIdx.x];
  if (threadIdx.x == 0) {
    const int st = parse_header(f.data, f.size, f.h, f.w, f.nc, R, *f.hdr);
    f.hdr->status = st;
    a.status[blockIdx.x] = st;
  }
}

__global__ void __launch_bounds__(kThreads) jpeg_scan_kernel(const __grid_constant__ DecArgs a) {
  __shared__ int64_t sh[32];
  __shared__ int64_t s_end;
  __shared__ int s_bad;
  const DecFile& f = a.f[blockIdx.x];
  Hdr& H = *f.hdr;
  if (H.status != LEDB200_JPEG_OK) return;
  const int t = threadIdx.x;
  const int64_t scan0 = H.scan0, size = f.size;
  constexpr int kPer = 16;
  constexpr int64_t kTile = (int64_t)kThreads * kPer;
  // zero the coefficients
  const int64_t nco = (int64_t)H.nmcu * H.bpm * 64 / 8;               // int4 stores (64 int16 = 8 x 16 bytes)
  for (int64_t i = t; i < nco; i += kThreads) reinterpret_cast<int4*>(f.coef)[i] = make_int4(0, 0, 0, 0);
  // the end of the scan: the first marker other than RSTn
  if (t == 0) { s_end = size; s_bad = 0; }
  __syncthreads();
  for (int64_t base = scan0; base < size; base += kTile) {
    const int64_t i0 = base + (int64_t)t * kPer;
    for (int64_t i = i0; i < i0 + kPer && i < size; ++i)
      if (is_end(f.data, i, size)) { atomicMin((unsigned long long*)&s_end, (unsigned long long)i); break; }
    __syncthreads();
    if (s_end < size) break;
    __syncthreads();
  }
  const int64_t end = s_end;
  if (end >= size) {
    if (t == 0) H.status = a.status[blockIdx.x] = LEDB200_JPEG_ETRUNC;
    return;
  }
  if (end + 1 >= size || f.data[end + 1] != 0xD9) {                   // the scan must be followed by EOI
    if (t == 0) H.status = a.status[blockIdx.x] = LEDB200_JPEG_ESEGMENT;
    return;
  }
  // de-stuff: kept bytes to cs, RSTn -> interval starts
  const int maxint = f.maxint, want = expected_intervals(H);
  int64_t kept = 0, rsts = 0;
  for (int64_t base = scan0; base < end; base += kTile) {
    const int64_t i0 = base + (int64_t)t * kPer;
    uint32_t km = 0, rm = 0;
    for (int k = 0; k < kPer; ++k) {
      const int64_t i = i0 + k;
      if (i >= end) break;
      bool keep, rst;
      classify(f.data, i, scan0, keep, rst);
      km |= (uint32_t)keep << k;
      rm |= (uint32_t)rst << k;
    }
    int64_t tk, tr;
    int64_t ok = block_excl_sum(__popc(km), sh, tk) + kept;
    int64_t orr = block_excl_sum(__popc(rm), sh, tr) + rsts;
    for (int k = 0; k < kPer; ++k) {
      const int64_t i = i0 + k;
      if (km >> k & 1) f.cs[ok++] = f.data[i];
      if (rm >> k & 1) {
        if (orr + 2 > want || orr + 1 > maxint || f.data[i + 1] != 0xD0 + (orr & 7)) s_bad = 1;
        else f.ivl[orr + 1] = (int32_t)(ok * 8);
        ++orr;
      }
    }
    kept += tk;
    rsts += tr;
  }
  __syncthreads();
  if (s_bad || rsts + 1 != want) {
    if (t == 0) H.status = a.status[blockIdx.x] = LEDB200_JPEG_ERESTART;
    return;
  }
  // subsequences per interval and their prefix
  const int nint = want;
  int32_t* chunk0 = f.ivl + maxint + 1;
  if (t == 0) { f.ivl[0] = 0; f.ivl[nint] = (int32_t)(kept * 8); }
  __syncthreads();
  const int per = (nint + kThreads - 1) / kThreads, k0 = min(nint, t * per), k1 = min(nint, k0 + per);
  int64_t cnt = 0;
  for (int k = k0; k < k1; ++k) cnt += max(1, (f.ivl[k + 1] - f.ivl[k] + kChunkBits - 1) / kChunkBits);
  int64_t total;
  int64_t c = block_excl_sum(cnt, sh, total);
  for (int k = k0; k < k1; ++k) {
    chunk0[k] = (int32_t)c;
    c += max(1, (f.ivl[k + 1] - f.ivl[k] + kChunkBits - 1) / kChunkBits);
  }
  if (t == 0) {
    chunk0[nint] = (int32_t)total;
    H.nint = nint;
    H.nchunks = (int32_t)total;
  }
}

__global__ void __launch_bounds__(kThreads) jpeg_huffman_kernel(const __grid_constant__ DecArgs a) {
  __shared__ Hdr H;
  __shared__ int64_t sh[32];
  __shared__ int s_changed;
  __shared__ unsigned long long s_err;
  __shared__ uint32_t s_dc[kThreads / 32][4];
  const DecFile& f = a.f[blockIdx.x];
  if (f.hdr->status != LEDB200_JPEG_OK) return;
  const int t = threadIdx.x;
  {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(f.hdr);
    uint32_t* dst = reinterpret_cast<uint32_t*>(&H);
    for (int i = t; i < (int)(sizeof(Hdr) / 4); i += kThreads) dst[i] = src[i];
  }
  const HuffTab* T = H.tabs;
  if (t == 0) s_err = ~0ull;
  __syncthreads();
  const Chunks X = chunks_of(f);
  const int nc = H.nchunks, per = (nc + kThreads - 1) / kThreads;
  const int a0 = min(nc, t * per), a1 = min(nc, a0 + per);
  // round 0: every thread from a guess (or its interval's start)
  if (a0 < a1) {
    const ChunkGeo g = chunk_geo(X, H.nint, a0);
    sync_run(H, T, f.cs, X, a0, a1, g.c0, 0, false);
  }
  // rounds: a thread whose entry differs from its predecessor's exit re-decodes until its states stop changing
  for (;;) {
    __syncthreads();
    int32_t pos = 0, st = 0;
    bool redo = false;
    if (a0 < a1 && a0 > 0) {
      entry_of(H, X, a0, pos, st);
      redo = pos != X.ent_pos[a0] || st != X.ent_st[a0];
    }
    if (t == 0) s_changed = 0;
    __syncthreads();
    if (redo) {
      sync_run(H, T, f.cs, X, a0, a1, pos, st, true);
      s_changed = 1;
    }
    __syncthreads();
    if (!s_changed) break;
  }
  // output blocks: exclusive scan of the block counts
  int64_t local = 0, total;
  for (int c = a0; c < a1; ++c) local += X.nblk[c];
  int64_t p = block_excl_sum(local, sh, total);
  for (int c = a0; c < a1; ++c) { X.pref[c] = (int32_t)p; p += X.nblk[c]; }
  __syncthreads();
  // the synchronised pass: coefficients; the first failing subsequence's status
  for (int c = a0; c < a1; ++c) {
    const int e = final_chunk(H, T, f.cs, X, c, f.coef);
    if (e) { atomicMin(&s_err, (unsigned long long)c << 8 | (unsigned)e); break; }
  }
  __syncthreads();
  if (s_err != ~0ull) {
    if (t == 0) f.hdr->status = a.status[blockIdx.x] = (int)(s_err & 255);
    return;
  }
  // DC: segmented scan over MCUs (per component, reset at every interval)
  const int32_t M = H.nmcu, mper = (M + kThreads - 1) / kThreads, m0 = min(M, t * mper), m1 = min(M, m0 + mper);
  bool reset = false;
  uint16_t sum[3] = {0, 0, 0};
  dc_range(H, f.coef, m0, m1, false, reset, sum);
  // Hillis-Steele over (reset, sums): (fa, sa) + (fb, sb) = (fa | fb, fb ? sb : sa + sb)
  const int lane = t & 31, wid = t >> 5;
  uint32_t fl = reset, s0 = sum[0], s1 = sum[1], s2 = sum[2];
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t pf = __shfl_up_sync(0xffffffffu, fl, o), p0 = __shfl_up_sync(0xffffffffu, s0, o),
                   p1 = __shfl_up_sync(0xffffffffu, s1, o), p2 = __shfl_up_sync(0xffffffffu, s2, o);
    if (lane >= o && !fl) { s0 += p0; s1 += p1; s2 += p2; fl = pf; }
  }
  if (lane == 31) { s_dc[wid][0] = fl; s_dc[wid][1] = s0; s_dc[wid][2] = s1; s_dc[wid][3] = s2; }
  __syncthreads();
  if (wid == 0) {
    uint32_t wf = s_dc[lane][0], w0 = s_dc[lane][1], w1 = s_dc[lane][2], w2 = s_dc[lane][3];
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t pf = __shfl_up_sync(0xffffffffu, wf, o), p0 = __shfl_up_sync(0xffffffffu, w0, o),
                     p1 = __shfl_up_sync(0xffffffffu, w1, o), p2 = __shfl_up_sync(0xffffffffu, w2, o);
      if (lane >= o && !wf) { w0 += p0; w1 += p1; w2 += p2; wf = pf; }
    }
    s_dc[lane][0] = wf; s_dc[lane][1] = w0; s_dc[lane][2] = w1; s_dc[lane][3] = w2;
  }
  __syncthreads();
  // carry into this thread: the inclusive value of the thread before it
  uint32_t c0 = __shfl_up_sync(0xffffffffu, s0, 1), c1 = __shfl_up_sync(0xffffffffu, s1, 1),
           c2 = __shfl_up_sync(0xffffffffu, s2, 1), cf = __shfl_up_sync(0xffffffffu, fl, 1);
  if (lane == 0) { c0 = c1 = c2 = 0; cf = 0; }
  if (wid > 0 && !cf) { c0 += s_dc[wid - 1][1]; c1 += s_dc[wid - 1][2]; c2 += s_dc[wid - 1][3]; }
  uint16_t carry[3] = {(uint16_t)c0, (uint16_t)c1, (uint16_t)c2};
  reset = false;
  dc_range(H, f.coef, m0, m1, true, reset, carry);
}

// 8 threads per block, 32 blocks per CTA: column pass into shared memory, row pass into the component's plane
__global__ void __launch_bounds__(256) jpeg_idct_kernel(const __grid_constant__ DecArgs a) {
  __shared__ int16_t ws[32][64];
  const DecFile& f = a.f[blockIdx.y];
  const Hdr& H = *f.hdr;
  if (H.status != LEDB200_JPEG_OK) return;
  const int j = threadIdx.x & 7, lb = threadIdx.x >> 3;
  const int64_t g = (int64_t)blockIdx.x * 32 + lb;
  const bool on = g < (int64_t)H.nmcu * H.bpm;
  int c = 0;
  int32_t bx = 0, by = 0;
  if (on) {
    block_xy(H, (int32_t)(g / H.bpm), (int)(g % H.bpm), c, bx, by);
    idct_col(f.coef + g * 64, H.q[c], j, block_has_ac(f.coef + g * 64), ws[lb]);
  }
  __syncwarp();
  if (on) {
    const int32_t ps = plane_stride(H, c);
    idct_row(ws[lb], j, f.planes + c * f.plane_bytes + ((int64_t)by * 8 + j) * ps + (int64_t)bx * 8);
  }
}

__global__ void __launch_bounds__(256) jpeg_color_kernel(const __grid_constant__ DecArgs a) {
  const DecFile& f = a.f[blockIdx.y];
  const Hdr& H = *f.hdr;
  if (H.status != LEDB200_JPEG_OK) return;
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= (int64_t)f.h * f.w) return;
  uint8_t* planes[3] = {f.planes, f.planes + f.plane_bytes, f.planes + 2 * f.plane_bytes};
  color_pixel(H, planes, f.h, f.w, f.out, (int32_t)(i % f.w), (int32_t)(i / f.w));
}

// ---- host side ------------------------------------------------------------------------------------------------------
struct Slot { int64_t hdr, cs, ivl, ch, coef, planes, plane_bytes; int32_t maxint, maxch; };

int64_t align16(int64_t v) { return (v + 15) / 16 * 16; }

// Bounds for any accepted sampling: at most 3 (bx + 1) (by + 1) blocks, each plane at most (bx + 1) (by + 1) blocks
Slot slot_of(const ledb200_jpeg_file& d, int64_t& at) {
  Slot s;
  const int64_t bx = (d.w + 7) / 8, by = (d.h + 7) / 8, blocks = (bx + 1) * (by + 1);
  const int64_t mcu_max = bx * by;
  s.maxint = (int32_t)std::min<int64_t>(mcu_max, d.size / 2 + 1);
  s.maxch = (int32_t)((d.size * 8 + kChunkBits - 1) / kChunkBits + s.maxint + 1);
  s.hdr = at; at += align16(sizeof(Hdr));
  s.cs = at; at += align16(d.size + 16);
  s.ivl = at; at += align16(8 * ((int64_t)s.maxint + 1));
  s.ch = at; at += align16(24 * (int64_t)s.maxch);
  s.coef = at; at += 3 * blocks * 128;
  s.plane_bytes = blocks * 64;
  s.planes = at; at += 3 * s.plane_bytes;
  return s;
}

int check_files(const ledb200_jpeg_file* files, int n, const char* who) {
  const std::string w(who);
  if (!files) return fail(LEDB200_EINVAL, w + ": null file descriptors");
  if (n < 1) return fail(LEDB200_EINVAL, w + ": at least one file");
  for (int i = 0; i < n; ++i) {
    const ledb200_jpeg_file& d = files[i];
    const std::string at = w + ": file " + std::to_string(i) + ": ";
    if (!d.data || !d.out) return fail(LEDB200_EINVAL, at + "null data or output");
    if (d.size < 4 || d.size >= kMaxSize) return fail(LEDB200_EINVAL, at + "size must be in [4, 2^28)");
    if (d.h < 1 || d.w < 1 || d.h > 65535 || d.w > 65535 || (int64_t)d.h * d.w > (int64_t)1 << 30)
      return fail(LEDB200_EINVAL, at + "h and w must be in [1, 65535] and h * w at most 2^30");
    if (d.components != 1 && d.components != 3) return fail(LEDB200_EINVAL, at + "components must be 1 or 3");
  }
  return LEDB200_OK;
}

DecFile dec_file(const ledb200_jpeg_file& d, const Slot& s, uint8_t* ws) {
  DecFile f;
  f.data = d.data; f.size = d.size; f.out = d.out;
  f.hdr = reinterpret_cast<Hdr*>(ws + s.hdr);
  f.cs = ws + s.cs;
  f.ivl = reinterpret_cast<int32_t*>(ws + s.ivl);
  f.ch = reinterpret_cast<int32_t*>(ws + s.ch);
  f.coef = reinterpret_cast<int16_t*>(ws + s.coef);
  f.planes = ws + s.planes;
  f.plane_bytes = s.plane_bytes;
  f.h = d.h; f.w = d.w; f.nc = d.components; f.maxint = s.maxint; f.maxch = s.maxch;
  return f;
}

// the device pipeline on the CPU, for one file whose buffers are all host memory
int decode_host(const DecFile& f) {
  std::vector<Raw> R(1);
  Hdr& H = *f.hdr;
  int st = parse_header(f.data, f.size, f.h, f.w, f.nc, R[0], H);
  if (st) return st;
  std::memset(f.coef, 0, (size_t)H.nmcu * H.bpm * 128);
  int64_t end = f.size;
  for (int64_t i = H.scan0; i < f.size; ++i)
    if (is_end(f.data, i, f.size)) { end = i; break; }
  if (end >= f.size) return LEDB200_JPEG_ETRUNC;
  if (end + 1 >= f.size || f.data[end + 1] != 0xD9) return LEDB200_JPEG_ESEGMENT;
  const int want = expected_intervals(H);
  int64_t kept = 0, rsts = 0;
  for (int64_t i = H.scan0; i < end; ++i) {
    bool keep, rst;
    classify(f.data, i, H.scan0, keep, rst);
    if (keep) f.cs[kept++] = f.data[i];
    if (rst) {
      if (rsts + 2 > want || rsts + 1 > f.maxint || f.data[i + 1] != 0xD0 + (rsts & 7)) return LEDB200_JPEG_ERESTART;
      f.ivl[rsts + 1] = (int32_t)(kept * 8);
      ++rsts;
    }
  }
  if (rsts + 1 != want) return LEDB200_JPEG_ERESTART;
  int32_t* chunk0 = f.ivl + f.maxint + 1;
  f.ivl[0] = 0;
  f.ivl[want] = (int32_t)(kept * 8);
  int32_t nch = 0;
  for (int k = 0; k < want; ++k) {
    chunk0[k] = nch;
    nch += std::max(1, (f.ivl[k + 1] - f.ivl[k] + kChunkBits - 1) / kChunkBits);
  }
  chunk0[want] = nch;
  H.nint = want;
  H.nchunks = nch;
  // the Huffman stage, serially over the device's threads
  const Chunks X = chunks_of(f);
  const int per = (nch + kThreads - 1) / kThreads;
  for (int t = 0; t < kThreads; ++t) {
    const int a0 = std::min(nch, t * per), a1 = std::min(nch, a0 + per);
    if (a0 < a1) sync_run(H, H.tabs, f.cs, X, a0, a1, chunk_geo(X, H.nint, a0).c0, 0, false);
  }
  for (bool changed = true; changed;) {
    changed = false;
    std::vector<int32_t> pos(kThreads), stt(kThreads);
    std::vector<char> redo(kThreads, 0);
    for (int t = 0; t < kThreads; ++t) {
      const int a0 = std::min(nch, t * per), a1 = std::min(nch, a0 + per);
      if (a0 < a1 && a0 > 0) {
        entry_of(H, X, a0, pos[t], stt[t]);
        redo[t] = pos[t] != X.ent_pos[a0] || stt[t] != X.ent_st[a0];
      }
    }
    for (int t = 0; t < kThreads; ++t) {
      if (!redo[t]) continue;
      const int a0 = std::min(nch, t * per), a1 = std::min(nch, a0 + per);
      sync_run(H, H.tabs, f.cs, X, a0, a1, pos[t], stt[t], true);
      changed = true;
    }
  }
  int32_t p = 0;
  for (int c = 0; c < nch; ++c) { X.pref[c] = p; p += X.nblk[c]; }
  for (int c = 0; c < nch; ++c)
    if (int e = final_chunk(H, H.tabs, f.cs, X, c, f.coef)) return e;
  bool reset = false;
  uint16_t sum[3] = {0, 0, 0};
  dc_range(H, f.coef, 0, H.nmcu, true, reset, sum);
  // IDCT and colour
  uint8_t* planes[3] = {f.planes, f.planes + f.plane_bytes, f.planes + 2 * f.plane_bytes};
  int16_t ws[64];
  for (int64_t g = 0; g < (int64_t)H.nmcu * H.bpm; ++g) {
    int c;
    int32_t bx, by;
    block_xy(H, (int32_t)(g / H.bpm), (int)(g % H.bpm), c, bx, by);
    const bool ac = block_has_ac(f.coef + g * 64);
    for (int j = 0; j < 8; ++j) idct_col(f.coef + g * 64, H.q[c], j, ac, ws);
    const int32_t ps = plane_stride(H, c);
    for (int r = 0; r < 8; ++r) idct_row(ws, r, planes[c] + ((int64_t)by * 8 + r) * ps + (int64_t)bx * 8);
  }
  for (int32_t y = 0; y < f.h; ++y)
    for (int32_t x = 0; x < f.w; ++x) color_pixel(H, planes, f.h, f.w, f.out, x, y);
  return LEDB200_JPEG_OK;
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int64_t ledb200_jpeg_decode_workspace_bytes(const ledb200_jpeg_file* files, int32_t n) {
  if (int rc = check_files(files, n, "jpeg_decode_workspace_bytes")) return rc;
  int64_t at = 0;
  for (int i = 0; i < n; ++i) slot_of(files[i], at);
  return at;
}

int ledb200_jpeg_decode(const ledb200_jpeg_file* files, int32_t n, void* workspace, int32_t* status, void* stream) {
  if (int rc = check_files(files, n, "jpeg_decode")) return rc;
  if (!workspace || !status) return fail(LEDB200_EINVAL, "jpeg_decode: null workspace or status");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  int64_t at = 0;
  for (int i0 = 0; i0 < n; i0 += kDecMax) {
    DecArgs a;
    a.n = n - i0 < kDecMax ? n - i0 : kDecMax;
    a.status = status + i0;
    int64_t blocks = 1, pixels = 1;
    for (int i = 0; i < a.n; ++i) {
      const ledb200_jpeg_file& d = files[i0 + i];
      const Slot s = slot_of(d, at);
      a.f[i] = dec_file(d, s, ws);
      blocks = std::max<int64_t>(blocks, 3 * s.plane_bytes / 64);
      pixels = std::max<int64_t>(pixels, (int64_t)d.h * d.w);
    }
    jpeg_header_kernel<<<a.n, 32, 0, st>>>(a);
    LEDB_LAUNCH_OK("jpeg_header_kernel");
    jpeg_scan_kernel<<<a.n, kThreads, 0, st>>>(a);
    LEDB_LAUNCH_OK("jpeg_scan_kernel");
    jpeg_huffman_kernel<<<a.n, kThreads, 0, st>>>(a);
    LEDB_LAUNCH_OK("jpeg_huffman_kernel");
    jpeg_idct_kernel<<<dim3((unsigned)((blocks + 31) / 32), a.n), 256, 0, st>>>(a);
    LEDB_LAUNCH_OK("jpeg_idct_kernel");
    jpeg_color_kernel<<<dim3((unsigned)((pixels + 255) / 256), a.n), 256, 0, st>>>(a);
    LEDB_LAUNCH_OK("jpeg_color_kernel");
  }
  return LEDB200_OK;
}

int ledb200_jpeg_decode_host(const ledb200_jpeg_file* files, int32_t n, int32_t* status) {
  if (int rc = check_files(files, n, "jpeg_decode_host")) return rc;
  if (!status) return fail(LEDB200_EINVAL, "jpeg_decode_host: null status");
  for (int i = 0; i < n; ++i) {
    int64_t at = 0;
    const Slot s = slot_of(files[i], at);
    std::vector<uint8_t> ws((size_t)at + 16);
    uint8_t* base = reinterpret_cast<uint8_t*>(align16(reinterpret_cast<int64_t>(ws.data())));
    status[i] = decode_host(dec_file(files[i], s, base));
  }
  return LEDB200_OK;
}

}  // extern "C"
