// Label maps and drawn pictures -> PNG files on the device (IoUMetric's output_dir / format_only, mmseg's
// `tools/test.py --out` and `--show-dir`).
//
// A label map becomes an 8-bit PNG (no interlace) whose pixels are lut[label & 255]: (label + add) mod 256 for
// IoUMetric, what `Image.fromarray((pred + reduce_zero_label).astype(np.uint8))` saves, or CityscapesMetric's trainId ->
// labelId table.  The file is the signature, IHDR, one IDAT holding one zlib stream (header 78 01, deflate, big-endian
// Adler-32) and IEND: grayscale (colour type 0), or with `palette` colour type 3 and, before the IDAT, the 256-entry grey
// PLTE that PIL's `.convert('P')` writes for a grayscale image.  Every scanline of these has filter type 0.  An RGB image
// ([H,W,3] uint8, SegLocalVisualizer's pictures) becomes colour type 2, each scanline with the filter libpng's heuristic
// picks.  S = C * W + 1 is the bytes of one filtered scanline (C = 1 or 3 bytes per pixel).
//
//  * png_filter_kernel   : the filtered scanline stream (a 0 filter byte, then W pixels, per row) into the workspace.
//  * png_filter_rgb_kernel : the same for RGB rows, each with the filter whose residuals have the least sum of
//      |signed byte| (None, Sub, Up, Average, Paeth; the first on a tie).
//  * png_band_kernel     : one warp per band of R rows (R * S <= 65535 bytes where a row allows it).  The band is
//      one dynamic-Huffman deflate block, or stored blocks when that is smaller.  Matches take the longer of distance 1
//      (a run) and S (the byte one row up) when S <= 32768; they may reach back into the previous band, since
//      the image is one zlib stream.  The warp first writes two bitmaps of the band (byte equals the byte 1 / S
//      back), so a match length is a search for the next clear bit, a few words per 258 bytes.  The greedy parse is split over the 32 lanes: lane k parses from where lane k - 1's
//      last match ended, found by re-parsing until no lane's start moves (lane k's start is final after k + 1 rounds,
//      typically two in all), so the tokens are exactly those of one sequential greedy parse of the band.  The parse
//      then runs twice more with the band's codes: once to count each lane's bits (a warp scan gives the offsets), once
//      to write them with atomicOr into 32-bit words.  A non-final band ends in an empty stored block (a sync flush:
//      00 00 FF FF once byte-aligned) so that the next band starts on a byte; the last band sets BFINAL.
//  * png_size_kernel     : per image, the scan of the band sizes and the Adler-32 combined from the per-band sums.
//  * png_scan_kernel     : the file offsets of the batch.
//  * png_assemble_kernel : per image, the headers, the bands back to back, and the IDAT CRC-32 (per-thread CRCs merged
//      with the GF(2) combine identity crc(AB) = crc(A) * x^(8 |B|) + crc(B) mod P).
#include <algorithm>
#include <string>

#include "kernels.h"
#include "png_common.cuh"

namespace ledb {
namespace {

constexpr int kLL = 286, kDist = 30, kCL = 19;
constexpr int64_t kStoredMax = 65535;
// file bytes outside the zlib data: signature 8, IHDR 25, IDAT length + type 8, zlib header 2, Adler-32 4, IDAT CRC 4,
// IEND 12
constexpr int64_t kFileOverhead = 8 + 25 + 8 + 2 + 4 + 4 + 12;
constexpr int64_t kIdatData = 8 + 25 + 8;    // offset of the zlib header within the file (no palette)
constexpr int64_t kPlteChunk = 12 + 768;     // the grey PLTE chunk of a palette file, between IHDR and IDAT

struct Lut { uint8_t v[256]; };

struct Plan {
  int64_t S, n, R, nb, band_cap;              // row bytes, stream bytes, rows per band, bands, slot bytes per band
  int64_t bm_words;                           // words of one match bitmap of a band
  int64_t slot_off, info_off, adler_off, bm_off, total;
};

__host__ __device__ inline int64_t stored_bytes(int64_t L) { return L + 5 * ((L + kStoredMax - 1) / kStoredMax); }

Plan make_plan(int N, int H, int W, int C) {
  Plan p;
  p.S = (int64_t)C * W + 1;
  p.n = (int64_t)H * p.S;
  p.R = std::max<int64_t>(1, std::min<int64_t>(H, kStoredMax / p.S));
  p.nb = (H + p.R - 1) / p.R;
  p.band_cap = (stored_bytes(p.R * p.S) + 16 + 15) / 16 * 16;
  auto al = [](int64_t v) { return (v + 255) / 256 * 256; };
  p.slot_off = al((int64_t)N * p.n);
  p.info_off = p.slot_off + al((int64_t)N * p.nb * p.band_cap);
  p.adler_off = p.info_off + al((int64_t)N * p.nb * 4 * 8);
  p.bm_words = (p.R * p.S + 31) / 32 + 1;
  p.bm_off = p.adler_off + al((int64_t)N * 8);
  p.total = p.bm_off + al((int64_t)N * p.nb * 2 * p.bm_words * 4);
  return p;
}

int64_t bound_of(const Plan& p) {
  const int64_t last = p.n - (p.nb - 1) * p.R * p.S;
  return kFileOverhead + (p.nb - 1) * stored_bytes(p.R * p.S) + stored_bytes(last);
}

// ---- filtered scanlines --------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) png_filter_kernel(const T* __restrict__ labels, int W, int64_t S,
                                                        const __grid_constant__ Lut lut, uint8_t* __restrict__ raw) {
  __shared__ uint8_t tab[256];
  tab[threadIdx.x] = lut.v[threadIdx.x];
  __syncthreads();
  const int64_t row = blockIdx.x;
  const T* src = labels + row * W;
  uint8_t* dst = raw + row * S;
  for (int c = threadIdx.x; c <= W; c += blockDim.x)
    dst[c] = c == 0 ? (uint8_t)0 : tab[(uint8_t)src[c - 1]];
}

// libpng's filter heuristic: the residual byte v costs min(v, 256 - v), its magnitude as a signed byte
__device__ __forceinline__ uint32_t sad(uint32_t v) { v &= 255u; return v < 128u ? v : 256u - v; }

__device__ __forceinline__ uint32_t paeth(int a, int b, int c) {
  const int p = a + b - c, pa = abs(p - a), pb = abs(p - b), pc = abs(p - c);
  return (uint32_t)(pa <= pb && pa <= pc ? a : pb <= pc ? b : c);
}

// residual of byte j (j >= 0) of a row under filter f, x the byte, a / b / c the bytes left, up and up-left
__device__ __forceinline__ uint32_t residual(int f, uint32_t x, uint32_t a, uint32_t b, uint32_t c) {
  switch (f) {
    case 0: return x;
    case 1: return x - a;
    case 2: return x - b;
    case 3: return x - ((a + b) >> 1);
    default: return x - paeth((int)a, (int)b, (int)c);
  }
}

// One block per row of rgb [N*H, W*3]: the five filters' costs, a block reduction, then the chosen filter's row.
__global__ void __launch_bounds__(256) png_filter_rgb_kernel(const uint8_t* __restrict__ rgb, int H, int W, int64_t S,
                                                            uint8_t* __restrict__ raw) {
  __shared__ unsigned long long part[8][5];
  __shared__ int best_s;
  const int64_t row = blockIdx.x;
  const int64_t B = 3 * (int64_t)W;
  const uint8_t* cur = rgb + row * B;
  const uint8_t* up = row % H ? cur - B : nullptr;
  auto bytes = [&](int64_t j, uint32_t& x, uint32_t& a, uint32_t& b, uint32_t& c) {
    x = cur[j];
    a = j >= 3 ? cur[j - 3] : 0u;
    b = up ? up[j] : 0u;
    c = up && j >= 3 ? up[j - 3] : 0u;
  };
  unsigned long long cost[5] = {0, 0, 0, 0, 0};
  for (int64_t j = threadIdx.x; j < B; j += blockDim.x) {
    uint32_t x, a, b, c;
    bytes(j, x, a, b, c);
#pragma unroll
    for (int f = 0; f < 5; ++f) cost[f] += sad(residual(f, x, a, b, c));
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int f = 0; f < 5; ++f) {
    for (int o = 16; o; o >>= 1) cost[f] += __shfl_xor_sync(0xffffffffu, cost[f], o);
    if (lane == 0) part[wid][f] = cost[f];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    unsigned long long mins = 0;
    for (int f = 0; f < 5; ++f) {
      unsigned long long s = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += part[w][f];
      if (f == 0 || s < mins) { mins = s; best = f; }
    }
    best_s = best;
  }
  __syncthreads();
  const int f = best_s;
  uint8_t* dst = raw + row * S;
  if (threadIdx.x == 0) dst[0] = (uint8_t)f;
  for (int64_t j = threadIdx.x; j < B; j += blockDim.x) {
    uint32_t x, a, b, c;
    bytes(j, x, a, b, c);
    dst[1 + j] = (uint8_t)residual(f, x, a, b, c);
  }
}

// ---- deflate symbols -------------------------------------------------------------------------------------------------
// length 3..258 -> lit/len code 257 + lc with `eb` extra bits of value `ev` (RFC 1951 3.2.5)
__device__ __forceinline__ void len_code(int L, int& lc, int& eb, int& ev) {
  const int v = L - 3;
  if (v < 8) { lc = v; eb = 0; ev = 0; return; }
  if (v == 255) { lc = 28; eb = 0; ev = 0; return; }
  const int nb = 31 - __clz(v) - 2;
  const int hi = (v >> nb) & 3;
  lc = 4 * nb + 4 + hi; eb = nb; ev = v - ((4 | hi) << nb);
}
// distance 1..32768 -> distance code with extra bits
__device__ __forceinline__ void dist_code(int d, int& dc, int& eb, int& ev) {
  const int u = d - 1;
  if (u < 4) { dc = u; eb = 0; ev = 0; return; }
  const int nb = 31 - __clz(u) - 1;
  const int hi = (u >> nb) & 1;
  dc = 2 * nb + 2 + hi; eb = nb; ev = u - ((2 | hi) << nb);
}

// Length of the run of set bits of a band's match bitmap from bit `off` (bit j: byte j of the band equals the byte one
// candidate distance back), capped at maxl (<= the bits left in the band).
__device__ __forceinline__ int run_len(const uint32_t* __restrict__ bm, int64_t off, int maxl) {
  int64_t w = off >> 5;
  uint32_t x = ~bm[w] >> (off & 31);
  int l = 0;
  for (int avail = 32 - (int)(off & 31); l < maxl; avail = 32, x = ~bm[++w]) {
    if (x) { l += __ffs(x) - 1; break; }
    l += avail;
  }
  return min(l, maxl);
}

// Greedy parse of [s, end) of the band starting at B0: a token starting before `end` may run on to band_end.  Returns
// where the last token ends.  f(lit, len, far): a literal when len == 0, else a match of `len` at distance 1
// (far == false, bitmap bm1) or S (bitmap bmS, empty when S > 32768).
template <class F>
__device__ int64_t parse(const uint8_t* __restrict__ raw, const uint32_t* bm1, const uint32_t* bmS, int64_t B0,
                         int64_t s, int64_t end, int64_t band_end, F&& f) {
  int64_t i = s;
  while (i < end) {
    const int maxl = (int)(band_end - i < 258 ? band_end - i : 258);
    const int l1 = run_len(bm1, i - B0, maxl);
    const int lS = l1 < maxl ? run_len(bmS, i - B0, maxl) : 0;
    if (lS > l1 && lS >= 3) { f(0, lS, true); i += lS; }
    else if (l1 >= 3) { f(0, l1, false); i += l1; }
    else { f(__ldg(raw + i), 0, false); ++i; }
  }
  return max(i, s);
}

struct BitWriter {
  uint32_t* out;
  int64_t word;
  uint64_t acc;
  int n;
  __device__ BitWriter(uint32_t* o, int64_t bit) : out(o), word(bit >> 5), acc(0), n((int)(bit & 31)) {}
  __device__ void put(uint32_t v, int nb) {
    acc |= (uint64_t)v << n;
    n += nb;
    if (n >= 32) { atomicOr(out + word, (uint32_t)acc); ++word; acc >>= 32; n -= 32; }
  }
  __device__ void flush() { if (n > 0) atomicOr(out + word, (uint32_t)acc); }
};

struct SymFreq { uint32_t key; uint16_t sym; };

// Code lengths of a length-limited Huffman code for freq[0..n) (warp-cooperative, result in len[]).  The used symbols
// are rank-sorted by (freq, symbol); lane 0 runs Moffat & Katajainen's in-place minimum-redundancy construction, folds
// lengths over `limit` into `limit`, restores the Kraft sum by lengthening the deepest shorter codes, and hands the
// shortest lengths to the most frequent symbols.  With two or more used symbols the code is complete.
__device__ __forceinline__ void huffman_lengths(const uint32_t* freq, int n, int limit, uint8_t* len, SymFreq* A, int* num, int lane) {
  int m = 0;
  for (int base = 0; base < n; base += 32) {
    const int s = base + lane;
    const bool used = s < n && freq[s] > 0;
    m += __popc(__ballot_sync(0xffffffffu, used));
    if (s < n) len[s] = 0;
  }
  for (int s = lane; s < n; s += 32) {
    if (!freq[s]) continue;
    int r = 0;
    for (int t = 0; t < n; ++t)
      r += freq[t] > 0 && (freq[t] < freq[s] || (freq[t] == freq[s] && t < s));
    A[r].key = freq[s]; A[r].sym = (uint16_t)s;
  }
  __syncwarp();
  if (lane == 0 && m > 0) {
    if (m == 1) {
      len[A[0].sym] = 1;
    } else {
      int root = 0, leaf = 2, next;
      A[0].key += A[1].key;
      for (next = 1; next < m - 1; ++next) {
        if (leaf >= m || A[root].key < A[leaf].key) { A[next].key = A[root].key; A[root++].key = next; }
        else A[next].key = A[leaf++].key;
        if (leaf >= m || (root < next && A[root].key < A[leaf].key)) { A[next].key += A[root].key; A[root++].key = next; }
        else A[next].key += A[leaf++].key;
      }
      A[m - 2].key = 0;
      for (next = m - 3; next >= 0; --next) A[next].key = A[A[next].key].key + 1;
      int avbl = 1, used = 0, dpth = 0;
      root = m - 2; next = m - 1;
      while (avbl > 0) {
        while (root >= 0 && (int)A[root].key == dpth) { ++used; --root; }
        while (avbl > used) { A[next--].key = dpth; --avbl; }
        avbl = 2 * used; ++dpth; used = 0;
      }
      for (int i = 0; i < 16; ++i) num[i] = 0;
      for (int i = 0; i < m; ++i) ++num[min((int)A[i].key, limit)];
      uint32_t total = 0;
      for (int i = limit; i > 0; --i) total += (uint32_t)num[i] << (limit - i);
      while (total != (1u << limit)) {
        --num[limit];
        for (int i = limit - 1; i > 0; --i)
          if (num[i]) { --num[i]; num[i + 1] += 2; break; }
        --total;
      }
      int j = m;
      for (int i = 1; i <= limit; ++i)
        for (int k = num[i]; k > 0; --k) len[A[--j].sym] = (uint8_t)i;
    }
  }
  __syncwarp();
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first stream; lane 0
__device__ __forceinline__ void canonical_codes(const uint8_t* len, int n, uint16_t* code, int* count, int* next) {
  for (int b = 0; b < 16; ++b) count[b] = 0;
  for (int s = 0; s < n; ++s) ++count[len[s]];
  count[0] = 0;
  int c = 0;
  for (int b = 1; b < 16; ++b) { c = (c + count[b - 1]) << 1; next[b] = c; }
  for (int s = 0; s < n; ++s)
    if (len[s]) code[s] = (uint16_t)(__brev((uint32_t)next[len[s]]++) >> (32 - len[s]));
}

__constant__ uint8_t kCLOrder[kCL] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct BandSmem {
  uint32_t freq_ll[kLL], freq_d[kDist], freq_cl[kCL];
  uint16_t code_ll[kLL], code_d[kDist], code_cl[kCL];
  uint8_t len_ll[kLL], len_d[kDist], len_cl[kCL];
  uint16_t rle[kLL + kDist];                   // code-length symbol | repeat extra << 5
  SymFreq sort[kLL];
  int num[16], next[16];                     // Huffman scratch
  int nrle, hlit, hdist, hclen;
  int64_t hdr_bits;
};

// Band b of image `img`: compressed (or stored) bytes into its slot, then {bytes, Adler sum s1, Adler sum s2, 0} into
// info.  s1 / s2 are the band's byte sum and sum of suffix-weighted bytes, mod 65521.
__global__ void __launch_bounds__(32) png_band_kernel(const uint8_t* __restrict__ raw_all, Plan p,
                                                      uint8_t* __restrict__ slots, int64_t* __restrict__ info,
                                                      uint32_t* __restrict__ bitmaps) {
  __shared__ BandSmem sm;
  const int lane = threadIdx.x;
  const int64_t img = blockIdx.x / p.nb, b = blockIdx.x % p.nb;
  const uint8_t* raw = raw_all + img * p.n;
  const int64_t B0 = b * p.R * p.S, B1 = min(p.n, B0 + p.R * p.S), L = B1 - B0;
  const bool final_band = b == p.nb - 1;
  const int64_t seg = (L + 31) / 32;
  const int64_t a_nom = min(B1, B0 + lane * seg), e_nom = min(B1, a_nom + seg);
  const bool use_far = p.S <= 32768;
  uint8_t* slot = slots + (int64_t)blockIdx.x * p.band_cap;
  uint32_t* slot32 = reinterpret_cast<uint32_t*>(slot);

  // match bitmaps: bit j of bm1 / bmS is set when byte B0 + j equals the byte 1 / S back
  uint32_t* bm1 = bitmaps + (int64_t)blockIdx.x * 2 * p.bm_words;
  uint32_t* bmS = bm1 + p.bm_words;
  for (int64_t w = 0; w < (L + 31) / 32; ++w) {
    const int64_t i = B0 + w * 32 + lane;
    bool e1 = false, eS = false;
    if (i < B1) {
      const uint8_t x = __ldg(raw + i);
      e1 = i >= 1 && x == __ldg(raw + i - 1);
      eS = use_far && i >= p.S && x == __ldg(raw + i - p.S);
    }
    const uint32_t m1 = __ballot_sync(0xffffffffu, e1), mS = __ballot_sync(0xffffffffu, eS);
    if (lane == 0) { bm1[w] = m1; bmS[w] = mS; }
  }
  __syncwarp();

  // Adler-32 sums of this lane's nominal segment (any partition works for the sums)
  uint64_t s1, s2;
  adler_sums(raw + a_nom, e_nom - a_nom, s1, s2);
  s2 = adler_shift(s1, s2, B1 - e_nom);
  for (int o = 16; o; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  s1 %= kAdlerMod; s2 %= kAdlerMod;

  // pass 1: find the lanes' starts of the sequential greedy parse, counting symbols in the round that confirms them
  const int64_t dfar = p.S;
  int fdc, feb, fev;
  dist_code(use_far ? (int)dfar : 1, fdc, feb, fev);
  int64_t start = a_nom, end;
  for (;;) {
    for (int s = lane; s < kLL; s += 32) sm.freq_ll[s] = 0;
    if (lane < kDist) sm.freq_d[lane] = 0;
    __syncwarp();
    end = parse(raw, bm1, bmS, B0, start, e_nom, B1, [&](int lit, int l, bool far) {
      if (!l) { atomicAdd(&sm.freq_ll[lit], 1u); return; }
      int lc, eb, ev;
      len_code(l, lc, eb, ev);
      atomicAdd(&sm.freq_ll[257 + lc], 1u);
      atomicAdd(&sm.freq_d[far ? fdc : 0], 1u);
    });
    int64_t nstart = __shfl_up_sync(0xffffffffu, end, 1);
    if (lane == 0) nstart = B0;
    nstart = max(nstart, a_nom);
    const bool moved = __any_sync(0xffffffffu, nstart != start);
    __syncwarp();
    if (!moved) break;
    start = nstart;
  }

  // codes
  if (lane == 0) sm.freq_ll[256] = 1;          // end of block
  __syncwarp();
  huffman_lengths(sm.freq_ll, kLL, 15, sm.len_ll, sm.sort, sm.num, lane);
  huffman_lengths(sm.freq_d, kDist, 15, sm.len_d, sm.sort, sm.num, lane);
  if (lane == 0) {
    int nd = 0;
    for (int s = 0; s < kDist; ++s) nd += sm.len_d[s] > 0;
    if (!nd) sm.len_d[0] = 1;                  // no match: one unused distance code of length 1
    int hlit = kLL, hdist = kDist;
    while (hlit > 257 && !sm.len_ll[hlit - 1]) --hlit;
    while (hdist > 1 && !sm.len_d[hdist - 1]) --hdist;
    sm.hlit = hlit; sm.hdist = hdist;
    for (int s = 0; s < kCL; ++s) sm.freq_cl[s] = 0;
    const int total = hlit + hdist;
    auto lens = [&](int i) { return i < hlit ? sm.len_ll[i] : sm.len_d[i - hlit]; };
    int nr = 0;
    auto emit = [&](int sym, int x) { sm.rle[nr++] = (uint16_t)(sym | (x << 5)); ++sm.freq_cl[sym]; };
    for (int i = 0; i < total;) {
      const int v = lens(i);
      int run = 1;
      while (i + run < total && lens(i + run) == v) ++run;
      i += run;
      if (v == 0) {
        while (run >= 11) { const int r = min(run, 138); emit(18, r - 11); run -= r; }
        if (run >= 3) { emit(17, run - 3); run = 0; }
        while (run > 0) { emit(0, 0); --run; }
      } else {
        emit(v, 0); --run;
        while (run >= 3) { const int r = min(run, 6); emit(16, r - 3); run -= r; }
        while (run > 0) { emit(v, 0); --run; }
      }
    }
    sm.nrle = nr;
    int used = 0;
    for (int s = 0; s < kCL; ++s) used += sm.freq_cl[s] > 0;
    if (used < 2) sm.freq_cl[sm.freq_cl[0] ? 1 : 0] = 1;   // zlib rejects an incomplete code-length code
  }
  __syncwarp();
  huffman_lengths(sm.freq_cl, kCL, 7, sm.len_cl, sm.sort, sm.num, lane);
  if (lane == 0) {
    canonical_codes(sm.len_ll, kLL, sm.code_ll, sm.num, sm.next);
    canonical_codes(sm.len_d, kDist, sm.code_d, sm.num, sm.next);
    canonical_codes(sm.len_cl, kCL, sm.code_cl, sm.num, sm.next);
    int hclen = kCL;
    while (hclen > 4 && !sm.len_cl[kCLOrder[hclen - 1]]) --hclen;
    sm.hclen = hclen;
    int64_t bits = 3 + 14 + 3 * hclen;
    for (int r = 0; r < sm.nrle; ++r) {
      const int sym = sm.rle[r] & 31;
      bits += sm.len_cl[sym] + (sym == 16 ? 2 : sym == 17 ? 3 : sym == 18 ? 7 : 0);
    }
    sm.hdr_bits = bits;
  }
  __syncwarp();

  // pass 2: this lane's bits, offsets by a warp scan
  const int dfar_bits = sm.len_d[fdc] + feb, dnear_bits = sm.len_d[0];
  int64_t mybits = 0;
  parse(raw, bm1, bmS, B0, start, e_nom, B1, [&](int lit, int l, bool far) {
    if (!l) { mybits += sm.len_ll[lit]; return; }
    int lc, eb, ev;
    len_code(l, lc, eb, ev);
    mybits += sm.len_ll[257 + lc] + eb + (far ? dfar_bits : dnear_bits);
  });
  int64_t incl = mybits;
  for (int o = 1; o < 32; o <<= 1) {
    const int64_t v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  const int64_t tok_end = sm.hdr_bits + __shfl_sync(0xffffffffu, incl, 31);
  const int64_t eob_end = tok_end + sm.len_ll[256];
  const int64_t sync_byte = (eob_end + 3 + 7) / 8;  // empty stored block: 3 header bits, byte alignment, 00 00 FF FF
  const int64_t comp = final_band ? (eob_end + 7) / 8 : sync_byte + 4;
  const int64_t stored = stored_bytes(L);

  if (comp > stored) {
    // stored blocks of <= 65535 bytes
    const int64_t nblk = (L + kStoredMax - 1) / kStoredMax;
    for (int64_t k = 0; k < nblk; ++k) {
      const int64_t off = k * (kStoredMax + 5), src = B0 + k * kStoredMax, len = min(kStoredMax, B1 - src);
      if (lane == 0) {
        slot[off] = (final_band && k == nblk - 1) ? 1 : 0;
        slot[off + 1] = (uint8_t)len; slot[off + 2] = (uint8_t)(len >> 8);
        slot[off + 3] = (uint8_t)~len; slot[off + 4] = (uint8_t)(~len >> 8);
      }
      for (int64_t i = lane; i < len; i += 32) slot[off + 5 + i] = __ldg(raw + src + i);
    }
  } else {
    // pass 3: write the block
    for (int64_t w = lane; w < (comp + 3) / 4; w += 32) slot32[w] = 0;
    __syncwarp();
    if (lane == 0) {
      BitWriter bw(slot32, 0);
      bw.put(final_band ? 1 : 0, 1); bw.put(2, 2);
      bw.put(sm.hlit - 257, 5); bw.put(sm.hdist - 1, 5); bw.put(sm.hclen - 4, 4);
      for (int k = 0; k < sm.hclen; ++k) bw.put(sm.len_cl[kCLOrder[k]], 3);
      for (int r = 0; r < sm.nrle; ++r) {
        const int sym = sm.rle[r] & 31, x = sm.rle[r] >> 5;
        bw.put(sm.code_cl[sym], sm.len_cl[sym]);
        if (sym == 16) bw.put(x, 2);
        else if (sym == 17) bw.put(x, 3);
        else if (sym == 18) bw.put(x, 7);
      }
      bw.flush();
    }
    BitWriter bw(slot32, sm.hdr_bits + incl - mybits);
    parse(raw, bm1, bmS, B0, start, e_nom, B1, [&](int lit, int l, bool far) {
      if (!l) { bw.put(sm.code_ll[lit], sm.len_ll[lit]); return; }
      int lc, eb, ev;
      len_code(l, lc, eb, ev);
      bw.put(sm.code_ll[257 + lc], sm.len_ll[257 + lc]);
      if (eb) bw.put(ev, eb);
      if (far) { bw.put(sm.code_d[fdc], sm.len_d[fdc]); if (feb) bw.put(fev, feb); }
      else bw.put(sm.code_d[0], sm.len_d[0]);
    });
    bw.flush();
    if (lane == 0) {
      BitWriter tail(slot32, tok_end);
      tail.put(sm.code_ll[256], sm.len_ll[256]);
      tail.flush();
      if (!final_band) {
        BitWriter ff(slot32, (sync_byte + 2) * 8);
        ff.put(0xffffu, 16);
        ff.flush();
      }
    }
  }
  if (lane == 0) {
    int64_t* o = info + (int64_t)blockIdx.x * 4;
    o[0] = comp > stored ? stored : comp;
    o[1] = (int64_t)s1; o[2] = (int64_t)s2; o[3] = 0;
  }
}

// Per image: band offsets within the zlib data (info[.][3]), the file size into sizes[img + 1], the Adler-32.
__global__ void __launch_bounds__(32) png_size_kernel(Plan p, int64_t extra, int64_t* __restrict__ info,
                                                      int64_t* __restrict__ sizes, uint32_t* __restrict__ adler) {
  const int lane = threadIdx.x;
  const int64_t img = blockIdx.x;
  int64_t* inf = info + img * p.nb * 4;
  int64_t carry = 2;                           // after the zlib header
  uint64_t A = 0, B = 0;
  for (int64_t b0 = 0; b0 < p.nb; b0 += 32) {
    const int64_t b = b0 + lane;
    int64_t bytes = 0;
    if (b < p.nb) {
      bytes = inf[b * 4];
      const int64_t band_end = min(p.n, (b + 1) * p.R * p.S);
      const uint64_t a1 = (uint64_t)inf[b * 4 + 1], a2 = (uint64_t)inf[b * 4 + 2];
      A += a1;
      B += a2 + a1 * ((uint64_t)(p.n - band_end) % kAdlerMod);
      A %= kAdlerMod; B %= kAdlerMod;
    }
    int64_t incl = bytes;
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (b < p.nb) inf[b * 4 + 3] = carry + incl - bytes;
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
  for (int o = 16; o; o >>= 1) {
    A += __shfl_xor_sync(0xffffffffu, A, o);
    B += __shfl_xor_sync(0xffffffffu, B, o);
  }
  if (lane == 0) {
    const uint64_t s1 = (1 + A) % kAdlerMod, s2 = ((uint64_t)p.n % kAdlerMod + B) % kAdlerMod;
    adler[img] = (uint32_t)(s2 << 16 | s1);
    sizes[img + 1] = carry - 2 + kFileOverhead + extra;
  }
}

// offsets[0] = 0, offsets[i + 1] = offsets[i] + sizes[i + 1] (in place), one block of 1024
__global__ void __launch_bounds__(1024) png_scan_kernel(int64_t* __restrict__ offsets, int N) {
  __shared__ int64_t warp_sum[32];
  __shared__ int64_t carry_s;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) { carry_s = 0; offsets[0] = 0; }
  __syncthreads();
  for (int base = 0; base < N; base += 1024) {
    const int i = base + t;
    int64_t v = i < N ? offsets[i + 1] : 0;
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += u;
    }
    if (lane == 31) warp_sum[wid] = v;
    __syncthreads();
    if (wid == 0) {
      int64_t w = warp_sum[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const int64_t u = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += u;
      }
      warp_sum[lane] = w;
    }
    __syncthreads();
    const int64_t total = carry_s + v + (wid ? warp_sum[wid - 1] : 0);
    if (i < N) offsets[i + 1] = total;
    __syncthreads();
    if (t == 1023) carry_s = total;
    __syncthreads();
  }
}

__device__ __forceinline__ void put_be32(uint8_t* p, uint32_t v) {
  p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// palette_crc: the CRC-32 of the grey PLTE chunk (type and data), 0 for a file without one
__global__ void __launch_bounds__(256) png_assemble_kernel(Plan p, int H, int W, int color_type, uint32_t palette_crc,
                                                           const uint8_t* __restrict__ slots,
                                                           const int64_t* __restrict__ info,
                                                           const uint32_t* __restrict__ adler,
                                                           const int64_t* __restrict__ offsets, uint8_t* __restrict__ out) {
  __shared__ uint32_t tab[256], x2n[32], crc_s[256];
  __shared__ int64_t len_s[256];
  const int t = threadIdx.x;
  const int64_t img = blockIdx.x;
  const int64_t pre = palette_crc ? kPlteChunk : 0;        // bytes before the IDAT chunk move by the PLTE chunk
  uint8_t* f = out + offsets[img];
  const int64_t size = offsets[img + 1] - offsets[img];
  const int64_t idat_len = size - pre - kFileOverhead + 2 + 4;   // zlib header + deflate data + Adler-32
  tab[t] = crc_table_entry((uint32_t)t);
  if (pre) {
    uint8_t* c = f + 33;
    if (t == 0) {
      put_be32(c, 768);
      c[4] = 'P'; c[5] = 'L'; c[6] = 'T'; c[7] = 'E';
      put_be32(c + 8 + 768, palette_crc);
    }
    for (int k = 0; k < 3; ++k) c[8 + 3 * t + k] = (uint8_t)t;
  }
  f += pre;                                                // from here on f is the file shifted by the PLTE chunk
  __syncthreads();
  if (t == 0) {
    crc_x2n_table(x2n);
    uint8_t* f0 = f - pre;
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    for (int k = 0; k < 8; ++k) f0[k] = sig[k];
    uint8_t* h = f0 + 8;
    put_be32(h, 13);
    h[4] = 'I'; h[5] = 'H'; h[6] = 'D'; h[7] = 'R';
    put_be32(h + 8, (uint32_t)W); put_be32(h + 12, (uint32_t)H);
    // bit depth 8, grayscale (0), RGB (2) or palette (3), deflate, filter method 0, no interlace
    h[16] = 8; h[17] = (uint8_t)color_type; h[18] = 0; h[19] = 0; h[20] = 0;
    put_be32(h + 21, ~crc_update(tab, 0xffffffffu, h + 4, 17));
    uint8_t* d = f + 33;
    put_be32(d, (uint32_t)idat_len);
    d[4] = 'I'; d[5] = 'D'; d[6] = 'A'; d[7] = 'T';
    d[8] = 0x78; d[9] = 0x01;
    put_be32(f + kIdatData + idat_len - 4, adler[img]);
    uint8_t* e = f + size - pre - 12;
    put_be32(e, 0);
    e[4] = 'I'; e[5] = 'E'; e[6] = 'N'; e[7] = 'D';
    put_be32(e + 8, 0xae426082u);
  }
  const int64_t* inf = info + img * p.nb * 4;
  const uint8_t* sl = slots + img * p.nb * p.band_cap;
  for (int64_t b = 0; b < p.nb; ++b) {
    const int64_t bytes = inf[b * 4], dst = kIdatData + inf[b * 4 + 3];
    const uint8_t* src = sl + b * p.band_cap;
    for (int64_t i = t; i < bytes; i += 256) f[dst + i] = src[i];
  }
  __syncthreads();
  // CRC-32 of "IDAT" + data: contiguous chunks per thread, merged pairwise
  const int64_t clen = 4 + idat_len, per = (clen + 255) / 256;
  const int64_t c0 = min(clen, t * per), c1 = min(clen, c0 + per);
  const uint8_t* q = f + 37;
  crc_s[t] = ~crc_update(tab, 0xffffffffu, q + c0, c1 - c0); len_s[t] = c1 - c0;
  __syncthreads();
  for (int s = 1; s < 256; s <<= 1) {
    if ((t & (2 * s - 1)) == 0) {
      crc_s[t] = crc_combine(crc_s[t], crc_s[t + s], len_s[t + s], x2n);
      len_s[t] += len_s[t + s];
    }
    __syncthreads();
  }
  if (t == 0) put_be32(f + 37 + clen, crc_s[0]);
}

// Everything after the filter kernel, which the caller has launched into the workspace.
int encode_filtered(const Plan& p, int N, int H, int W, int color_type, uint32_t palette_crc, uint8_t* out,
                    int64_t* offsets, uint8_t* ws, cudaStream_t st) {
  uint8_t* slots = ws + p.slot_off;
  int64_t* info = (int64_t*)(ws + p.info_off);
  uint32_t* adler = (uint32_t*)(ws + p.adler_off);
  png_band_kernel<<<(unsigned)(N * p.nb), 32, 0, st>>>(ws, p, slots, info, (uint32_t*)(ws + p.bm_off));
  LEDB_LAUNCH_OK("png_band_kernel");
  png_size_kernel<<<(unsigned)N, 32, 0, st>>>(p, palette_crc ? kPlteChunk : 0, info, offsets, adler);
  LEDB_LAUNCH_OK("png_size_kernel");
  png_scan_kernel<<<1, 1024, 0, st>>>(offsets, N);
  LEDB_LAUNCH_OK("png_scan_kernel");
  png_assemble_kernel<<<(unsigned)N, 256, 0, st>>>(p, H, W, color_type, palette_crc, slots, info, adler, offsets, out);
  LEDB_LAUNCH_OK("png_assemble_kernel");
  return LEDB200_OK;
}

int64_t checked_bound(int32_t H, int32_t W, int C, const char* who) {
  if (H < 1 || W < 1) return fail(LEDB200_EINVAL, std::string(who) + ": H and W must be at least 1");
  const int64_t b = bound_of(make_plan(1, H, W, C));
  if (b - 8 - 25 - 12 - 12 > INT32_MAX)
    return fail(LEDB200_EINVAL, std::string(who) + ": the image is too large for one IDAT chunk");
  return b;
}

}  // namespace
}  // namespace ledb

using namespace ledb;

extern "C" {

int64_t ledb200_png_bound(int32_t H, int32_t W) { return checked_bound(H, W, 1, "png_bound"); }

int64_t ledb200_png_rgb_bound(int32_t H, int32_t W) { return checked_bound(H, W, 3, "png_rgb_bound"); }

int64_t ledb200_png_lut_bound(int32_t H, int32_t W, int32_t palette) {
  if (palette != 0 && palette != 1) return fail(LEDB200_EINVAL, "png_lut_bound: palette must be 0 or 1");
  const int64_t b = ledb200_png_bound(H, W);
  return b < 0 ? b : b + (palette ? kPlteChunk : 0);
}

int64_t ledb200_png_workspace_bytes(int32_t N, int32_t H, int32_t W) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "png_workspace_bytes: N, H and W must be at least 1");
  return make_plan(N, H, W, 1).total;
}

int64_t ledb200_png_rgb_workspace_bytes(int32_t N, int32_t H, int32_t W) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "png_rgb_workspace_bytes: N, H and W must be at least 1");
  return make_plan(N, H, W, 3).total;
}

int ledb200_png_encode_lut(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, const uint8_t* lut,
                           int32_t palette, uint8_t* out, int64_t* offsets, void* workspace, void* stream) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "png_encode: N, H and W must be at least 1");
  if (dtype != LEDB200_U8 && dtype != LEDB200_I64) return fail(LEDB200_EINVAL, "png_encode: labels must be U8 or I64");
  if (palette != 0 && palette != 1) return fail(LEDB200_EINVAL, "png_encode: palette must be 0 or 1");
  if (!labels || !lut || !out || !offsets || !workspace) return fail(LEDB200_EINVAL, "png_encode: null buffer");
  if (ledb200_png_bound(H, W) < 0) return LEDB200_EINVAL;
  const Plan p = make_plan(N, H, W, 1);
  if ((int64_t)N * p.nb > INT32_MAX) return fail(LEDB200_EINVAL, "png_encode: too many bands in one call");
  // the grey palette's CRC is the same for every file: computed here once
  static const uint32_t palette_crc = [] {
    uint32_t tab[256];
    for (uint32_t i = 0; i < 256; ++i) tab[i] = crc_table_entry(i);
    uint8_t chunk[4 + 768] = {'P', 'L', 'T', 'E'};
    for (int i = 0; i < 768; ++i) chunk[4 + i] = (uint8_t)(i / 3);
    return ~crc_update(tab, 0xffffffffu, chunk, sizeof chunk);
  }();
  Lut tab;
  for (int i = 0; i < 256; ++i) tab.v[i] = lut[i];
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  const unsigned rows = (unsigned)((int64_t)N * H);
  if (dtype == LEDB200_I64) png_filter_kernel<int64_t><<<rows, 256, 0, st>>>((const int64_t*)labels, W, p.S, tab, ws);
  else png_filter_kernel<uint8_t><<<rows, 256, 0, st>>>((const uint8_t*)labels, W, p.S, tab, ws);
  LEDB_LAUNCH_OK("png_filter_kernel");
  return encode_filtered(p, N, H, W, palette ? 3 : 0, palette ? palette_crc : 0u, out, offsets, ws, st);
}

int ledb200_png_encode_rgb(const uint8_t* rgb, int32_t N, int32_t H, int32_t W, uint8_t* out, int64_t* offsets,
                           void* workspace, void* stream) {
  if (N < 1 || H < 1 || W < 1) return fail(LEDB200_EINVAL, "png_encode_rgb: N, H and W must be at least 1");
  if (!rgb || !out || !offsets || !workspace) return fail(LEDB200_EINVAL, "png_encode_rgb: null buffer");
  if (ledb200_png_rgb_bound(H, W) < 0) return LEDB200_EINVAL;
  const Plan p = make_plan(N, H, W, 3);
  if ((int64_t)N * p.nb > INT32_MAX) return fail(LEDB200_EINVAL, "png_encode_rgb: too many bands in one call");
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  png_filter_rgb_kernel<<<(unsigned)((int64_t)N * H), 256, 0, st>>>(rgb, H, W, p.S, ws);
  LEDB_LAUNCH_OK("png_filter_rgb_kernel");
  return encode_filtered(p, N, H, W, 2, 0u, out, offsets, ws, st);
}

int ledb200_png_encode(const void* labels, int32_t dtype, int32_t N, int32_t H, int32_t W, int32_t add, uint8_t* out,
                       int64_t* offsets, void* workspace, void* stream) {
  if (add != 0 && add != 1) return fail(LEDB200_EINVAL, "png_encode: add must be 0 or 1");
  uint8_t lut[256];
  for (int i = 0; i < 256; ++i) lut[i] = (uint8_t)(i + add);
  return ledb200_png_encode_lut(labels, dtype, N, H, W, lut, 0, out, offsets, workspace, stream);
}

}  // extern "C"
