// Baseline JPEG decode for the batch feeder: file bytes -> packed HWC uint8 RGB, bit-identical to Pillow's
// `Image.open(f).convert("RGB")` (Pillow 12.2 over libjpeg-turbo 3.1) for the streams of the device subset; everything else
// is decoded by Pillow on the host (xfm_b200/feed.py).
//
// Host (xfm_jpeg_plan / xfm_jpeg_tables): marker walk by segment lengths, every length checked against the blob, the
// supported / fallback decision, quantisation tables, canonical Huffman decode tables, component geometry and the byte range
// of every restart interval.  Device (xfm_jpeg_decode), three launches on the caller's stream, no host synchronisation:
//   1. jpeg_entropy_kernel  one thread per restart interval (one per image without DRI): Huffman decode into int16 blocks;
//   2. jpeg_idct_kernel     one thread per 8x8 block: dequantise + ISLOW IDCT into component planes;
//   3. jpeg_color_kernel    one thread per output pixel: fancy upsampling + YCbCr -> RGB into the caller's ragged layout.
// The arithmetic is the one Pillow's libjpeg-turbo runs on x86-64 (tests/jpeg_ref.py restates it in numpy and is compared
// with Pillow byte for byte; DESIGN.md §8 lists where it differs from libjpeg-turbo's C code).
#include <algorithm>
#include <cstring>
#include <thread>
#include <vector>
#include "common.cuh"
#include "internal.h"

namespace xfm {

struct HuffTab {
  uint16_t look[512];    // first 9 bits of the window -> (code length << 8) | symbol; 0 = the code is longer (or invalid)
  int32_t maxcode[18];   // largest code of each length 1..16, -1 if none; [17] = sentinel
  int32_t valoff[17];    // symbol = val[code + valoff[length]]
  uint8_t val[256];
};

struct JpegDesc {
  HuffTab tab[4];        // DC table 0, DC table 1, AC table 0, AC table 1
  uint16_t qt[3][64];    // per component, natural order
  int64_t blob_off, coef_off, plane_off, out_off, first_interval;
  int64_t comp_coef[4];  // first block of each component (relative to coef_off); [ncomp] = block count of the image
  int64_t comp_plane[3]; // byte offset of each component plane (relative to plane_off)
  int32_t W, H, ncomp, mcux, n_int, mcus_per_int, total_mcus;
  int32_t h[3], v[3], bw[3], dw[3], dh[3], dct[3], act[3];
};
static_assert(sizeof(HuffTab) * 4 % 16 == 0 && sizeof(JpegDesc) % 16 == 0, "JpegDesc layout");

enum JpegStatus {
  J_OK = 0, J_NOT_JPEG = 1, J_MALFORMED = 2, J_CODING = 3, J_COLOR = 4, J_SAMPLING = 5, J_TABLES = 6, J_SCAN = 7,
  J_RESTART = 8, J_SIZE = 9,
  // set on the device (OR-ed)
  J_BAD_CODE = 16, J_BAD_RUN = 32, J_SHORT_DATA = 64, J_MARKER = 128,
};

static const uint8_t kZigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                    41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                    30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

// ------------------------------------------------------------------------------------------------------------ host parser
struct Parsed {
  int W = 0, H = 0, ncomp = 0, dri = 0;
  int id[3], h[3], v[3], tq[3], td[3], ta[3];
  bool jfif = false;
  int adobe = -1;
  bool qdef[4] = {false, false, false, false};
  uint16_t qt[4][64];
  bool hdef[4] = {false, false, false, false};   // DC0 DC1 AC0 AC1
  uint8_t counts[4][16];
  uint8_t syms[4][256];
  int64_t ecs_begin = 0, ecs_end = 0;
  int64_t n_int = 0, mcux = 0, mcuy = 0, hmax = 1, vmax = 1;
};

static int rd16(const uint8_t* p) { return (p[0] << 8) | p[1]; }

// jpeg_make_d_derived_tbl's checks: a code never exceeds its length; DC symbols <= 15.
static bool huff_valid(const uint8_t* counts, const uint8_t* syms, bool dc) {
  int maxlen = 0, k = 0;
  for (int l = 1; l <= 16; ++l)
    if (counts[l - 1]) maxlen = l;
  int64_t code = 0;
  for (int l = 1; l <= maxlen; ++l) {
    code += counts[l - 1];
    k += counts[l - 1];
    if (code >= (int64_t(1) << l)) return false;
    code <<= 1;
  }
  if (k > 256) return false;
  if (dc)
    for (int i = 0; i < k; ++i)
      if (syms[i] > 15) return false;
  return true;
}

// Walk one blob.  ivals (optional): the byte range [begin, end) of every restart interval, relative to the blob.
static int parse_jpeg(const uint8_t* b, int64_t n, Parsed& P, int64_t* ivals) {
  if (n < 4 || b[0] != 0xFF || b[1] != 0xD8) return J_NOT_JPEG;
  int64_t p = 2;
  bool sof = false;
  for (;;) {
    if (p >= n || b[p] != 0xFF) return J_MALFORMED;      // libjpeg skips (and warns about) garbage; Pillow decides
    while (p < n && b[p] == 0xFF) ++p;                   // fill bytes before a marker
    if (p + 3 > n) return J_MALFORMED;
    const int m = b[p++];
    if (!((m >= 0xC0 && m <= 0xFE) && !(m >= 0xD0 && m <= 0xD9))) return J_MALFORMED;   // standalone / reserved markers
    const int L = rd16(b + p);
    if (L < 2 || p + L > n) return J_MALFORMED;
    const uint8_t* s = b + p + 2;
    const int len = L - 2;
    if (m == 0xE0) {
      if (len >= 14 && !memcmp(s, "JFIF", 5)) P.jfif = true;
    } else if (m == 0xEE) {
      if (len >= 12 && !memcmp(s, "Adobe", 5)) P.adobe = s[11];
    } else if (m == 0xDB) {
      for (int i = 0; i < len;) {
        const int pq = s[i] >> 4, tq = s[i] & 15;
        if (pq != 0) return J_CODING;                   // 16-bit tables: not in the device subset
        if (tq > 3 || i + 65 > len) return J_TABLES;
        for (int k = 0; k < 64; ++k) P.qt[tq][kZigzag[k]] = s[i + 1 + k];
        P.qdef[tq] = true;
        i += 65;
      }
    } else if (m == 0xC4) {
      for (int i = 0; i < len;) {
        const int tc = s[i] >> 4, th = s[i] & 15;
        if (tc > 1 || th > 1 || i + 17 > len) return J_TABLES;
        int cnt = 0;
        for (int l = 0; l < 16; ++l) cnt += s[i + 1 + l];
        if (cnt > 256 || i + 17 + cnt > len) return J_TABLES;
        const int t = tc * 2 + th;
        memcpy(P.counts[t], s + i + 1, 16);
        memcpy(P.syms[t], s + i + 17, cnt);
        if (!huff_valid(P.counts[t], P.syms[t], tc == 0)) return J_TABLES;
        P.hdef[t] = true;
        i += 17 + cnt;
      }
    } else if (m == 0xDD) {
      if (len != 2) return J_MALFORMED;
      P.dri = rd16(s);
    } else if (m == 0xC0 || m == 0xC1) {
      if (sof) return J_SCAN;
      sof = true;
      if (len < 6) return J_MALFORMED;
      if (s[0] != 8) return J_CODING;
      P.H = rd16(s + 1);
      P.W = rd16(s + 3);
      P.ncomp = s[5];
      if (P.W == 0 || P.H == 0) return J_SIZE;
      if (P.ncomp != 1 && P.ncomp != 3) return J_COLOR;
      if (len != 6 + 3 * P.ncomp) return J_MALFORMED;       // libjpeg: JERR_BAD_LENGTH
      for (int c = 0; c < P.ncomp; ++c) {
        P.id[c] = s[6 + 3 * c];
        P.h[c] = s[7 + 3 * c] >> 4;
        P.v[c] = s[7 + 3 * c] & 15;
        P.tq[c] = s[8 + 3 * c];
        if (P.h[c] < 1 || P.h[c] > 4 || P.v[c] < 1 || P.v[c] > 4 || P.tq[c] > 3) return J_SAMPLING;
      }
    } else if (m == 0xDA) {
      if (!sof) return J_SCAN;
      if (len < 1 || s[0] != P.ncomp || len != 4 + 2 * P.ncomp) return J_SCAN;   // one scan with every component
      for (int c = 0; c < P.ncomp; ++c) {
        if (s[1 + 2 * c] != P.id[c]) return J_SCAN;
        P.td[c] = s[2 + 2 * c] >> 4;
        P.ta[c] = s[2 + 2 * c] & 15;
        if (P.td[c] > 1 || P.ta[c] > 1 || !P.hdef[P.td[c]] || !P.hdef[2 + P.ta[c]]) return J_TABLES;
        if (!P.qdef[P.tq[c]]) return J_TABLES;
      }
      if (s[1 + 2 * P.ncomp] != 0 || s[2 + 2 * P.ncomp] != 63 || s[3 + 2 * P.ncomp] != 0) return J_CODING;
      // libjpeg's default_decompress_parms: JFIF -> YCbCr; else Adobe transform 0 -> RGB; else IDs 'R' 'G' 'B' -> RGB.
      if (P.ncomp == 3 && !P.jfif) {
        if (P.adobe == 0) return J_COLOR;
        if (P.adobe < 0 && P.id[0] == 82 && P.id[1] == 71 && P.id[2] == 66) return J_COLOR;
      }
      P.hmax = P.vmax = 1;
      for (int c = 0; c < P.ncomp; ++c) { P.hmax = std::max<int64_t>(P.hmax, P.h[c]); P.vmax = std::max<int64_t>(P.vmax, P.v[c]); }
      if (P.ncomp == 1) {
        P.h[0] = P.v[0] = 1;                           // a single-component scan is not interleaved: one block per MCU
        P.hmax = P.vmax = 1;
      }
      int bpm = 0;
      for (int c = 0; c < P.ncomp; ++c) {
        if (P.hmax % P.h[c] || P.vmax % P.v[c]) return J_SAMPLING;
        const int fh = (int)(P.hmax / P.h[c]), fv = (int)(P.vmax / P.v[c]);
        if (!((fh == 1 && fv == 1) || (fh == 2 && fv == 1) || (fh == 2 && fv == 2))) return J_SAMPLING;
        bpm += P.h[c] * P.v[c];
      }
      if (bpm > 10) return J_SAMPLING;
      P.mcux = (P.W + 8 * P.hmax - 1) / (8 * P.hmax);
      P.mcuy = (P.H + 8 * P.vmax - 1) / (8 * P.vmax);
      const int64_t total = P.mcux * P.mcuy, ri = P.dri ? P.dri : total;
      P.n_int = (total + ri - 1) / ri;
      // Entropy-coded segment: up to the first marker other than RSTn; RSTn in sequence, exactly n_int - 1 of them; EOI after.
      P.ecs_begin = p + L;
      int64_t q = P.ecs_begin, k = 0, begin = P.ecs_begin;
      for (;;) {
        const uint8_t* f = (const uint8_t*)memchr(b + q, 0xFF, (size_t)(n - q));
        if (!f || f + 1 >= b + n) return J_SCAN;         // truncated: no marker ends the scan
        q = f - b;
        const int c = b[q + 1];
        if (c == 0x00) { q += 2; continue; }
        if (c >= 0xD0 && c <= 0xD7) {
          if (c - 0xD0 != (k & 7) || k + 1 >= P.n_int) return J_RESTART;
          if (ivals) { ivals[2 * k] = begin; ivals[2 * k + 1] = q; }
          ++k;
          q += 2;
          begin = q;
          continue;
        }
        if (c != 0xD9) return J_SCAN;                    // fill bytes, another scan, DNL, ...
        if (k + 1 != P.n_int) return J_RESTART;
        if (ivals) { ivals[2 * k] = begin; ivals[2 * k + 1] = q; }
        P.ecs_end = q;
        return J_OK;
      }
    } else if (m >= 0xC0 && m <= 0xCF && m != 0xC4) {
      return J_CODING;                                   // progressive, lossless, arithmetic, hierarchical
    } else if (!(m >= 0xE0 && m <= 0xEF) && m != 0xFE) {
      return J_MALFORMED;                                // DNL, EXP, JPGn, ... (not in the device subset)
    }
    p += L;
  }
}

static void plan_geometry(const Parsed& P, int64_t* blocks, int64_t* plane_bytes) {
  int64_t nb = 0, pb = 0;
  for (int c = 0; c < P.ncomp; ++c) {
    const int64_t bw = P.mcux * P.h[c], bh = P.mcuy * P.v[c];
    nb += bw * bh;
    pb += bw * bh * 64;
  }
  *blocks = nb;
  *plane_bytes = pb;
}

static void fill_huff(HuffTab& t, const uint8_t* counts, const uint8_t* syms) {
  memset(&t, 0, sizeof(t));
  int code = 0, k = 0;
  for (int l = 1; l <= 16; ++l) {
    t.valoff[l] = k - code;
    for (int i = 0; i < counts[l - 1]; ++i, ++k, ++code) {
      if (l <= 9)
        for (int j = 0; j < (1 << (9 - l)); ++j) t.look[(code << (9 - l)) | j] = (uint16_t)((l << 8) | syms[k]);
    }
    t.maxcode[l] = counts[l - 1] ? code - 1 : -1;
    code <<= 1;
  }
  t.maxcode[17] = 0x7fffffff;
  memcpy(t.val, syms, 256);
}

template <class F>
static void parallel_for(int n, int threads, F f) {
  int T = std::max(1, std::min(threads, n));
  if (T <= 1) { for (int i = 0; i < n; ++i) f(i); return; }
  std::vector<std::thread> pool;
  for (int t = 0; t < T; ++t)
    pool.emplace_back([=, &f] { for (int i = (int)((int64_t)n * t / T); i < (int)((int64_t)n * (t + 1) / T); ++i) f(i); });
  for (auto& th : pool) th.join();
}

int jpeg_plan(const void* const* blobs, const int64_t* nbytes, int n, int64_t* info, int threads) {
  if (n < 0 || (n > 0 && (!blobs || !nbytes || !info))) { set_error("jpeg_plan: null pointer"); return XFM_ERR_BAD_ARG; }
  for (int i = 0; i < n; ++i)
    if (nbytes[i] < 0 || (nbytes[i] > 0 && !blobs[i])) { set_error("jpeg_plan: bad blob %d", i); return XFM_ERR_BAD_ARG; }
  parallel_for(n, threads, [&](int i) {
    Parsed P;
    int64_t* r = info + (int64_t)i * XFM_JPEG_INFO;
    memset(r, 0, sizeof(int64_t) * XFM_JPEG_INFO);
    const int st = parse_jpeg((const uint8_t*)blobs[i], nbytes[i], P, nullptr);
    r[0] = st;
    r[1] = P.W;
    r[2] = P.H;
    if (st == J_OK) {
      r[3] = P.n_int;
      plan_geometry(P, &r[4], &r[5]);
    }
  });
  return 0;
}

int jpeg_tables(const void* const* blobs, const int64_t* nbytes, int n, const int64_t* info, const int64_t* offs, void* desc,
                int64_t* intervals, int threads) {
  if (n < 0 || (n > 0 && (!blobs || !nbytes || !info || !offs || !desc))) { set_error("jpeg_tables: null pointer"); return XFM_ERR_BAD_ARG; }
  std::vector<int64_t> first(n + 1, 0);
  for (int i = 0; i < n; ++i) first[i + 1] = first[i] + (info[(int64_t)i * XFM_JPEG_INFO] == J_OK ? info[(int64_t)i * XFM_JPEG_INFO + 3] : 0);
  if (first[n] > 0 && !intervals) { set_error("jpeg_tables: null intervals"); return XFM_ERR_BAD_ARG; }
  std::vector<int> bad(n, 0);
  parallel_for(n, threads, [&](int i) {
    JpegDesc& d = ((JpegDesc*)desc)[i];
    memset(&d, 0, sizeof(d));
    const int64_t* r = info + (int64_t)i * XFM_JPEG_INFO;
    const int64_t* o = offs + (int64_t)i * 4;
    d.out_off = o[3];
    if (r[0] != J_OK) return;                            // n_int = 0: every kernel skips the image
    Parsed P;
    if (parse_jpeg((const uint8_t*)blobs[i], nbytes[i], P, intervals + 2 * first[i]) != J_OK || P.n_int != r[3]) { bad[i] = 1; return; }
    for (int64_t k = 0; k < P.n_int; ++k) {
      intervals[2 * (first[i] + k)] += o[0];
      intervals[2 * (first[i] + k) + 1] += o[0];
    }
    for (int t = 0; t < 4; ++t)
      if (P.hdef[t]) fill_huff(d.tab[t], P.counts[t], P.syms[t]);
    d.blob_off = o[0];
    d.coef_off = o[1];
    d.plane_off = o[2];
    d.first_interval = first[i];
    d.W = P.W;
    d.H = P.H;
    d.ncomp = P.ncomp;
    d.mcux = (int32_t)P.mcux;
    d.n_int = (int32_t)P.n_int;
    d.total_mcus = (int32_t)(P.mcux * P.mcuy);
    d.mcus_per_int = P.dri ? P.dri : d.total_mcus;
    int64_t cb = 0, pb = 0;
    for (int c = 0; c < P.ncomp; ++c) {
      memcpy(d.qt[c], P.qt[P.tq[c]], sizeof(d.qt[c]));
      d.h[c] = P.h[c];
      d.v[c] = P.v[c];
      d.bw[c] = (int32_t)(P.mcux * P.h[c]);
      d.dw[c] = (int32_t)((P.W * P.h[c] + P.hmax - 1) / P.hmax);    // libjpeg's downsampled_width / _height
      d.dh[c] = (int32_t)((P.H * P.v[c] + P.vmax - 1) / P.vmax);
      d.dct[c] = P.td[c];
      d.act[c] = 2 + P.ta[c];
      d.comp_coef[c] = cb;
      d.comp_plane[c] = pb;
      const int64_t nbk = (int64_t)d.bw[c] * P.mcuy * P.v[c];
      cb += nbk;
      pb += nbk * 64;
    }
    d.comp_coef[P.ncomp] = cb;
  });
  for (int i = 0; i < n; ++i)
    if (bad[i]) { set_error("jpeg_tables: image %d does not match its plan", i); return XFM_ERR_BAD_ARG; }
  return 0;
}

// ------------------------------------------------------------------------------------------------------- 1. entropy decode
// Bit reader over [p, end): 0xFF00 -> 0xFF; past the end it feeds zero bits (as libjpeg does) and counts them, so that a
// read that consumed any of them is detected.  No byte outside [p, end) is ever read.
struct BitReader {
  const uint8_t* p;
  const uint8_t* end;
  uint64_t acc;
  int nbits, pad;
  int status;
  XFM_DEVINL void fill() {
    while (nbits <= 56) {
      uint32_t c = 0;
      if (p < end) {
        c = *p++;
        if (c == 0xFF) {
          if (p < end && *p == 0x00) ++p;
          else { status |= J_MARKER; p = end; c = 0; pad += 8; }
        }
      } else {
        pad += 8;
      }
      acc = (acc << 8) | c;
      nbits += 8;
    }
  }
  XFM_DEVINL uint32_t peek16() { return (uint32_t)(acc >> (nbits - 16)) & 0xFFFFu; }
  XFM_DEVINL void skip(int n) { nbits -= n; }
  XFM_DEVINL int get(int s) {            // s <= 16; caller has filled
    const int v = (int)((acc >> (nbits - s)) & ((1u << s) - 1));
    nbits -= s;
    return v;
  }
  XFM_DEVINL bool overrun() const { return nbits < pad; }
};

XFM_DEVINL int huff_decode(BitReader& br, const HuffTab& t) {
  br.fill();
  const uint32_t w = br.peek16();
  const uint32_t lk = t.look[w >> 7];
  if (lk) { br.skip((int)(lk >> 8)); return (int)(lk & 255u); }
  int l = 10;
  int code = (int)(w >> 6);
  while (l <= 16 && code > t.maxcode[l]) { ++l; code = (int)(w >> (16 - l)); }
  if (l > 16) { br.status |= J_BAD_CODE; return 0; }
  br.skip(l);
  const int idx = code + t.valoff[l];
  if (idx < 0 || idx > 255) { br.status |= J_BAD_CODE; return 0; }
  return t.val[idx];
}

XFM_DEVINL int huff_extend(int v, int s) { return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v; }

__global__ void __launch_bounds__(128)
jpeg_entropy_kernel(const uint8_t* __restrict__ bytes, const JpegDesc* __restrict__ descs, const int64_t* __restrict__ ivals,
                    int16_t* __restrict__ coef, int32_t* __restrict__ status) {
  __shared__ __align__(16) HuffTab tabs[4];
  const JpegDesc& d = descs[blockIdx.x];
  const int n_int = d.n_int;
  if (n_int == 0) return;
  {
    const int4* src = (const int4*)d.tab;
    int4* dst = (int4*)tabs;
    for (int i = threadIdx.x; i < (int)(sizeof(tabs) / 16); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int ncomp = d.ncomp, mcux = d.mcux, mpi = d.mcus_per_int, total = d.total_mcus;
  int h[3], v[3], bw[3], dct[3], act[3];
  int64_t cbase[3];
  for (int c = 0; c < 3; ++c) {
    h[c] = d.h[c]; v[c] = d.v[c]; bw[c] = d.bw[c]; dct[c] = d.dct[c]; act[c] = d.act[c];
    cbase[c] = d.coef_off + d.comp_coef[c];
  }
  int st = 0;
  for (int iv = threadIdx.x; iv < n_int; iv += blockDim.x) {
    BitReader br;
    br.p = bytes + ivals[2 * (d.first_interval + iv)];
    br.end = bytes + ivals[2 * (d.first_interval + iv) + 1];
    br.acc = 0; br.nbits = 0; br.pad = 0; br.status = 0;
    int pred[3] = {0, 0, 0};
    const int m1 = min(total, (iv + 1) * mpi);
    for (int m = iv * mpi; m < m1 && br.status == 0; ++m) {
      const int my = m / mcux, mx = m - my * mcux;
      for (int c = 0; c < ncomp; ++c) {
        for (int by = 0; by < v[c]; ++by) {
          for (int bx = 0; bx < h[c]; ++bx) {
            int16_t* blk = coef + (cbase[c] + (int64_t)(my * v[c] + by) * bw[c] + mx * h[c] + bx) * 64;
#pragma unroll
            for (int i = 0; i < 8; ++i) ((int4*)blk)[i] = make_int4(0, 0, 0, 0);
            int s = huff_decode(br, tabs[dct[c]]);
            if (s) { br.fill(); s = huff_extend(br.get(s), s); }
            pred[c] += s;
            blk[0] = (int16_t)pred[c];                  // JCOEF: the predictor is an int, the stored coefficient int16
            for (int k = 1; k < 64;) {
              const int rs = huff_decode(br, tabs[act[c]]);
              const int r = rs >> 4;
              s = rs & 15;
              if (s == 0) {
                if (r != 15) break;
                if (k + 15 > 63) { br.status |= J_BAD_RUN; break; }
                k += 16;
                continue;
              }
              k += r;
              if (k > 63) { br.status |= J_BAD_RUN; break; }
              br.fill();
              blk[c_zigzag[k]] = (int16_t)huff_extend(br.get(s), s);
              ++k;
            }
          }
        }
      }
      if (br.overrun()) br.status |= J_SHORT_DATA;
    }
    st |= br.status;
  }
  if (st) atomicOr(status + blockIdx.x, st);
}

// --------------------------------------------------------------------------------------------- 2. dequantise + ISLOW IDCT
// libjpeg-turbo's jsimd_idct_islow (the code Pillow runs on x86-64): jidctint.c's CONST_BITS 13 / PASS1_BITS 2 algorithm with
// 16-bit dequantisation products, 16-bit sums where the SIMD code adds 16-bit lanes (x0 +- x4, x7 + x3, x5 + x1), 16-bit
// saturation of the first pass, the whole-block "no vertical AC term" shortcut (dc << 2, 16-bit), and a final clamp to [0, 255].
XFM_DEVINL int s16(int x) { return (int)(int16_t)x; }

XFM_DEVINL void islow_1d(int x0, int x1, int x2, int x3, int x4, int x5, int x6, int x7, int shift, int* o) {
  const int tmp0 = s16(x0 + x4) * 8192, tmp1 = s16(x0 - x4) * 8192;
  const int tmp2 = x2 * 4433 + x6 * (4433 - 15137);
  const int tmp3 = x2 * (4433 + 6270) + x6 * 4433;
  const int t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
  const int z3 = s16(x7 + x3), z4 = s16(x5 + x1);
  const int z3p = z3 * (9633 - 16069) + z4 * 9633;
  const int z4p = z3 * 9633 + z4 * (9633 - 3196);
  const int o0 = x7 * (2446 - 7373) - x1 * 7373 + z3p;
  const int o3 = -x7 * 7373 + x1 * (12299 - 7373) + z4p;
  const int o1 = x5 * (16819 - 20995) - x3 * 20995 + z4p;
  const int o2 = -x5 * 20995 + x3 * (25172 - 20995) + z3p;
  const int r = 1 << (shift - 1);
  o[0] = (t10 + o3 + r) >> shift; o[7] = (t10 - o3 + r) >> shift;
  o[1] = (t11 + o2 + r) >> shift; o[6] = (t11 - o2 + r) >> shift;
  o[2] = (t12 + o1 + r) >> shift; o[5] = (t12 - o1 + r) >> shift;
  o[3] = (t13 + o0 + r) >> shift; o[4] = (t13 - o0 + r) >> shift;
}

__global__ void __launch_bounds__(128)
jpeg_idct_kernel(const JpegDesc* __restrict__ descs, const int16_t* __restrict__ coef, uint8_t* __restrict__ planes) {
  const JpegDesc& d = descs[blockIdx.y];
  const int64_t blk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (d.n_int == 0 || blk >= d.comp_coef[d.ncomp]) return;
  const int c = blk >= d.comp_coef[2] && d.ncomp > 2 ? 2 : (blk >= d.comp_coef[1] && d.ncomp > 1 ? 1 : 0);
  const int64_t local = blk - d.comp_coef[c];
  const int bw = d.bw[c];
  const int by = (int)(local / bw), bx = (int)(local - (int64_t)by * bw);
  int w[64];
  bool ac_zero = true;
  {
    const int4* src = (const int4*)(coef + (d.coef_off + blk) * 64);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int4 q4 = src[i];
      const int16_t* e = (const int16_t*)&q4;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        w[i * 8 + j] = e[j];
        if (i > 0 && e[j] != 0) ac_zero = false;
      }
    }
  }
  const uint16_t* q = d.qt[c];
#pragma unroll
  for (int i = 0; i < 64; ++i) w[i] = s16(w[i] * (int)q[i]);
  if (ac_zero) {
#pragma unroll
    for (int col = 0; col < 8; ++col) {
      const int dc = s16(w[col] * 4);
#pragma unroll
      for (int row = 0; row < 8; ++row) w[row * 8 + col] = dc;
    }
  } else {
#pragma unroll
    for (int col = 0; col < 8; ++col) {
      int o[8];
      islow_1d(w[col], w[8 + col], w[16 + col], w[24 + col], w[32 + col], w[40 + col], w[48 + col], w[56 + col], 11, o);
#pragma unroll
      for (int row = 0; row < 8; ++row) w[row * 8 + col] = max(-32768, min(32767, o[row]));
    }
  }
  const int pw = bw * 8;
  uint8_t* dst = planes + d.plane_off + d.comp_plane[c] + ((int64_t)by * 8) * pw + bx * 8;
#pragma unroll
  for (int row = 0; row < 8; ++row) {
    int o[8];
    islow_1d(w[row * 8], w[row * 8 + 1], w[row * 8 + 2], w[row * 8 + 3], w[row * 8 + 4], w[row * 8 + 5], w[row * 8 + 6],
             w[row * 8 + 7], 18, o);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      lo |= (uint32_t)(max(-128, min(127, o[j])) + 128) << (8 * j);
      hi |= (uint32_t)(max(-128, min(127, o[j + 4])) + 128) << (8 * j);
    }
    *(uint2*)(dst + (int64_t)row * pw) = make_uint2(lo, hi);
  }
}

// ----------------------------------------------------------------------------------------- 3. upsample + colour convert
// jdsample.c fancy upsampling, evaluated per output pixel: h2v1 out[2i] = (3 p[i] + p[i-1] + 1) >> 2, out[2i+1] =
// (3 p[i] + p[i+1] + 2) >> 2; h2v2 column sums cs = 3 p[nearer row] + p[further row], out = (3 cs[i] + cs[i-+1] + 8 | 7) >> 4;
// neighbours clamped at the downsampled width / height (libjpeg replicates the edge column and the last real row); plain
// replication when the downsampled width is <= 2.  jdcolor.c ycc_rgb_convert: FIX(x) = round(x * 2^16), ONE_HALF rounding.
XFM_DEVINL int sample(const uint8_t* p, int pw, int x, int y) { return p[(int64_t)y * pw + x]; }

XFM_DEVINL int upsampled(const JpegDesc& d, const uint8_t* p, int c, int x, int y, int hmax, int vmax) {
  const int pw = d.bw[c] * 8, dw = d.dw[c], dh = d.dh[c];
  const int fh = hmax / d.h[c], fv = vmax / d.v[c];
  if (fh == 1) return sample(p, pw, x, y);
  const int i = x >> 1;
  if (dw <= 2) return sample(p, pw, i, fv == 2 ? y >> 1 : y);
  const int il = max(i - 1, 0), ir = min(i + 1, dw - 1);
  if (fv == 1) {
    const int m = 3 * sample(p, pw, i, y);
    return (x & 1) ? (m + sample(p, pw, ir, y) + 2) >> 2 : (m + sample(p, pw, il, y) + 1) >> 2;
  }
  const int r = y >> 1, rn = (y & 1) ? min(r + 1, dh - 1) : max(r - 1, 0);
  const int j = (x & 1) ? ir : il;
  const int cs = 3 * sample(p, pw, i, r) + sample(p, pw, i, rn);
  const int cn = 3 * sample(p, pw, j, r) + sample(p, pw, j, rn);
  return (x & 1) ? (3 * cs + cn + 7) >> 4 : (3 * cs + cn + 8) >> 4;
}

__global__ void __launch_bounds__(128)
jpeg_color_kernel(const JpegDesc* __restrict__ descs, const uint8_t* __restrict__ planes, uint8_t* __restrict__ out) {
  const JpegDesc& d = descs[blockIdx.z];
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (d.n_int == 0 || x >= d.W || y >= d.H) return;
  uint8_t* o = out + d.out_off + ((int64_t)y * d.W + x) * 3;
  const uint8_t* base = planes + d.plane_off;
  if (d.ncomp == 1) {
    const uint8_t g = base[(int64_t)y * d.bw[0] * 8 + x];
    o[0] = g; o[1] = g; o[2] = g;
    return;
  }
  const int hmax = max(d.h[0], max(d.h[1], d.h[2])), vmax = max(d.v[0], max(d.v[1], d.v[2]));
  const int Y = upsampled(d, base + d.comp_plane[0], 0, x, y, hmax, vmax);
  const int cb = upsampled(d, base + d.comp_plane[1], 1, x, y, hmax, vmax) - 128;
  const int cr = upsampled(d, base + d.comp_plane[2], 2, x, y, hmax, vmax) - 128;
  const int r = Y + ((91881 * cr + 32768) >> 16);
  const int g = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
  const int b = Y + ((116130 * cb + 32768) >> 16);
  o[0] = (uint8_t)max(0, min(255, r));
  o[1] = (uint8_t)max(0, min(255, g));
  o[2] = (uint8_t)max(0, min(255, b));
}

int jpeg_decode(const uint8_t* bytes, const void* desc, const int64_t* intervals, int n, int16_t* coef, uint8_t* planes, uint8_t* out,
                int32_t* status, int64_t max_blocks, int max_w, int max_h, cudaStream_t s) {
  if (n < 0 || n > 65535 || max_blocks < 0 || max_w < 0 || max_h < 0 || max_h > 65535) {
    set_error("jpeg_decode: need 0 <= n <= 65535 and 0 <= max_h <= 65535");
    return XFM_ERR_BAD_ARG;
  }
  if (n == 0) return 0;
  if (!desc || !out || !status) { set_error("jpeg_decode: null pointer"); return XFM_ERR_BAD_ARG; }
  if (max_blocks > 0 && (!bytes || !intervals || !coef || !planes)) { set_error("jpeg_decode: null pointer"); return XFM_ERR_BAD_ARG; }
  if (((uintptr_t)desc & 15) || ((uintptr_t)coef & 15) || ((uintptr_t)planes & 7)) {
    set_error("jpeg_decode: desc and coef must be 16-byte, planes 8-byte aligned");
    return XFM_ERR_BAD_ARG;
  }
  const JpegDesc* d = (const JpegDesc*)desc;
  jpeg_entropy_kernel<<<n, 128, 0, s>>>(bytes, d, intervals, coef, status);
  const unsigned gx = (unsigned)std::max<int64_t>(1, (max_blocks + 127) / 128);
  jpeg_idct_kernel<<<dim3(gx, n), 128, 0, s>>>(d, coef, planes);
  jpeg_color_kernel<<<dim3((unsigned)std::max(1, (max_w + 127) / 128), (unsigned)std::max(1, max_h), n), 128, 0, s>>>(d, planes, out);
  count_launch(3);
  return (int)cudaGetLastError();
}

size_t jpeg_desc_bytes() { return sizeof(JpegDesc); }

}  // namespace xfm
