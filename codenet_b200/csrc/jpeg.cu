// Baseline JPEG decoding on the device: what cv2.imdecode(buf, cv2.IMREAD_COLOR) returns (OpenCV's bundled libjpeg-turbo),
// element for element, for the streams cdn_jpeg_parse accepts (include/codenet_b200.h, DESIGN.md section 9).
//   * cdn_jpeg_parse: host-only marker parser.  Every read is bounded by nbytes; the Huffman tables are checked as
//     jpeg_make_d_derived_tbl checks them and stored in its decoding form (8-bit lookahead + maxcode / valoffset).
//   * cdn_jpeg_decode_batch: four kernels over a ragged batch on one stream --
//       jpeg_restart_index_kernel   one CTA per frame with restart markers: the byte offset of every restart interval;
//       jpeg_entropy_kernel         one thread per restart interval (the whole scan without restart markers): Huffman
//                                   decoding with 0xFF00 unstuffing and DC prediction, coefficients de-zigzagged;
//       jpeg_idct_kernel            dequantisation + jpeg_idct_islow (jidctint.c), 8 threads per block;
//       jpeg_color_kernel           h2v1 / h2v2 fancy upsampling (jdsample.c) + ycc_rgb_convert (jdcolor.c), BGR out.
//     oracle/jpeg_ref.py restates the same steps in numpy; the CPU tests check it against cv2.
#include "common.cuh"
#include <cstring>
#include <algorithm>

static_assert(sizeof(cdn_jpeg_huff) == 912, "cdn_jpeg_huff layout (codenet_b200.jpeg.JPEG_HUFF)");
static_assert(sizeof(cdn_jpeg_frame) == 4256, "cdn_jpeg_frame layout (codenet_b200.jpeg.JPEG_FRAME)");

namespace {

#define CDN_JPEG_ZIGZAG {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, \
                         13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, \
                         52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63}
constexpr uint8_t kZigzag[64] = CDN_JPEG_ZIGZAG;               // zigzag index -> natural (row-major) index
__constant__ uint8_t c_zigzag[64] = CDN_JPEG_ZIGZAG;
constexpr int64_t kMaxPixels = 1LL << 26;
constexpr int kWsAlign = 256;
// the window inside which libjpeg-turbo's C islow (wrapping range-limit table, 32-bit arithmetic) and its SIMD islow (16-bit
// lanes, saturating packs) compute the same samples; a frame that leaves it is flagged CDN_JPEG_BAD_RANGE (DESIGN.md section 9)
constexpr int kCoefLimit = 2047;      // |dequantised coefficient|
constexpr int kPass1Limit = 8191;     // |column-pass output|: sums of four of them still fit 16 bits
constexpr int kOutLo = -512, kOutHi = 511;

int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// jpeg_make_d_derived_tbl: canonical codes, the code-space check, DC symbols <= 15, lookahead table.  The code space is checked
// for every length before anything is written: an oversubscribed length (e.g. three 1-bit codes) would otherwise index past
// the lookahead table.
int derive_huff(const uint8_t* counts, const uint8_t* vals, int nsym, bool dc, cdn_jpeg_huff* h) {
  int code = 0;
  for (int l = 1; l <= 16; ++l) {
    code += counts[l - 1];
    if (code >= (1 << l)) return CDN_JPEG_ERR_TABLE;      // "no code is allowed to be all ones"
    code <<= 1;
  }
  if (dc)
    for (int i = 0; i < nsym; ++i)
      if (vals[i] > 15) return CDN_JPEG_ERR_TABLE;
  std::memset(h, 0, sizeof(*h));
  int p = 0;
  code = 0;
  for (int l = 1; l <= 16; ++l) {
    const int c = counts[l - 1];
    h->maxcode[l] = -1;
    if (c) {
      h->valoffset[l] = p - code;
      for (int k = 0; k < c; ++k, ++p, ++code)
        if (l <= CDN_JPEG_LOOKAHEAD) {
          const int base = code << (CDN_JPEG_LOOKAHEAD - l);          // code < 2^l: base + j < 2^LOOKAHEAD
          for (int j = 0; j < (1 << (CDN_JPEG_LOOKAHEAD - l)); ++j) h->look[base + j] = (uint16_t)((l << 8) | vals[p]);
        }
      h->maxcode[l] = code - 1;
    }
    code <<= 1;
  }
  h->maxcode[17] = 0xFFFFF;
  std::memcpy(h->huffval, vals, nsym);
  return 0;
}

// orientation tag (0x0112) of IFD0 of an Exif APP1 payload after "Exif\0\0": 1 when absent, -1 when unreadable
int exif_orientation(const uint8_t* p, int64_t len) {
  if (len < 8) return -1;
  const bool le = p[0] == 'I' && p[1] == 'I', be = p[0] == 'M' && p[1] == 'M';
  if (!le && !be) return -1;
  auto u16 = [&](int64_t o) { return le ? (int)(p[o] | (p[o + 1] << 8)) : (int)((p[o] << 8) | p[o + 1]); };
  auto u32 = [&](int64_t o) { return le ? ((int64_t)u16(o + 2) << 16) | u16(o) : ((int64_t)u16(o) << 16) | u16(o + 2); };
  if (u16(2) != 42) return -1;
  const int64_t ifd = u32(4);
  if (ifd + 2 > len) return -1;
  const int cnt = u16(ifd);
  for (int k = 0; k < cnt; ++k) {
    const int64_t e = ifd + 2 + 12LL * k;
    if (e + 12 > len) return -1;
    if (u16(e) == 0x0112) return u16(e + 2) == 3 ? u16(e + 8) : -1;
  }
  return 1;
}

// MCU grid, block grids, downsampled sizes, segments and workspace layout from width, height, ncomp, comp_h / comp_v and the
// restart interval (the parser fills those; decode_batch re-derives the rest to check a descriptor)
void frame_geometry(cdn_jpeg_frame* f) {
  const int W = f->width, H = f->height;
  f->hmax = f->ncomp == 1 ? 1 : f->comp_h[0];
  f->vmax = f->ncomp == 1 ? 1 : f->comp_v[0];
  f->mcux = (W + 8 * f->hmax - 1) / (8 * f->hmax);
  f->mcuy = (H + 8 * f->vmax - 1) / (8 * f->vmax);
  const int64_t mcus = (int64_t)f->mcux * f->mcuy;
  f->nsegments = f->restart_interval ? (int)((mcus + f->restart_interval - 1) / f->restart_interval) : 1;
  int64_t off = align_up(4LL * f->nsegments, kWsAlign), blocks = 0;
  for (int c = 0; c < 3; ++c) {
    if (c >= f->ncomp) { f->comp_h[c] = f->comp_v[c] = f->comp_bw[c] = f->comp_bh[c] = f->comp_dw[c] = f->comp_dh[c] = 0; continue; }
    f->comp_bw[c] = f->mcux * f->comp_h[c];
    f->comp_bh[c] = f->mcuy * f->comp_v[c];
    f->comp_dw[c] = (W * f->comp_h[c] + f->hmax - 1) / f->hmax;
    f->comp_dh[c] = (H * f->comp_v[c] + f->vmax - 1) / f->vmax;
    blocks += (int64_t)f->comp_bw[c] * f->comp_bh[c];
  }
  f->coef_rel = off;
  off = align_up(off + blocks * 128, kWsAlign);
  for (int c = 0; c < 3; ++c) {
    f->plane_rel[c] = off;
    off = align_up(off + (int64_t)f->comp_bw[c] * f->comp_bh[c] * 64, kWsAlign);
  }
  f->ws_bytes = off;
}

int parse(const uint8_t* d, int64_t n, cdn_jpeg_frame* f) {
  if (!d || n < 4 || d[0] != 0xFF || d[1] != 0xD8) return CDN_JPEG_ERR_NOT_JPEG;
  if (n >= (1LL << 31)) return CDN_JPEG_HOST_SIZE;
  uint16_t qt[4][64];
  cdn_jpeg_huff dc[4], ac[4];
  bool have_q[4] = {}, have_dc[4] = {}, have_ac[4] = {};
  bool sof = false, jfif = false, adobe = false;
  int adobe_transform = -1, exif_count = 0, orientation = 1;
  int W = 0, H = 0, nc = 0, ids[3] = {}, tq[3] = {}, td[3] = {}, ta[3] = {};
  int64_t pos = 2;
  for (;;) {
    if (pos + 2 > n) return CDN_JPEG_ERR_TRUNCATED;
    if (d[pos] != 0xFF) return CDN_JPEG_ERR_SEGMENT;
    while (pos + 1 < n && d[pos + 1] == 0xFF) ++pos;      // fill bytes
    if (pos + 4 > n) return CDN_JPEG_ERR_TRUNCATED;
    const int m = d[pos + 1];
    if (m == 0xD9) return CDN_JPEG_ERR_TRUNCATED;         // EOI before a scan
    if (m == 0x00 || m == 0x01 || m == 0xD8 || (m >= 0xD0 && m <= 0xD7)) return CDN_JPEG_ERR_SEGMENT;
    const int64_t L = (d[pos + 2] << 8) | d[pos + 3];
    if (L < 2) return CDN_JPEG_ERR_SEGMENT;
    if (pos + 2 + L > n) return CDN_JPEG_ERR_TRUNCATED;
    const uint8_t* p = d + pos + 4;
    const int64_t len = L - 2;
    pos += 2 + L;
    if (m == 0xC0 || m == 0xC1) {
      if (sof || len < 6) return CDN_JPEG_ERR_SEGMENT;
      sof = true;
      nc = p[5];
      if (len != 6 + 3 * nc) return CDN_JPEG_ERR_SEGMENT;
      if (p[0] != 8) return CDN_JPEG_HOST_PRECISION;
      H = (p[1] << 8) | p[2];
      W = (p[3] << 8) | p[4];
      if (W == 0) return CDN_JPEG_ERR_SEGMENT;
      if (H == 0) return CDN_JPEG_HOST_SCAN;                // height defined by DNL
      if (nc != 1 && nc != 3) return nc == 0 ? CDN_JPEG_ERR_SEGMENT : CDN_JPEG_HOST_COLOR;
      for (int c = 0; c < nc; ++c) {
        const int h = p[7 + 3 * c] >> 4, v = p[7 + 3 * c] & 15;
        if (h < 1 || h > 4 || v < 1 || v > 4 || p[8 + 3 * c] > 3) return CDN_JPEG_ERR_SEGMENT;
        ids[c] = p[6 + 3 * c];
        f->comp_h[c] = h; f->comp_v[c] = v;
        tq[c] = p[8 + 3 * c];
      }
    } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4) {
      return CDN_JPEG_HOST_PROCESS;                         // progressive, lossless, hierarchical, arithmetic (DAC too)
    } else if (m == 0xC4) {
      for (int64_t i = 0; i < len;) {
        if (i + 17 > len) return CDN_JPEG_ERR_SEGMENT;
        const int tc = p[i] >> 4, th = p[i] & 15;
        if (tc > 1 || th > 3) return CDN_JPEG_ERR_SEGMENT;
        int nsym = 0;
        for (int k = 0; k < 16; ++k) nsym += p[i + 1 + k];
        if (nsym > 256 || i + 17 + nsym > len) return CDN_JPEG_ERR_TABLE;
        const int rc = derive_huff(p + i + 1, p + i + 17, nsym, tc == 0, tc ? &ac[th] : &dc[th]);
        if (rc) return rc;
        (tc ? have_ac : have_dc)[th] = true;
        i += 17 + nsym;
      }
    } else if (m == 0xDB) {
      for (int64_t i = 0; i < len;) {
        const int pq = p[i] >> 4, t = p[i] & 15;
        if (pq > 1 || t > 3 || i + 1 + 64 * (pq + 1) > len) return CDN_JPEG_ERR_SEGMENT;
        for (int k = 0; k < 64; ++k)
          qt[t][kZigzag[k]] = pq ? (uint16_t)((p[i + 1 + 2 * k] << 8) | p[i + 2 + 2 * k]) : p[i + 1 + k];
        have_q[t] = true;
        i += 1 + 64 * (pq + 1);
      }
    } else if (m == 0xDD) {
      if (len != 2) return CDN_JPEG_ERR_SEGMENT;
      f->restart_interval = (p[0] << 8) | p[1];
    } else if (m == 0xDC) {
      return CDN_JPEG_HOST_SCAN;                            // DNL
    } else if (m == 0xE0) {
      if (len >= 14 && !std::memcmp(p, "JFIF", 5)) jfif = true;
    } else if (m == 0xEE) {
      if (len >= 12 && !std::memcmp(p, "Adobe", 5)) { adobe = true; adobe_transform = p[11]; }
    } else if (m == 0xE1) {
      if (len >= 6 && !std::memcmp(p, "Exif\0\0", 6)) { ++exif_count; orientation = exif_orientation(p + 6, len - 6); }
    } else if (m == 0xDA) {
      if (!sof || len < 1) return CDN_JPEG_ERR_SEGMENT;
      const int ns = p[0];
      if (ns < 1 || ns > 4 || len != 4 + 2 * ns) return CDN_JPEG_ERR_SEGMENT;
      if (ns != nc) return CDN_JPEG_HOST_SCAN;
      for (int c = 0; c < ns; ++c) {
        if (p[1 + 2 * c] != ids[c]) return CDN_JPEG_HOST_SCAN;
        td[c] = p[2 + 2 * c] >> 4; ta[c] = p[2 + 2 * c] & 15;
        if (td[c] > 3 || ta[c] > 3) return CDN_JPEG_ERR_SEGMENT;
      }
      if (p[1 + 2 * ns] != 0 || p[2 + 2 * ns] != 63 || p[3 + 2 * ns] != 0) return CDN_JPEG_HOST_SCAN;
      break;
    } else if (!((m >= 0xE0 && m <= 0xEF) || m == 0xFE)) {
      return CDN_JPEG_ERR_SEGMENT;                          // reserved markers libjpeg rejects
    }
  }
  // colour space as libjpeg's default_decompress_parms decides it
  if (nc == 3) {
    const bool rgb = jfif ? false : adobe ? adobe_transform == 0 : (ids[0] == 'R' && ids[1] == 'G' && ids[2] == 'B');
    if (rgb) return CDN_JPEG_HOST_COLOR;
    for (int c = 0; c < 3; ++c) {
      if (c > 0 && (f->comp_h[c] != 1 || f->comp_v[c] != 1)) return CDN_JPEG_HOST_SAMPLING;
    }
    const int h = f->comp_h[0], v = f->comp_v[0];
    if (!((h == 1 && v == 1) || (h == 2 && v == 1) || (h == 2 && v == 2))) return CDN_JPEG_HOST_SAMPLING;
    for (int c = 0; c < 3; ++c)
      for (int k = 0; k < c; ++k)
        if (ids[k] == ids[c]) return CDN_JPEG_HOST_SCAN;
  } else {
    f->comp_h[0] = f->comp_v[0] = 1;                        // a single-component scan is not interleaved: 1 block per MCU
  }
  if (exif_count > 1 || orientation != 1) return CDN_JPEG_HOST_ORIENTATION;
  if ((int64_t)W * H > kMaxPixels) return CDN_JPEG_HOST_SIZE;
  // tables: every referenced one defined; at most two distinct DC and two distinct AC tables (slots 0-1 and 2-3)
  int dc_ids[2] = {-1, -1}, ac_ids[2] = {-1, -1};
  for (int c = 0; c < nc; ++c) {
    if (!have_q[tq[c]] || !have_dc[td[c]] || !have_ac[ta[c]]) return CDN_JPEG_HOST_SCAN;
    int s = 0;
    while (s < 2 && dc_ids[s] != -1 && dc_ids[s] != td[c]) ++s;
    if (s == 2) return CDN_JPEG_HOST_SCAN;
    dc_ids[s] = td[c]; f->comp_dc[c] = s; f->huff[s] = dc[td[c]];
    s = 0;
    while (s < 2 && ac_ids[s] != -1 && ac_ids[s] != ta[c]) ++s;
    if (s == 2) return CDN_JPEG_HOST_SCAN;
    ac_ids[s] = ta[c]; f->comp_ac[c] = 2 + s; f->huff[2 + s] = ac[ta[c]];
    std::memcpy(f->qt[c], qt[tq[c]], sizeof(f->qt[c]));
  }
  // the entropy-coded data ends at the first marker that is neither RSTn nor a stuffed 0xFF; the device takes one scan only,
  // so that marker must be EOI (or the data simply ends: a frame that needs the missing bytes is flagged on the device)
  int64_t i = pos, end = n;
  while (i < n) {
    const uint8_t* q = (const uint8_t*)std::memchr(d + i, 0xFF, (size_t)(n - i));
    if (!q) break;
    const int64_t j = q - d;
    if (j + 1 >= n) { end = j; break; }
    const int nx = d[j + 1];
    if (nx == 0x00 || (nx >= 0xD0 && nx <= 0xD7)) { i = j + 2; continue; }
    if (nx == 0xFF) { i = j + 1; continue; }
    if (nx != 0xD9) return CDN_JPEG_HOST_SCAN;
    end = j;
    break;
  }
  f->width = W; f->height = H; f->ncomp = nc;
  f->nbytes = n; f->scan_offset = pos; f->scan_end = end;
  frame_geometry(f);
  return 0;
}

// ---- device ------------------------------------------------------------------------------------------------------------
struct BitReader {
  const uint8_t* p;
  const uint8_t* end;
  uint64_t buf;                 // left-aligned
  int n;                        // bits in buf
  int pad;                      // zero bits appended after a marker or the end of the data
  bool stop;

  __device__ void fill() {
    while (n <= 56) {
      uint32_t b = 0;
      bool real = false;
      if (!stop) {
        if (p < end && *p != 0xFF) { b = *p++; real = true; }
        else if (p + 1 < end && p[1] == 0) { b = 0xFF; p += 2; real = true; }
        else stop = true;
      }
      if (!real) pad += 8;
      buf |= (uint64_t)b << (56 - n);
      n += 8;
    }
  }
  __device__ __forceinline__ uint32_t peek(int k) const { return (uint32_t)(buf >> (64 - k)); }
  __device__ __forceinline__ void skip(int k) { buf <<= k; n -= k; }
  __device__ __forceinline__ bool overrun() const { return pad > n; }   // padding bits were consumed
};

__device__ __forceinline__ int huff_decode(BitReader& br, const cdn_jpeg_huff& h) {
  br.fill();
  const uint32_t look = h.look[br.peek(CDN_JPEG_LOOKAHEAD)];
  if (look) { br.skip(look >> 8); return look & 255; }
  for (int l = CDN_JPEG_LOOKAHEAD + 1; l <= 16; ++l) {
    const int code = (int)br.peek(l);
    if (code <= h.maxcode[l]) { br.skip(l); return h.huffval[(code + h.valoffset[l]) & 255]; }
  }
  return -1;
}

__device__ __forceinline__ int huff_extend(uint32_t r, int s) { return (int)r - ((r < (1u << (s - 1))) ? (1 << s) - 1 : 0); }

__device__ __forceinline__ uint8_t* frame_ws(uint8_t* ws, const cdn_jpeg_frame& F) { return ws + F.ws_offset; }

__global__ void __launch_bounds__(256) jpeg_restart_index_kernel(const uint8_t* __restrict__ pool, const cdn_jpeg_frame* __restrict__ frames,
                                                                 uint8_t* __restrict__ ws, int32_t* __restrict__ status) {
  const cdn_jpeg_frame& F = frames[blockIdx.x];
  if (F.restart_interval == 0) return;
  const uint8_t* d = pool + F.data_offset;
  int32_t* seg = reinterpret_cast<int32_t*>(frame_ws(ws, F));
  const int expect = F.nsegments - 1, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t end = F.scan_end;
  __shared__ int s_cnt[8];
  int found = 0;
  bool bad = false;
  for (int64_t base = F.scan_offset; base < end; base += 256) {
    const int64_t i = base + threadIdx.x;
    const bool mk = i + 1 < end && d[i] == 0xFF && (d[i + 1] & 0xF8) == 0xD0;
    const unsigned b = __ballot_sync(0xffffffffu, mk);
    if (lane == 0) s_cnt[warp] = __popc(b);
    __syncthreads();
    int before = found + __popc(b & ((1u << lane) - 1)), total = 0;
    for (int k = 0; k < 8; ++k) {
      total += s_cnt[k];
      if (k < warp) before += s_cnt[k];
    }
    if (mk) {
      if (before < expect && (d[i + 1] & 7) == (before & 7)) seg[before + 1] = (int32_t)(i + 2);
      else bad = true;
    }
    found += total;
    __syncthreads();
  }
  if (bad || (threadIdx.x == 0 && found != expect)) atomicOr(&status[blockIdx.x], CDN_JPEG_BAD_RESTART);
}

// grid (restart intervals / 32, frames); thread k decodes restart interval k of its frame
__global__ void __launch_bounds__(32) jpeg_entropy_kernel(const uint8_t* __restrict__ pool, const cdn_jpeg_frame* __restrict__ frames,
                                                          uint8_t* __restrict__ ws, int32_t* __restrict__ status) {
  __shared__ uint8_t s_zz[64];
  for (int k = threadIdx.x; k < 64; k += 32) s_zz[k] = c_zigzag[k];
  __syncthreads();
  const int fi = blockIdx.y;
  const cdn_jpeg_frame& F = frames[fi];
  const int seg = blockIdx.x * 32 + threadIdx.x;
  if (seg >= F.nsegments || status[fi] != 0) return;
  uint8_t* w = frame_ws(ws, F);
  const uint8_t* d = pool + F.data_offset;
  int64_t start = F.scan_offset;
  if (seg > 0) {
    start = reinterpret_cast<const int32_t*>(w)[seg];
    if (start < F.scan_offset || start > F.scan_end) { atomicOr(&status[fi], CDN_JPEG_BAD_RESTART); return; }
  }
  BitReader br{d + start, d + F.scan_end, 0, 0, 0, false};
  const int64_t mcus = (int64_t)F.mcux * F.mcuy;
  const int64_t m0 = F.restart_interval ? (int64_t)seg * F.restart_interval : 0;
  const int64_t m1 = F.restart_interval ? min(m0 + F.restart_interval, mcus) : mcus;
  int16_t* coef = reinterpret_cast<int16_t*>(w + F.coef_rel);
  int64_t comp_base[3];
  comp_base[0] = 0;
  comp_base[1] = (int64_t)F.comp_bw[0] * F.comp_bh[0];
  comp_base[2] = comp_base[1] + (int64_t)F.comp_bw[1] * F.comp_bh[1];
  int pred[3] = {0, 0, 0};
  int flag = 0;
  for (int64_t m = m0; m < m1 && !flag; ++m) {
    const int my = (int)(m / F.mcux), mx = (int)(m - (int64_t)my * F.mcux);
    for (int c = 0; c < F.ncomp && !flag; ++c) {
      const cdn_jpeg_huff& hdc = F.huff[F.comp_dc[c]];
      const cdn_jpeg_huff& hac = F.huff[F.comp_ac[c]];
      const uint16_t* q = F.qt[c];
      const int ch = F.comp_h[c], cv = F.comp_v[c], bw = F.comp_bw[c];
      for (int b = 0; b < ch * cv && !flag; ++b) {
        const int by = my * cv + b / ch, bx = mx * ch + b % ch;
        int16_t* blk = coef + (comp_base[c] + (int64_t)by * bw + bx) * 64;
        uint4* b4 = reinterpret_cast<uint4*>(blk);
#pragma unroll
        for (int k = 0; k < 8; ++k) b4[k] = make_uint4(0, 0, 0, 0);
        int s = huff_decode(br, hdc);
        if (s < 0) { flag = CDN_JPEG_BAD_CODE; break; }
        if (s) { const uint32_t r = br.peek(s); br.skip(s); pred[c] += huff_extend(r, s); }
        if (abs((long long)pred[c] * q[0]) > kCoefLimit) { flag = CDN_JPEG_BAD_RANGE; break; }
        blk[0] = (int16_t)pred[c];
        for (int k = 1; k < 64;) {
          const int rs = huff_decode(br, hac);
          if (rs < 0) { flag = CDN_JPEG_BAD_CODE; break; }
          const int r = rs >> 4;
          s = rs & 15;
          if (s) {
            k += r;
            if (k > 63) { flag = CDN_JPEG_BAD_CODE; break; }
            const uint32_t bits = br.peek(s);
            br.skip(s);
            const int v = huff_extend(bits, s), pos = s_zz[k];
            if (abs((long long)v * q[pos]) > kCoefLimit) { flag = CDN_JPEG_BAD_RANGE; break; }
            blk[pos] = (int16_t)v;
            ++k;
          } else {
            if (r != 15) break;
            k += 16;
          }
        }
        if (!flag && br.overrun()) flag = CDN_JPEG_BAD_END;
      }
    }
  }
  if (flag) atomicOr(&status[fi], flag);
}

constexpr int CONST_BITS = 13, PASS1_BITS = 2;
constexpr int FIX_0_298631336 = 2446, FIX_0_390180644 = 3196, FIX_0_541196100 = 4433, FIX_0_765366865 = 6270,
              FIX_0_899976223 = 7373, FIX_1_175875602 = 9633, FIX_1_501321110 = 12299, FIX_1_847759065 = 15137,
              FIX_1_961570560 = 16069, FIX_2_053119869 = 16819, FIX_2_562915447 = 20995, FIX_3_072711026 = 25172;

// the even / odd butterfly of jpeg_idct_islow; o[k] before descaling
__device__ __forceinline__ void idct_1d(const int s[8], int o[8]) {
  int z1 = (s[2] + s[6]) * FIX_0_541196100;
  const int tmp2 = z1 + s[6] * -FIX_1_847759065, tmp3 = z1 + s[2] * FIX_0_765366865;
  int tmp0 = (s[0] + s[4]) * (1 << CONST_BITS), tmp1 = (s[0] - s[4]) * (1 << CONST_BITS);
  const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
  int t0 = s[7], t1 = s[5], t2 = s[3], t3 = s[1];
  z1 = t0 + t3;
  int z2 = t1 + t2, z3 = t0 + t2, z4 = t1 + t3;
  const int z5 = (z3 + z4) * FIX_1_175875602;
  t0 *= FIX_0_298631336; t1 *= FIX_2_053119869; t2 *= FIX_3_072711026; t3 *= FIX_1_501321110;
  z1 *= -FIX_0_899976223; z2 *= -FIX_2_562915447; z3 *= -FIX_1_961570560; z4 *= -FIX_0_390180644;
  z3 += z5; z4 += z5;
  t0 += z1 + z3; t1 += z2 + z4; t2 += z2 + z3; t3 += z1 + z4;
  o[0] = tmp10 + t3; o[7] = tmp10 - t3; o[1] = tmp11 + t2; o[6] = tmp11 - t2;
  o[2] = tmp12 + t1; o[5] = tmp12 - t1; o[3] = tmp13 + t0; o[4] = tmp13 - t0;
}

constexpr int IDCT_BLOCKS = 32;   // 8x8 blocks per CTA, 8 threads each

// grid (blocks / 32, frames): thread r of a block runs column r of pass 1 and row r of pass 2
__global__ void __launch_bounds__(IDCT_BLOCKS * 8) jpeg_idct_kernel(const cdn_jpeg_frame* __restrict__ frames, uint8_t* __restrict__ ws,
                                                                    int32_t* __restrict__ status) {
  __shared__ int s_ws[IDCT_BLOCKS][64];
  const int fi = blockIdx.y;
  const cdn_jpeg_frame& F = frames[fi];
  const int lb = threadIdx.x >> 3, r = threadIdx.x & 7;
  int64_t b = (int64_t)blockIdx.x * IDCT_BLOCKS + lb;
  int c = 0;
  for (; c < F.ncomp; ++c) {
    const int64_t nb = (int64_t)F.comp_bw[c] * F.comp_bh[c];
    if (b < nb) break;
    b -= nb;
  }
  const bool active = c < F.ncomp && status[fi] == 0;
  uint8_t* w = frame_ws(ws, F);
  int flag = 0;
  int by = 0, bx = 0;
  if (active) {
    by = (int)(b / F.comp_bw[c]); bx = (int)(b - (int64_t)by * F.comp_bw[c]);
    int64_t gb = b;
    for (int k = 0; k < c; ++k) gb += (int64_t)F.comp_bw[k] * F.comp_bh[k];
    const int16_t* blk = reinterpret_cast<const int16_t*>(w + F.coef_rel) + gb * 64;
    const uint16_t* q = F.qt[c];
    int s[8], o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = (int)blk[k * 8 + r] * (int)q[k * 8 + r];
    idct_1d(s, o);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int v = (o[k] + (1 << (CONST_BITS - PASS1_BITS - 1))) >> (CONST_BITS - PASS1_BITS);
      if (v < -kPass1Limit || v > kPass1Limit) flag = CDN_JPEG_BAD_RANGE;
      s_ws[lb][k * 8 + r] = min(max(v, -kPass1Limit), kPass1Limit);     // keeps pass 2 in 32 bits on a flagged frame
    }
  }
  __syncthreads();
  if (active) {
    int s[8], o[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s[k] = s_ws[lb][r * 8 + k];
    idct_1d(s, o);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int x = (o[k] + (1 << (CONST_BITS + PASS1_BITS + 3 - 1))) >> (CONST_BITS + PASS1_BITS + 3);
      if (x < kOutLo || x > kOutHi) flag = CDN_JPEG_BAD_RANGE;
      const uint32_t v = (uint32_t)min(max(x + 128, 0), 255);
      if (k < 4) lo |= v << (8 * k); else hi |= v << (8 * (k - 4));
    }
    const int64_t pitch = (int64_t)F.comp_bw[c] * 8;
    *reinterpret_cast<uint2*>(w + F.plane_rel[c] + (int64_t)(by * 8 + r) * pitch + bx * 8) = make_uint2(lo, hi);
    if (flag) atomicOr(&status[fi], flag);
  }
}

// chroma at full resolution (x, y): jdsample.c's fancy upsampling with edge replication, box replication when dw <= 2
__device__ __forceinline__ int chroma_at(const uint8_t* p, int64_t pitch, int dw, int dh, int hs, int vs, int x, int y) {
  if (hs == 1) return p[(int64_t)y * pitch + x];
  const int j = x >> 1;
  if (dw <= 2) return p[(int64_t)(vs == 2 ? y >> 1 : y) * pitch + j];
  const int j2 = min(max(j + ((x & 1) ? 1 : -1), 0), dw - 1);
  if (vs == 1) {
    const uint8_t* row = p + (int64_t)y * pitch;
    return (3 * row[j] + row[j2] + ((x & 1) ? 2 : 1)) >> 2;
  }
  const int i = y >> 1, i2 = min(max(i + ((y & 1) ? 1 : -1), 0), dh - 1);
  const uint8_t* r0 = p + (int64_t)i * pitch;
  const uint8_t* r1 = p + (int64_t)i2 * pitch;
  const int cs = 3 * r0[j] + r1[j], cs2 = 3 * r0[j2] + r1[j2];
  return (3 * cs + cs2 + ((x & 1) ? 7 : 8)) >> 4;
}

// grid (pixels / 256, frames): one output pixel per thread
__global__ void __launch_bounds__(256) jpeg_color_kernel(const cdn_jpeg_frame* __restrict__ frames, const uint8_t* __restrict__ ws,
                                                         uint8_t* __restrict__ out, const int32_t* __restrict__ status) {
  const int fi = blockIdx.y;
  const cdn_jpeg_frame& F = frames[fi];
  const int64_t px = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (px >= (int64_t)F.width * F.height || status[fi] != 0) return;
  const int y = (int)(px / F.width), x = (int)(px - (int64_t)y * F.width);
  const uint8_t* w = ws + F.ws_offset;
  uint8_t* o = out + F.out_offset + px * 3;
  const int Y = w[F.plane_rel[0] + (int64_t)y * F.comp_bw[0] * 8 + x];
  if (F.ncomp == 1) { o[0] = o[1] = o[2] = (uint8_t)Y; return; }
  const int64_t cp = (int64_t)F.comp_bw[1] * 8;
  const int cb = chroma_at(w + F.plane_rel[1], cp, F.comp_dw[1], F.comp_dh[1], F.hmax, F.vmax, x, y) - 128;
  const int cr = chroma_at(w + F.plane_rel[2], cp, F.comp_dw[2], F.comp_dh[2], F.hmax, F.vmax, x, y) - 128;
  // build_ycc_rgb_table: FIX(x) = (int)(x * 65536 + 0.5), ONE_HALF = 1 << 15
  const int R = Y + ((91881 * cr + 32768) >> 16);
  const int G = Y + ((-22554 * cb + 32768 - 46802 * cr) >> 16);
  const int B = Y + ((116130 * cb + 32768) >> 16);
  o[0] = (uint8_t)min(max(B, 0), 255);
  o[1] = (uint8_t)min(max(G, 0), 255);
  o[2] = (uint8_t)min(max(R, 0), 255);
}

// a descriptor as cdn_jpeg_parse leaves it and the caller's offsets, checked against the buffers it names
int check_frame(const cdn_jpeg_frame& f, int i, int64_t pool_bytes, int64_t ws_bytes, int64_t out_bytes) {
  CDN_CHECK(f.ncomp == 1 || f.ncomp == 3, CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: %d components", i, f.ncomp);
  CDN_CHECK(f.width > 0 && f.height > 0 && (int64_t)f.width * f.height <= kMaxPixels, CDN_ERR_INVALID,
            "jpeg_decode_batch: frame %d: bad size %d x %d", i, f.width, f.height);
  CDN_CHECK(f.restart_interval >= 0 && f.restart_interval <= 65535, CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: restart interval", i);
  cdn_jpeg_frame g;
  g.width = f.width; g.height = f.height; g.ncomp = f.ncomp; g.restart_interval = f.restart_interval;
  for (int c = 0; c < 3; ++c) { g.comp_h[c] = f.comp_h[c]; g.comp_v[c] = f.comp_v[c]; }
  const bool sampling = f.ncomp == 1 ? (f.comp_h[0] == 1 && f.comp_v[0] == 1)
                                     : (f.comp_h[1] == 1 && f.comp_v[1] == 1 && f.comp_h[2] == 1 && f.comp_v[2] == 1 &&
                                        f.comp_h[0] >= 1 && f.comp_h[0] <= 2 && f.comp_v[0] >= 1 && f.comp_v[0] <= f.comp_h[0]);
  CDN_CHECK(sampling, CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: sampling not accepted", i);
  frame_geometry(&g);
  bool same = g.hmax == f.hmax && g.vmax == f.vmax && g.mcux == f.mcux && g.mcuy == f.mcuy && g.nsegments == f.nsegments &&
              g.ws_bytes == f.ws_bytes && g.coef_rel == f.coef_rel;
  for (int c = 0; c < 3; ++c)
    same = same && g.comp_bw[c] == f.comp_bw[c] && g.comp_bh[c] == f.comp_bh[c] && g.comp_dw[c] == f.comp_dw[c] &&
           g.comp_dh[c] == f.comp_dh[c] && g.plane_rel[c] == f.plane_rel[c];
  CDN_CHECK(same, CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: geometry does not match its size and sampling", i);
  for (int c = 0; c < f.ncomp; ++c)
    CDN_CHECK(f.comp_dc[c] >= 0 && f.comp_dc[c] <= 1 && f.comp_ac[c] >= 2 && f.comp_ac[c] <= 3, CDN_ERR_INVALID,
              "jpeg_decode_batch: frame %d: Huffman table slots", i);
  for (int t = 0; t < 4; ++t)
    for (int k = 0; k < (1 << CDN_JPEG_LOOKAHEAD); ++k)
      CDN_CHECK((f.huff[t].look[k] >> 8) <= CDN_JPEG_LOOKAHEAD, CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: lookahead table", i);
  CDN_CHECK(f.nbytes > 0 && f.nbytes < (1LL << 31) && f.scan_offset >= 0 && f.scan_offset <= f.scan_end && f.scan_end <= f.nbytes,
            CDN_ERR_INVALID, "jpeg_decode_batch: frame %d: scan range", i);
  CDN_CHECK(f.data_offset >= 0 && f.data_offset <= pool_bytes - f.nbytes, CDN_ERR_INVALID,
            "jpeg_decode_batch: frame %d: stream [%lld, +%lld) outside the pool of %lld bytes", i, (long long)f.data_offset,
            (long long)f.nbytes, (long long)pool_bytes);
  CDN_CHECK(f.ws_offset >= 0 && f.ws_offset % kWsAlign == 0 && f.ws_offset <= ws_bytes - f.ws_bytes, CDN_ERR_INVALID,
            "jpeg_decode_batch: frame %d: workspace [%lld, +%lld) outside %lld bytes or not 256-byte aligned", i,
            (long long)f.ws_offset, (long long)f.ws_bytes, (long long)ws_bytes);
  CDN_CHECK(f.out_offset >= 0 && f.out_offset <= out_bytes - 3LL * f.width * f.height, CDN_ERR_INVALID,
            "jpeg_decode_batch: frame %d: output outside %lld bytes", i, (long long)out_bytes);
  return 0;
}

}  // namespace

extern "C" int cdn_jpeg_parse(const uint8_t* data, int64_t nbytes, cdn_jpeg_frame* out) {
  CDN_CHECK(out != nullptr && nbytes >= 0, CDN_ERR_INVALID, "jpeg_parse: bad arguments");
  std::memset(out, 0, sizeof(*out));
  const int rc = parse(data, nbytes, out);
  if (rc != 0) {
    std::memset(out, 0, sizeof(*out));
  }
  return rc;
}

extern "C" int cdn_jpeg_decode_batch(const uint8_t* d_pool, int64_t pool_bytes, const cdn_jpeg_frame* h_frames,
                                     const cdn_jpeg_frame* d_frames, int n, uint8_t* d_ws, int64_t ws_bytes, uint8_t* d_out,
                                     int64_t out_bytes, int32_t* d_status, cdn_stream_t stream) {
  CDN_CHECK(n >= 0 && n <= 65535, CDN_ERR_INVALID, "jpeg_decode_batch: n = %d outside [0, 65535]", n);
  if (n == 0) return 0;
  CDN_CHECK(h_frames, CDN_ERR_INVALID, "jpeg_decode_batch: null descriptor array");
  int64_t max_seg = 1, max_blocks = 1, max_px = 1;
  bool restart = false;
  for (int i = 0; i < n; ++i) {
    const int rc = check_frame(h_frames[i], i, pool_bytes, ws_bytes, out_bytes);
    if (rc) return rc;
    const cdn_jpeg_frame& f = h_frames[i];
    max_seg = std::max<int64_t>(max_seg, f.nsegments);
    int64_t blocks = 0;
    for (int c = 0; c < f.ncomp; ++c) blocks += (int64_t)f.comp_bw[c] * f.comp_bh[c];
    max_blocks = std::max(max_blocks, blocks);
    max_px = std::max(max_px, (int64_t)f.width * f.height);
    restart = restart || f.restart_interval > 0;
  }
  // the device pointers last: every descriptor check above can be exercised without a device
  CDN_CHECK(d_pool && d_frames && d_ws && d_out && d_status, CDN_ERR_INVALID, "jpeg_decode_batch: null device pointer");
  cudaStream_t st = (cudaStream_t)stream;
  CDN_CUDA(cudaMemsetAsync(d_status, 0, sizeof(int32_t) * n, st));
  if (restart) {
    jpeg_restart_index_kernel<<<n, 256, 0, st>>>(d_pool, d_frames, d_ws, d_status);
    CDN_LAUNCH_CHECK("jpeg_restart_index_kernel");
  }
  jpeg_entropy_kernel<<<dim3((unsigned)((max_seg + 31) / 32), n), 32, 0, st>>>(d_pool, d_frames, d_ws, d_status);
  CDN_LAUNCH_CHECK("jpeg_entropy_kernel");
  jpeg_idct_kernel<<<dim3((unsigned)((max_blocks + IDCT_BLOCKS - 1) / IDCT_BLOCKS), n), IDCT_BLOCKS * 8, 0, st>>>(d_frames, d_ws, d_status);
  CDN_LAUNCH_CHECK("jpeg_idct_kernel");
  jpeg_color_kernel<<<dim3((unsigned)((max_px + 255) / 256), n), 256, 0, st>>>(d_frames, d_ws, d_out, d_status);
  CDN_LAUNCH_CHECK("jpeg_color_kernel");
  return 0;
}
