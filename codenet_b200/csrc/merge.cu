// The multi-scale merge of CtdetDetector (lib/detectors/ctdet.py:59-74) on the device:
//   * cdn_soft_nms     -- the reference's soft_nms (lib/models/external/nms.pyx:77-170) over independent segments, one warp per
//     segment, bit-identical to the sequential mirror compat.soft_nms (in-place rows, copy-from-the-tail discards, stale tail).
//   * cdn_ctdet_merge  -- merge_outputs for a batch of images with S test scales each: gather per class in scale order, divide
//     by the scale (post_process), soft-NMS per class, cut at the max_per_image-th score, rows grouped by class + counts.
//
// Parallel form of one outer iteration i of soft-NMS (restated in numpy and checked against the mirror in
// oracle/soft_nms_place.py): every row of [i+1, N) is examined exactly once and always against the same max row, so its decayed
// score and its discard flag are computed in parallel.  Only the placement is sequential in the mirror, and it depends on the
// flags alone: with F flagged rows and N' = N - F, the k-th flagged row of [i+1, N') (a hole) receives the k-th unflagged row
// of [N', N) counted from the top; back rows keep their pre-pass content except that, when flagged rows lie under the lowest
// unflagged back row R (R > N'), slot N' ends as the decayed row N'+1 (R - N' >= 2) or N' (the mirror's last self-copy).
//
// Arithmetic: the mirror's float / double sequence (compat/nms.py:40-53) with every operation spelled as a correctly rounded
// intrinsic, so that nvcc's FMA contraction cannot fuse (p*q) + area into one DFMA.  exp is CUDA's double exp rounded to
// float; the mirror rounds numpy's double exp (both within about an ulp in double).
#include <climits>
#include "common.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int MERGE_THREADS = 512;

struct NmsParams { float sigma, Nt, threshold; int method; };

// Python's min(a, b) / max(a, b) on two floats: the first argument unless the second is strictly smaller / larger.
__device__ __forceinline__ float py_min(float a, float b) { return b < a ? b : a; }
__device__ __forceinline__ float py_max(float a, float b) { return b > a ? b : a; }

// decayed score of row r against the max row t; *hit = the weight was applied (the row overlaps, iw > 0 and ih > 0)
__device__ __forceinline__ float decay_score(const float t[5], const float* r, const NmsParams& p, bool* hit) {
  const float x1 = r[0], y1 = r[1], x2 = r[2], y2 = r[3], s = r[4];
  *hit = false;
  const float area = __double2float_rn(__dmul_rn(__dadd_rn((double)__fsub_rn(x2, x1), 1.0), __dadd_rn((double)__fsub_rn(y2, y1), 1.0)));
  const float iw = __double2float_rn(__dadd_rn((double)__fsub_rn(py_min(t[2], x2), py_max(t[0], x1)), 1.0));
  if (!(iw > 0.f)) return s;
  const float ih = __double2float_rn(__dadd_rn((double)__fsub_rn(py_min(t[3], y2), py_max(t[1], y1)), 1.0));
  if (!(ih > 0.f)) return s;
  const float inter = __fmul_rn(iw, ih);
  double u = __dmul_rn(__dadd_rn((double)__fsub_rn(t[2], t[0]), 1.0), __dadd_rn((double)__fsub_rn(t[3], t[1]), 1.0));
  u = __dsub_rn(__dadd_rn(u, (double)area), (double)inter);
  const float ov = __fdiv_rn(inter, __double2float_rn(u));
  float w;
  if (p.method == 1) w = ov > p.Nt ? __double2float_rn(__dsub_rn(1.0, (double)ov)) : 1.f;
  else if (p.method == 2) w = __double2float_rn(exp((double)__fdiv_rn(-__fmul_rn(ov, ov), p.sigma)));
  else w = ov > p.Nt ? 0.f : 1.f;
  *hit = true;
  return __fmul_rn(w, s);
}

// flagged rows among the relative indices [0, x) of the current pass: fw[0..31] flag words, fw[32..63] their exclusive prefix
__device__ __forceinline__ int flagged_before(const unsigned* fw, int x, int n, int F) {
  if (x >= n) return F;
  return (int)fw[32 + (x >> 5)] + __popc(fw[x >> 5] & ((1u << (x & 31)) - 1u));
}
__device__ __forceinline__ bool is_flagged(const unsigned* fw, int x) { return (fw[x >> 5] >> (x & 31)) & 1u; }

// Soft-NMS of one segment by one warp, all in shared memory: rows [len][5] in place, sc [len] decayed scores, hole [len],
// fw [64] flag words.  len <= CDN_SOFT_NMS_MAX_LEN.  Returns the final N.
__device__ int warp_soft_nms(float* rows, float* sc, short* hole, unsigned* fw, int len, const NmsParams p) {
  const int lane = threadIdx.x & 31;
  int N = len;
  for (int i = 0; i < N; ++i) {
    // first maximum of [i, N) (strict `<` of the mirror: row i and then the lowest index win ties)
    float best = 0.f; int bi = INT_MAX;
    for (int j = i + lane; j < N; j += 32) {
      const float s = rows[j * 5 + 4];
      if (bi == INT_MAX || s > best) { best = s; bi = j; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ob = __shfl_xor_sync(FULL, best, o);
      const int oi = __shfl_xor_sync(FULL, bi, o);
      if (oi != INT_MAX && (bi == INT_MAX || ob > best || (!(best > ob) && oi < bi))) { best = ob; bi = oi; }
    }
    __syncwarp();
    if (lane < 5 && bi != i) {
      const float a = rows[i * 5 + lane], b = rows[bi * 5 + lane];
      rows[i * 5 + lane] = b; rows[bi * 5 + lane] = a;
    }
    __syncwarp();
    float t[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) t[c] = rows[i * 5 + c];
    const int A = i + 1, n = N - A;
    if (n <= 0) break;
    const int nw = (n + 31) >> 5;
    for (int c = 0; c < nw; ++c) {
      const int k = c * 32 + lane;
      bool flag = false;
      if (k < n) {
        bool hit;
        const float ds = decay_score(t, rows + (A + k) * 5, p, &hit);
        sc[A + k] = ds;
        flag = hit && ds < p.threshold;
      }
      const unsigned w = __ballot_sync(FULL, flag);
      if (lane == 0) fw[c] = w;
    }
    __syncwarp();
    const int v = lane < nw ? __popc(fw[lane]) : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += u;
    }
    fw[32 + lane] = (unsigned)(incl - v);
    const int F = __shfl_sync(FULL, incl, 31);
    __syncwarp();
    if (F == 0) {                                    // nothing discarded: scores in place
      for (int k = lane; k < n; k += 32) rows[(A + k) * 5 + 4] = sc[A + k];
      __syncwarp();
      continue;
    }
    const int nk = n - F;
    for (int k = lane; k < nk; k += 32) {            // front rows: kept in place, flagged ones become holes
      if (is_flagged(fw, k)) hole[flagged_before(fw, k, n, F)] = (short)k;
      else rows[(A + k) * 5 + 4] = sc[A + k];
    }
    __syncwarp();
    int R = n;                                       // lowest unflagged back row
    for (int k = nk + lane; k < n; k += 32) {        // unflagged back rows fill the holes, the top one the first hole
      if (is_flagged(fw, k)) continue;
      R = min(R, k);
      const int rank = (n - 1 - k) - (F - flagged_before(fw, k + 1, n, F));
      float* d = rows + (A + hole[rank]) * 5;
      const float* s = rows + (A + k) * 5;
      d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = s[3]; d[4] = sc[A + k];
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) R = min(R, __shfl_xor_sync(FULL, R, o));
    if (lane == 0 && R > nk) {                       // the mirror's last discard copies slot N' onto itself
      const int src = R - nk >= 2 ? nk + 1 : nk;
      float* d = rows + (A + nk) * 5;
      const float* s = rows + (A + src) * 5;
      d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = s[3]; d[4] = sc[A + src];
    }
    __syncwarp();
    N = A + nk;
  }
  return N;
}

__host__ __device__ __forceinline__ size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// one warp per segment; dynamic shared memory = nms_smem_bytes(max_len)
__global__ void __launch_bounds__(32) soft_nms_kernel(float* __restrict__ boxes, const int32_t* __restrict__ seg_off, int max_len,
                                                      NmsParams p, int32_t* __restrict__ keep) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int seg = blockIdx.x, lane = threadIdx.x;
  const int begin = seg_off[seg], end = seg_off[seg + 1], len = end - begin;
  if (begin < 0 || len < 0 || len > max_len) {       // outside the launch's promise: the segment is left untouched
    if (lane == 0) keep[seg] = -1;
    return;
  }
  unsigned* fw = (unsigned*)smem;
  float* rows = (float*)(smem + 64 * sizeof(unsigned));
  float* sc = rows + (size_t)max_len * 5;
  short* hole = (short*)(sc + max_len);
  float* g = boxes + (size_t)begin * 5;
  for (int e = lane; e < len * 5; e += 32) rows[e] = g[e];
  __syncwarp();
  const int n = warp_soft_nms(rows, sc, hole, fw, len, p);
  for (int e = lane; e < len * 5; e += 32) g[e] = rows[e];
  if (lane == 0) keep[seg] = n;
}

size_t nms_smem_bytes(int max_len) { return 64 * sizeof(unsigned) + (size_t)max_len * (6 * sizeof(float) + sizeof(short)); }

struct MergeParams {
  const float* grouped; const int32_t* counts;
  float* out_rows; int32_t* out_counts;
  int S, K, C, nms, max_per_image;
  NmsParams np;
  float scale[CDN_MERGE_MAX_SCALES];
};

// in-place exclusive scan of a[0..n) by one warp; a[n] = total
__device__ void warp_exclusive_scan(int* a, int n) {
  const int lane = threadIdx.x & 31;
  int carry = 0;
  for (int base = 0; base < n; base += 32) {
    const int k = base + lane;
    const int v = k < n ? a[k] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(FULL, incl, o);
      if (lane >= o) incl += u;
    }
    if (k < n) a[k] = carry + incl - v;
    carry += __shfl_sync(FULL, incl, 31);
  }
  if (lane == 0) a[n] = carry;
  __syncwarp();
}

size_t merge_smem_bytes(int S, int K, int C) {
  const size_t T = (size_t)S * K;
  return align16((size_t)(MERGE_THREADS / 32) * 64 * sizeof(unsigned)) + align16(T * 5 * sizeof(float)) + align16(T * sizeof(float)) +
         align16(T * sizeof(short)) * 2 + align16((size_t)S * (C + 1) * sizeof(int)) + align16((size_t)(C + 1) * sizeof(int)) +
         align16((size_t)C * sizeof(int)) + 64 * sizeof(int);
}

// one CTA per image
__global__ void __launch_bounds__(MERGE_THREADS) ctdet_merge_kernel(const MergeParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int S = p.S, K = p.K, C = p.C, T = S * K;
  unsigned char* q = smem;
  auto take = [&](size_t bytes) { unsigned char* r = q; q += align16(bytes); return r; };
  unsigned* fw = (unsigned*)take((size_t)(MERGE_THREADS / 32) * 64 * sizeof(unsigned));
  float* rows = (float*)take((size_t)T * 5 * sizeof(float));
  float* sc = (float*)take((size_t)T * sizeof(float));
  short* hole = (short*)take((size_t)T * sizeof(short));
  short* rcls = (short*)take((size_t)T * sizeof(short));
  int* pcs = (int*)take((size_t)S * (C + 1) * sizeof(int));      // per scale: exclusive prefix of the class counts, [C] = total
  int* coff = (int*)take((size_t)(C + 1) * sizeof(int));         // per class: first row of the merged class, [C] = total
  int* ccnt = (int*)take((size_t)C * sizeof(int));               // per class: rows kept by the cut
  int* red = (int*)take(64 * sizeof(int));

  const int32_t* cnt = p.counts + (size_t)b * S * C;
  for (int e = tid; e < S * C; e += blockDim.x) {
    const int s = e / C, j = e % C;
    pcs[s * (C + 1) + j] = min(max(cnt[e], 0), K);
  }
  for (int j = tid; j < C; j += blockDim.x) ccnt[j] = 0;
  for (int e = tid; e < T; e += blockDim.x) {        // defined rows even for counts that are not group_by_class's
    rcls[e] = 0;
#pragma unroll
    for (int c = 0; c < 5; ++c) rows[e * 5 + c] = 0.f;
  }
  __syncthreads();
  for (int j = tid; j < C; j += blockDim.x) {
    int t = 0;
    for (int s = 0; s < S; ++s) t += pcs[s * (C + 1) + j];
    coff[j] = t;
  }
  __syncthreads();
  for (int s = warp; s <= S; s += nwarps) warp_exclusive_scan(s < S ? pcs + s * (C + 1) : coff, C);
  __syncthreads();
  const int total = min(coff[C], T);

  // gather: class-major, scale order inside a class (np.vstack of merge_outputs), coordinates divided by the scale
  for (int e = tid; e < T; e += blockDim.x) {
    const int s = e / K, r = e % K;
    const int* pc = pcs + s * (C + 1);
    if (r >= pc[C]) continue;
    int lo = 0, hi = C - 1;                          // the class whose row range [pc[j], pc[j+1]) holds r
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (pc[mid] <= r) lo = mid; else hi = mid - 1;
    }
    const int j = lo;
    int dst = coff[j] + (r - pc[j]);
    for (int u = 0; u < s; ++u) dst += pcs[u * (C + 1) + j + 1] - pcs[u * (C + 1) + j];
    if (dst >= total) continue;
    const float* src = p.grouped + ((size_t)(b * S + s) * K + r) * 6;
    const float d = p.scale[s];
    float* o = rows + (size_t)dst * 5;
    o[0] = __fdiv_rn(src[0], d); o[1] = __fdiv_rn(src[1], d); o[2] = __fdiv_rn(src[2], d); o[3] = __fdiv_rn(src[3], d);
    o[4] = src[4];
    rcls[dst] = (short)j;
  }
  __syncthreads();

  if (S > 1 || p.nms) {
    for (int j = warp; j < C; j += nwarps) {
      const int o = coff[j], len = min(coff[j + 1], total) - o;
      if (len > 1) warp_soft_nms(rows + (size_t)o * 5, sc + o, hole + o, fw + warp * 64, len, p.np);
    }
    __syncthreads();
  }

  // cut: the score at ascending rank total - max_per_image (np.partition), rows with score >= cut survive in their order
  const bool do_cut = total > p.max_per_image;
  if (tid == 0) red[40] = __float_as_int(-INFINITY);
  __syncthreads();
  if (do_cut) {
    const int rank = total - p.max_per_image;
    for (int r = tid; r < total; r += blockDim.x) {
      const float s = rows[r * 5 + 4];
      int lt = 0, le = 0;
      for (int u = 0; u < total; ++u) {
        const float v = rows[u * 5 + 4];
        lt += v < s; le += v <= s;
      }
      if (lt <= rank && rank < le) red[40] = __float_as_int(s);
    }
  }
  __syncthreads();
  const float cut = __int_as_float(red[40]);
  float* out = p.out_rows + (size_t)b * T * 5;
  int carry = 0;
  for (int base = 0; base < total; base += blockDim.x) {
    const int r = base + tid;
    const bool keep = r < total && (!do_cut || rows[r * 5 + 4] >= cut);
    const unsigned m = __ballot_sync(FULL, keep);
    if (lane == 0) red[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
      const int v = lane < nwarps ? red[lane] : 0;
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += u;
      }
      red[lane] = incl - v;
      if (lane == 31) red[32] = incl;
    }
    __syncthreads();
    if (keep) {
      const int pos = carry + red[warp] + __popc(m & ((1u << lane) - 1u));
      const float* s = rows + (size_t)r * 5;
      float* d = out + (size_t)pos * 5;
      d[0] = s[0]; d[1] = s[1]; d[2] = s[2]; d[3] = s[3]; d[4] = s[4];
      atomicAdd(&ccnt[rcls[r]], 1);
    }
    carry += red[32];
    __syncthreads();
  }
  for (int j = tid; j < C; j += blockDim.x) p.out_counts[(size_t)b * C + j] = ccnt[j];
}

bool g_merge_attr[64], g_nms_attr[64];

}  // namespace

extern "C" int cdn_soft_nms(float* d_boxes, const int32_t* d_seg_off, int n_seg, int max_len, float sigma, float Nt, float threshold,
                            int method, int32_t* d_keep, cdn_stream_t stream) {
  CDN_CHECK(d_boxes && d_seg_off && d_keep && n_seg >= 0 && max_len >= 0 && method >= 0 && method <= 2, CDN_ERR_INVALID,
            "soft_nms: bad arguments");
  CDN_CHECK(max_len <= CDN_SOFT_NMS_MAX_LEN, CDN_ERR_INVALID, "soft_nms: segments of up to %d rows, %d requested",
            CDN_SOFT_NMS_MAX_LEN, max_len);
  CDN_CHECK(n_seg <= 0x7fffffff - 1, CDN_ERR_INVALID, "soft_nms: too many segments");
  if (n_seg == 0) return 0;
  const size_t smem = nms_smem_bytes(max_len);
  if (smem > 48 * 1024 && cdn_first_on_device(g_nms_attr))
    CDN_CUDA(cudaFuncSetAttribute(soft_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)nms_smem_bytes(CDN_SOFT_NMS_MAX_LEN)));
  NmsParams p{sigma, Nt, threshold, method};
  soft_nms_kernel<<<n_seg, 32, smem, (cudaStream_t)stream>>>(d_boxes, d_seg_off, max_len, p, d_keep);
  CDN_LAUNCH_CHECK("soft_nms_kernel");
  return 0;
}

extern "C" int cdn_ctdet_merge(const float* d_grouped, const int32_t* d_counts, int batch, int scales, int K, int num_classes,
                               const float* h_scales, int nms, int max_per_image, float* d_rows, int32_t* d_class_counts,
                               cdn_stream_t stream) {
  CDN_CHECK(d_grouped && d_counts && h_scales && d_rows && d_class_counts && batch >= 0 && K >= 1 && max_per_image >= 1,
            CDN_ERR_INVALID, "ctdet_merge: bad arguments");
  CDN_CHECK(scales >= 1 && scales <= CDN_MERGE_MAX_SCALES, CDN_ERR_INVALID, "ctdet_merge: 1 to %d scales, %d given",
            CDN_MERGE_MAX_SCALES, scales);
  CDN_CHECK(num_classes >= 1 && num_classes <= CDN_MERGE_MAX_CLASSES, CDN_ERR_INVALID, "ctdet_merge: 1 to %d classes, %d given",
            CDN_MERGE_MAX_CLASSES, num_classes);
  CDN_CHECK((long long)scales * K <= CDN_SOFT_NMS_MAX_LEN, CDN_ERR_INVALID,
            "ctdet_merge: scales x K = %lld rows per image, the limit is %d", (long long)scales * K, CDN_SOFT_NMS_MAX_LEN);
  MergeParams p;
  for (int s = 0; s < scales; ++s) {
    CDN_CHECK(h_scales[s] > 0.f && h_scales[s] <= 3.4e38f, CDN_ERR_INVALID, "ctdet_merge: scale %d is %g", s, (double)h_scales[s]);
    p.scale[s] = h_scales[s];
  }
  for (int s = scales; s < CDN_MERGE_MAX_SCALES; ++s) p.scale[s] = 1.f;
  if (batch == 0) return 0;
  p.grouped = d_grouped; p.counts = d_counts; p.out_rows = d_rows; p.out_counts = d_class_counts;
  p.S = scales; p.K = K; p.C = num_classes; p.nms = nms ? 1 : 0; p.max_per_image = max_per_image;
  p.np = NmsParams{0.5f, 0.5f, 0.001f, 2};                  // merge_outputs: soft_nms(Nt=0.5, method=2), ctdet.py:63-64
  const size_t smem = merge_smem_bytes(scales, K, num_classes);
  if (smem > 48 * 1024 && cdn_first_on_device(g_merge_attr))
    CDN_CUDA(cudaFuncSetAttribute(ctdet_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)merge_smem_bytes(CDN_MERGE_MAX_SCALES, CDN_SOFT_NMS_MAX_LEN / CDN_MERGE_MAX_SCALES,
                                                        CDN_MERGE_MAX_CLASSES)));
  ctdet_merge_kernel<<<batch, MERGE_THREADS, smem, (cudaStream_t)stream>>>(p);
  CDN_LAUNCH_CHECK("ctdet_merge_kernel");
  return 0;
}
