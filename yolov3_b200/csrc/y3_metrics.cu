// yolov3_b200 — validation metrics on the device (SURVEY §8(f) row f2, second half): the reference's ap_per_class +
// compute_ap (utils/metrics.py:22-120, called at val.py:424-426) and ConfusionMatrix.process_batch (utils/metrics.py:134-178,
// called per image at val.py:390,406).  The reference copies every detection's statistics to the host and runs numpy there.
//
// ap_per_class.  Rows (conf, cls, tp[niou]) are sorted by (class, conf descending, row) with a stable LSD radix sort on a 64-bit
// key (class << 32 | order-preserving conf bits), the row index as payload.  Padded rows and rows whose class is outside
// [0, nc) go to a sentinel bucket (class nc) behind every real class, so nothing needs the number of valid rows on the host.
// Per class the order equals the reference's argsort(-conf) followed by a boolean select, except among bit-equal
// confidences: numpy's argsort is unstable there, ours keeps the input row order (DESIGN.md §2).
// A curve (class c, IoU threshold j) is then described exactly by the sorted positions of its true positives: the t-th true
// positive (0-based) at position s has tpc = t + 1 and tpc + fpc = s + 1, every other position inherits tpc from the last
// true positive before it.  Precision restricted to a run of false positives falls, so the suffix maximum of precision (the
// reference's envelope) at position p is max(precision(p), max over true positives at or after p) — one suffix-max pass over
// the true positives, not over every row.  np.interp and np.trapezoid are then evaluated exactly as numpy does it (see
// ap_compute_kernel), so AP is bit-identical to the reference.
//
// ConfusionMatrix.process_batch.  One block per image: labels staged in shared memory, class-agnostic pairs with
// IoU > iou_thres; each detection keeps its highest-IoU label, each label the highest-IoU detection among those; counts go
// to the caller's int64 [(nc+1)^2] matrix with integer atomics (order-independent, so deterministic).  Ties on bit-equal IoU
// (numpy's argsort()[::-1] is unspecified there): the lower label index, then the lower detection index wins.
#include <algorithm>

#include "y3_box.cuh"
#include "y3_common.cuh"
#include "y3_internal.h"

namespace y3 {
namespace {

typedef unsigned long long u64;

constexpr int kRadixThreads = 256;
constexpr int kRadixItems = 16;
constexpr int kRadixTile = kRadixThreads * kRadixItems;
constexpr int kScanThreads = 1024;
constexpr int kPosThreads = 512;
constexpr int kPosItems = 4;
constexpr int kApThreads = 256;
constexpr int kApPoints = 101;   // compute_ap: np.linspace(0, 1, 101)
constexpr int kPrPoints = 1000;  // ap_per_class: px = np.linspace(0, 1, 1000)
constexpr int kConfMaxLabels = 1024;

// ------------------------------------------------------------------------------------------------ block helpers
// exclusive prefix sum of one int per thread; `total` = block sum.  NT threads, NT % 32 == 0; s_w holds >= 32 ints.
template <int NT>
__device__ __forceinline__ int block_excl_scan(int v, int& total, int* s_w) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_w[w] = x;
  __syncthreads();
  if (w == 0) {
    int t = lane < NT / 32 ? s_w[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, t, o);
      if (lane >= o) t += y;
    }
    if (lane < NT / 32) s_w[lane] = t;
  }
  __syncthreads();
  total = s_w[NT / 32 - 1];
  const int excl = x - v + (w ? s_w[w - 1] : 0);
  __syncthreads();
  return excl;
}

// ------------------------------------------------------------------------------------------------ ap_per_class
struct ApArgs {
  const float* conf;
  long long conf_stride;
  const float* cls;
  long long cls_stride;
  const uint8_t* tp;  // [n, niou]
  int niou, n;
  const int* det_count;  // [n / rows_per_image] or null
  long long rows_per_image;
  const float* tcls;
  long long tcls_stride;
  int nt, nc;
  double eps;
  // workspace
  u64* key[2];
  int* val[2];
  const u64* skey;  // sorted keys / row indices (the buffers the last radix pass wrote)
  const int* sval;
  int* hist;
  int nblocks;
  int* seg;     // [nc + 1] first sorted position of each class; seg[nc] = start of the sentinel bucket
  int* ntc;     // [nc] label count per class
  int* ntoff;   // [nc] exclusive prefix of ntc: a class's slice of tp_pos / smax
  int* tp_cnt;  // [niou, nc] true positives per curve
  int* tp_pos;  // [niou, nt] sorted position (inside the class) of each true positive, in order
  double* smax; // [niou, nt] suffix maximum of the true positives' precision
  double* pcurve;  // [nc, 1000]
  double* rcurve;
  // outputs
  double *ap, *p, *r, *f1, *tp_out, *fp_out;
  int64_t* nt_out;
  uint8_t* present;
  int* f1_index;
  int* status;  // [3]: prediction rows with a class outside [0,nc), target classes outside [0,nc), curves with tp > labels
};

// integral class id in [0, nc) (the reference compares pred_cls == unique target class values; NaN and fractions never match)
__device__ __forceinline__ int class_id(float v, int nc) {
  return (v >= 0.0f && v < static_cast<float>(nc) && v == floorf(v)) ? static_cast<int>(v) : -1;
}

// descending-confidence sort key: larger conf -> smaller key; -0 == +0; NaN last (numpy sorts NaN of -conf to the end)
__device__ __forceinline__ uint32_t conf_desc_key(float c) {
  if (c != c) return 0xffffffffu;
  const uint32_t u = (c == 0.0f) ? 0u : __float_as_uint(c);
  const uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ~asc;
}

__global__ void __launch_bounds__(256) ap_init_kernel(const ApArgs a) {
  pdl_entry();
  for (int i = threadIdx.x; i < a.nc; i += blockDim.x) a.ntc[i] = 0;
  if (threadIdx.x < 3) a.status[threadIdx.x] = 0;
}

__global__ void __launch_bounds__(256) ap_targets_kernel(const ApArgs a) {
  pdl_entry();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.nt; i += gridDim.x * blockDim.x) {
    const int c = class_id(a.tcls[static_cast<long long>(i) * a.tcls_stride], a.nc);
    if (c >= 0)
      atomicAdd(&a.ntc[c], 1);
    else
      atomicAdd(&a.status[1], 1);
  }
}

__global__ void __launch_bounds__(256) ap_keys_kernel(const ApArgs a) {
  pdl_entry();
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < a.n; r += gridDim.x * blockDim.x) {
    bool valid = true;
    if (a.det_count) valid = (r % a.rows_per_image) < a.det_count[r / a.rows_per_image];
    u64 key = (static_cast<u64>(a.nc) << 32) | 0xffffffffu;
    if (valid) {
      const int c = class_id(a.cls[static_cast<long long>(r) * a.cls_stride], a.nc);
      if (c >= 0)
        key = (static_cast<u64>(c) << 32) | conf_desc_key(a.conf[static_cast<long long>(r) * a.conf_stride]);
      else
        atomicAdd(&a.status[0], 1);
    }
    a.key[0][r] = key;
    a.val[0][r] = r;
  }
}

// radix pass, step 1: digit histogram of every tile, stored digit-major (hist[d * nblocks + tile])
__global__ void __launch_bounds__(kRadixThreads) radix_hist_kernel(const u64* __restrict__ keys, int n, int shift, int* hist,
                                                                   int nblocks) {
  pdl_entry();
  __shared__ int s[256];
  s[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kRadixTile;
#pragma unroll 4
  for (int i = 0; i < kRadixItems; ++i) {
    const int idx = base + i * kRadixThreads + threadIdx.x;
    if (idx < n) atomicAdd(&s[(keys[idx] >> shift) & 255u], 1);
  }
  __syncthreads();
  hist[threadIdx.x * nblocks + blockIdx.x] = s[threadIdx.x];
}

// in-place exclusive prefix sum of len ints by one block (the radix histograms: digit-major order = global offsets)
__global__ void __launch_bounds__(kScanThreads) scan_kernel(int* a, int len) {
  pdl_entry();
  __shared__ int s_w[32];
  int carry = 0;
  for (int base = 0; base < len; base += kScanThreads * 4) {
    int v[4], sum = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int idx = base + threadIdx.x * 4 + k;
      v[k] = idx < len ? a[idx] : 0;
      sum += v[k];
    }
    int tot;
    int run = carry + block_excl_scan<kScanThreads>(sum, tot, s_w);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int idx = base + threadIdx.x * 4 + k;
      if (idx < len) a[idx] = run;
      run += v[k];
    }
    carry += tot;
  }
}

// radix pass, step 2: stable scatter.  A tile is read in rounds of 256 consecutive items; inside a round an item's rank among
// equal digits is (earlier warps' counts) + (lower lanes of its own warp), so the input order survives inside a digit.
__global__ void __launch_bounds__(kRadixThreads) radix_scatter_kernel(const u64* __restrict__ kin, const int* __restrict__ vin,
                                                                      u64* __restrict__ kout, int* __restrict__ vout, int n,
                                                                      int shift, const int* __restrict__ hist, int nblocks) {
  pdl_entry();
  __shared__ int s_run[256];
  __shared__ int s_wc[kRadixThreads / 32][256];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  s_run[tid] = hist[tid * nblocks + blockIdx.x];
  const int base = blockIdx.x * kRadixTile;
  for (int it = 0; it < kRadixItems; ++it) {
#pragma unroll
    for (int k = 0; k < kRadixThreads / 32; ++k) s_wc[k][tid] = 0;
    __syncthreads();
    const int idx = base + it * kRadixThreads + tid;
    const bool ok = idx < n;
    const u64 key = ok ? kin[idx] : 0ull;
    const int val = ok ? vin[idx] : 0;
    const int d = ok ? static_cast<int>((key >> shift) & 255u) : 256 + lane;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (ok && rank == 0) s_wc[w][d] = __popc(peers);
    __syncthreads();
    {
      int run = s_run[tid];
#pragma unroll
      for (int k = 0; k < kRadixThreads / 32; ++k) {
        const int c = s_wc[k][tid];
        s_wc[k][tid] = run;
        run += c;
      }
      s_run[tid] = run;
    }
    __syncthreads();
    if (ok) {
      const int dst = s_wc[w][d] + rank;
      kout[dst] = key;
      vout[dst] = val;
    }
    __syncthreads();
  }
}

// class segments of the sorted order, label counts -> offsets, nt / present outputs
__global__ void __launch_bounds__(kScanThreads) ap_segments_kernel(const ApArgs a) {
  pdl_entry();
  __shared__ int s_w[32];
  for (int c = threadIdx.x; c <= a.nc; c += blockDim.x) {
    const u64 want = static_cast<u64>(c) << 32;
    int lo = 0, hi = a.n;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (a.skey[mid] < want)
        lo = mid + 1;
      else
        hi = mid;
    }
    a.seg[c] = lo;
  }
  int carry = 0;
  for (int base = 0; base < a.nc; base += kScanThreads) {
    const int c = base + threadIdx.x;
    const int v = c < a.nc ? a.ntc[c] : 0;
    int tot;
    const int ex = block_excl_scan<kScanThreads>(v, tot, s_w);
    if (c < a.nc) {
      a.ntoff[c] = carry + ex;
      a.nt_out[c] = v;
      a.present[c] = v > 0;
    }
    carry += tot;
  }
}

// grid (niou, nc): ordered list of the true positives' positions of curve (class, threshold), at most n_l of them
__global__ void __launch_bounds__(kPosThreads) ap_tp_positions_kernel(const ApArgs a) {
  pdl_entry();
  __shared__ int s_w[32];
  const int j = blockIdx.x, c = blockIdx.y;
  const int s0 = a.seg[c], m = a.seg[c + 1] - s0, nl = a.ntc[c];
  if (m == 0 || nl == 0) {
    if (threadIdx.x == 0) a.tp_cnt[j * a.nc + c] = 0;
    return;
  }
  int* pos = a.tp_pos + static_cast<long long>(j) * a.nt + a.ntoff[c];
  const int* perm = a.sval + s0;
  int carry = 0;
  for (int base = 0; base < m; base += kPosThreads * kPosItems) {
    int f[kPosItems], cnt = 0;
#pragma unroll
    for (int k = 0; k < kPosItems; ++k) {
      const int s = base + threadIdx.x * kPosItems + k;
      f[k] = s < m ? (a.tp[static_cast<long long>(perm[s]) * a.niou + j] != 0) : 0;
      cnt += f[k];
    }
    int tot;
    int o = carry + block_excl_scan<kPosThreads>(cnt, tot, s_w);
#pragma unroll
    for (int k = 0; k < kPosItems; ++k) {
      if (f[k]) {
        if (o < nl) pos[o] = base + threadIdx.x * kPosItems + k;
        ++o;
      }
    }
    carry += tot;
  }
  if (threadIdx.x == 0) {
    a.tp_cnt[j * a.nc + c] = carry;
    if (carry > nl) atomicAdd(&a.status[2], 1);  // outside the contract: the reference's mrec is not monotone then
  }
}

// One curve: K true positives at sorted positions pos[0..K) of a class with m predictions and n_l labels.
struct Curve {
  const int* pos;
  const double* smax;
  int K, m;
  double den_l;  // n_l + eps (the reference's recall denominator)
};
__device__ __forceinline__ int tpc_at(const Curve& cv, int s) {  // true positives at positions <= s
  int lo = 0, hi = cv.K;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cv.pos[mid] <= s)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}
__device__ __forceinline__ double recall_at(const Curve& cv, int s) {
  return __ddiv_rn(static_cast<double>(tpc_at(cv, s)), cv.den_l);
}
__device__ __forceinline__ double precision_at(const Curve& cv, int s) {  // tpc / (tpc + fpc), tpc + fpc = s + 1
  return __ddiv_rn(static_cast<double>(tpc_at(cv, s)), static_cast<double>(s + 1));
}
// max(precision[p..m), 0): precision at p itself or at a true positive at or after p
__device__ __forceinline__ double suffix_max_at(const Curve& cv, int p) {
  if (p >= cv.m) return 0.0;
  int lo = 0, hi = cv.K;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cv.pos[mid] < p)
      lo = mid + 1;
    else
      hi = mid;
  }
  double v = precision_at(cv, p);
  if (lo < cv.K) v = fmax(v, cv.smax[lo]);
  return v;
}
// compute_ap's arrays, never materialised: mrec = [0, recall..., 1], envelope = suffix max of [1, precision..., 0]
__device__ __forceinline__ double mrec_at(const Curve& cv, int i) {
  return i == 0 ? 0.0 : (i <= cv.m ? recall_at(cv, i - 1) : 1.0);
}
__device__ __forceinline__ double env_at(const Curve& cv, int i) {
  return i == 0 ? 1.0 : (i <= cv.m ? suffix_max_at(cv, i - 1) : 0.0);  // precision <= 1, so env[0] = 1
}
// numpy's interp step once the index is known: j = (number of xp <= x) - 1, len = number of xp, fp(j) = f(j)
template <typename XP, typename FP>
__device__ __forceinline__ double interp_at(double x, int j, int len, double left, XP xp, FP fp) {
  if (j < 0) return left;
  if (j >= len - 1) return fp(len - 1);
  const double xj = xp(j);
  if (xj == x) return fp(j);
  const double fj = fp(j);
  const double slope = __ddiv_rn(__dsub_rn(fp(j + 1), fj), __dsub_rn(xp(j + 1), xj));
  return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xj)), fj);
}

// grid (niou + 1, nc).  x < niou: AP of curve (class y, threshold x).  x == niou: the threshold-0 P and R curves at px.
__global__ void __launch_bounds__(kApThreads) ap_compute_kernel(const ApArgs a) {
  pdl_entry();
  __shared__ double s_y[kApPoints];
  __shared__ double s_wm[kApThreads / 32];
  const int j = blockIdx.x, c = blockIdx.y, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int s0 = a.seg[c], m = a.seg[c + 1] - s0, nl = a.ntc[c];
  const bool empty = (m == 0 || nl == 0);
  if (j == a.niou) {  // ---- P / R curves (ap_per_class: np.interp(-px, -conf[i], recall[:, 0] / precision[:, 0], left=0 / 1))
    double* pc = a.pcurve + static_cast<long long>(c) * kPrPoints;
    double* rc = a.rcurve + static_cast<long long>(c) * kPrPoints;
    Curve cv;
    cv.pos = a.tp_pos + a.ntoff[c];
    cv.smax = nullptr;
    cv.K = empty ? 0 : min(a.tp_cnt[c], nl);
    cv.m = m;
    cv.den_l = __dadd_rn(static_cast<double>(nl), a.eps);
    const int* perm = a.sval + s0;
    auto xp = [&](int s) { return -static_cast<double>(a.conf[static_cast<long long>(perm[s]) * a.conf_stride]); };
    for (int k = tid; k < kPrPoints; k += blockDim.x) {
      if (empty) {
        pc[k] = 0.0;
        rc[k] = 0.0;
        continue;
      }
      const double px = k == kPrPoints - 1 ? 1.0 : __dmul_rn(static_cast<double>(k), 1.0 / 999.0);
      const double x = -px;
      int lo = 0, hi = m;  // number of -conf <= -px
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (xp(mid) <= x)
          lo = mid + 1;
        else
          hi = mid;
      }
      rc[k] = interp_at(x, lo - 1, m, 0.0, xp, [&](int s) { return recall_at(cv, s); });
      pc[k] = interp_at(x, lo - 1, m, 1.0, xp, [&](int s) { return precision_at(cv, s); });
    }
    return;
  }
  // ---- AP (compute_ap, utils/metrics.py:94-120)
  if (empty) {
    if (tid == 0) a.ap[static_cast<long long>(c) * a.niou + j] = 0.0;
    return;
  }
  Curve cv;
  cv.pos = a.tp_pos + static_cast<long long>(j) * a.nt + a.ntoff[c];
  double* smax = a.smax + static_cast<long long>(j) * a.nt + a.ntoff[c];
  cv.smax = smax;
  cv.K = min(a.tp_cnt[j * a.nc + c], nl);
  cv.m = m;
  cv.den_l = __dadd_rn(static_cast<double>(nl), a.eps);
  // suffix maximum of the true positives' precision (t + 1) / (pos[t] + 1), in chunks from the end (max is exact: any order)
  double carry = 0.0;
  for (int hi = cv.K; hi > 0; hi -= kApThreads) {
    const int lo = max(hi - kApThreads, 0), t = lo + tid;
    double v = t < hi ? __ddiv_rn(static_cast<double>(t + 1), static_cast<double>(cv.pos[t] + 1)) : 0.0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_down_sync(0xffffffffu, v, o);
      if (lane + o < 32) v = fmax(v, y);
    }
    if (lane == 0) s_wm[w] = v;
    __syncthreads();
    double later = carry, all = carry;
    for (int k = 0; k < kApThreads / 32; ++k) {
      if (k > w) later = fmax(later, s_wm[k]);
      all = fmax(all, s_wm[k]);
    }
    if (t < hi) smax[t] = fmax(v, later);
    __syncthreads();
    carry = all;
  }
  __syncthreads();
  // np.interp(x, mrec, mpre) at x = np.linspace(0, 1, 101)
  if (tid < kApPoints) {
    const double x = tid < kApPoints - 1 ? __dmul_rn(static_cast<double>(tid), 0.01) : 1.0;
    int lo = 0, hi = m;  // number of recall values <= x
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (recall_at(cv, mid) <= x)
        lo = mid + 1;
      else
        hi = mid;
    }
    const int jj = lo + (x >= 1.0 ? 1 : 0);  // mrec[0] = 0 <= x always; mrec[m + 1] = 1
    s_y[tid] = interp_at(x, jj, m + 2, 0.0, [&](int i) { return mrec_at(cv, i); }, [&](int i) { return env_at(cv, i); });
  }
  __syncthreads();
  // np.trapezoid(y, x) = add.reduce(d * (y[1:] + y[:-1]) / 2.0): numpy's pairwise sum of 100 terms = eight interleaved
  // partial sums, combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the last 4 terms in order
  if (tid == 0) {
    auto xs = [](int i) { return i < kApPoints - 1 ? __dmul_rn(static_cast<double>(i), 0.01) : 1.0; };
    auto term = [&](int i) {
      return __ddiv_rn(__dmul_rn(__dsub_rn(xs(i + 1), xs(i)), __dadd_rn(s_y[i + 1], s_y[i])), 2.0);
    };
    double r8[8];
    for (int q = 0; q < 8; ++q) r8[q] = term(q);
    int i = 8;
    for (; i < 96; i += 8)
      for (int q = 0; q < 8; ++q) r8[q] = __dadd_rn(r8[q], term(i + q));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r8[0], r8[1]), __dadd_rn(r8[2], r8[3])),
                           __dadd_rn(__dadd_rn(r8[4], r8[5]), __dadd_rn(r8[6], r8[7])));
    for (; i < kApPoints - 1; ++i) res = __dadd_rn(res, term(i));
    a.ap[static_cast<long long>(c) * a.niou + j] = res;
  }
}

__device__ __forceinline__ double f1_of(double p, double r, double eps) {  // 2 * p * r / (p + r + eps)
  return __ddiv_rn(__dmul_rn(__dmul_rn(2.0, p), r), __dadd_rn(__dadd_rn(p, r), eps));
}
// np.argmax order: the first NaN, else the first maximum
__device__ __forceinline__ bool argmax_better(double va, int ia, double vb, int ib) {
  const bool na = va != va, nb = vb != vb;
  if (na || nb) return na && (!nb || ia < ib);
  return va > vb || (va == vb && ia < ib);
}

// one block: f1.mean(0) over the present classes (sequential in class order, as numpy reduces axis 0), smooth(, 0.1), argmax,
// then every class's p, r, f1, tp, fp at that index
__global__ void __launch_bounds__(kScanThreads) ap_finalize_kernel(const ApArgs a) {
  pdl_entry();
  __shared__ double s_y[kPrPoints];
  __shared__ double s_bv[32];
  __shared__ int s_bi[32];
  const int tid = threadIdx.x;
  for (int k = tid; k < kPrPoints; k += blockDim.x) {
    double s = 0.0;
    int cnt = 0;
    for (int c = 0; c < a.nc; ++c) {
      if (a.ntc[c] == 0) continue;
      s = __dadd_rn(s, f1_of(a.pcurve[static_cast<long long>(c) * kPrPoints + k], a.rcurve[static_cast<long long>(c) * kPrPoints + k],
                             a.eps));
      ++cnt;
    }
    s_y[k] = __ddiv_rn(s, static_cast<double>(cnt));
  }
  __syncthreads();
  // smooth(y, f=0.1) (ultralytics): nf = 101 taps of 1/101 over y padded with 50 copies of each end value
  constexpr int nf = 101, half = nf / 2;
  const double wgt = 1.0 / nf;
  double bv = 0.0;
  int bi = 0x7fffffff;
  for (int k = tid; k < kPrPoints; k += blockDim.x) {
    double acc = 0.0;
    for (int t = 0; t < nf; ++t) {
      const int i = k + t - half;
      const double v = s_y[i < 0 ? 0 : (i >= kPrPoints ? kPrPoints - 1 : i)];
      acc = __dadd_rn(acc, __dmul_rn(v, wgt));
    }
    if (bi == 0x7fffffff || argmax_better(acc, k, bv, bi)) {
      bv = acc;
      bi = k;
    }
  }
  const int lane = tid & 31, w = tid >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_down_sync(0xffffffffu, bv, o);
    const int oi = __shfl_down_sync(0xffffffffu, bi, o);
    if (oi != 0x7fffffff && (bi == 0x7fffffff || argmax_better(ov, oi, bv, bi))) {
      bv = ov;
      bi = oi;
    }
  }
  if (lane == 0) {
    s_bv[w] = bv;
    s_bi[w] = bi;
  }
  __syncthreads();
  if (tid == 0) {
    for (int k = 1; k < static_cast<int>(blockDim.x) / 32; ++k)
      if (s_bi[k] != 0x7fffffff && argmax_better(s_bv[k], s_bi[k], s_bv[0], s_bi[0])) {
        s_bv[0] = s_bv[k];
        s_bi[0] = s_bi[k];
      }
    *a.f1_index = s_bi[0];
  }
  __syncthreads();
  const int i = s_bi[0];
  for (int c = tid; c < a.nc; c += blockDim.x) {
    double p = 0.0, r = 0.0, f = 0.0, tp = 0.0, fp = 0.0;
    if (a.ntc[c] > 0) {
      p = a.pcurve[static_cast<long long>(c) * kPrPoints + i];
      r = a.rcurve[static_cast<long long>(c) * kPrPoints + i];
      f = f1_of(p, r, a.eps);
      tp = rint(__dmul_rn(r, static_cast<double>(a.ntc[c])));                  // (r * nt).round(): half to even
      fp = rint(__dsub_rn(__ddiv_rn(tp, __dadd_rn(p, a.eps)), tp));           // (tp / (p + eps) - tp).round()
    }
    a.p[c] = p;
    a.r[c] = r;
    a.f1[c] = f;
    a.tp_out[c] = tp;
    a.fp_out[c] = fp;
  }
}

struct ApLayout {
  size_t key0, key1, val0, val1, hist, seg, ntc, ntoff, tp_cnt, tp_pos, smax, pcurve, rcurve, total;
};
ApLayout ap_layout(long long n, long long nt, int niou, int nc) {
  ApLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~static_cast<size_t>(255);
    return at;
  };
  const long long nblocks = (n + kRadixTile - 1) / kRadixTile;
  L.key0 = take(8 * n);
  L.key1 = take(8 * n);
  L.val0 = take(4 * n);
  L.val1 = take(4 * n);
  L.hist = take(4 * 256 * nblocks);
  L.seg = take(4 * (static_cast<size_t>(nc) + 1));
  L.ntc = take(4 * static_cast<size_t>(nc));
  L.ntoff = take(4 * static_cast<size_t>(nc));
  L.tp_cnt = take(4 * static_cast<size_t>(niou) * nc);
  L.tp_pos = take(4 * static_cast<size_t>(niou) * nt);
  L.smax = take(8 * static_cast<size_t>(niou) * nt);
  L.pcurve = take(8 * static_cast<size_t>(nc) * kPrPoints);
  L.rcurve = take(8 * static_cast<size_t>(nc) * kPrPoints);
  L.total = off;
  return L;
}

// ------------------------------------------------------------------------------------------------ ConfusionMatrix
struct ConfArgs {
  const float* det;      // [bs, det_stride, 6]
  const int* det_count;  // [bs] or null (max_det rows each)
  int max_det, det_stride;
  const float* labels;   // [nl, 6] (image, cls, x1, y1, x2, y2)
  int nl, nc;
  float conf, iou, eps;
  u64* matrix;   // [(nc + 1)^2], [pred, true]
  int* status;   // [2]: class ids outside [0, nc) met while counting, labels beyond kConfMaxLabels in one image
};

__device__ __forceinline__ int trunc_class(float v, int nc) {  // tensor.int() (truncation), then the range check
  return (v > -1.0f && v < static_cast<float>(nc)) ? static_cast<int>(v) : -1;
}

__global__ void __launch_bounds__(256) confusion_kernel(const ConfArgs p) {
  pdl_entry();
  __shared__ float4 s_box[kConfMaxLabels];
  __shared__ int s_cls[kConfMaxLabels];
  __shared__ u64 s_key[kConfMaxLabels];  // (IoU bits << 32) | (~detection index): the label's best pair, 0 = none
  __shared__ int s_n, s_any;
  __shared__ int s_wcnt[8];
  const int img = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) {
    s_n = 0;
    s_any = 0;
  }
  __syncthreads();
  // this image's labels in index order (block-wide ordered compaction, 256 labels per round)
  for (int base = 0; base < p.nl; base += blockDim.x) {
    const int l = base + tid;
    const bool mine = l < p.nl && static_cast<int>(p.labels[static_cast<size_t>(l) * 6]) == img;
    const unsigned bal = __ballot_sync(0xffffffffu, mine);
    const int warp = tid >> 5, lane = tid & 31;
    if (lane == 0) s_wcnt[warp] = __popc(bal);
    __syncthreads();
    int off = s_n;
    for (int k = 0; k < warp; ++k) off += s_wcnt[k];
    const int at = off + __popc(bal & ((1u << lane) - 1u));
    if (mine && at < kConfMaxLabels) {
      const float* q = p.labels + static_cast<size_t>(l) * 6;
      s_cls[at] = trunc_class(q[1], p.nc);
      s_box[at] = make_float4(q[2], q[3], q[4], q[5]);
      s_key[at] = 0ull;
    }
    __syncthreads();
    if (tid == 0) {
      int tot = 0;
      for (int k = 0; k < 8; ++k) tot += s_wcnt[k];
      s_n += tot;
    }
    __syncthreads();
  }
  const int m = min(s_n, kConfMaxLabels);
  if (tid == 0 && s_n > kConfMaxLabels) atomicAdd(&p.status[1], s_n - kConfMaxLabels);
  const int n = p.det_count ? max(min(p.det_count[img], p.max_det), 0) : p.max_det;
  const float* det = p.det + static_cast<size_t>(img) * p.det_stride * 6;
  const int stride = p.nc + 1;
  // the detection's highest-IoU label with IoU > iou_thres (strict >: the lower label index wins a tie), or -1
  auto best_label = [&](int d, float* best_iou) -> int {
    const float* q = det + static_cast<size_t>(d) * 6;
    const float4 b = make_float4(q[0], q[1], q[2], q[3]);
    float best = 0.0f;
    int bl = -1;
    for (int l = 0; l < m; ++l) {
      const float v = iou_ld(s_box[l], b, p.eps);
      if (v > p.iou && (bl < 0 || v > best)) {
        best = v;
        bl = l;
      }
    }
    *best_iou = best;
    return bl;
  };
  auto kept = [&](int d) { return det[static_cast<size_t>(d) * 6 + 4] > p.conf; };
  // pass 1: every label learns its highest-IoU detection among those whose best label it is (ties: lower detection index)
  for (int d = tid; d < n; d += blockDim.x) {
    if (!kept(d)) continue;
    float v;
    const int bl = best_label(d, &v);
    if (bl < 0) continue;
    atomicMax(&s_key[bl], (static_cast<u64>(__float_as_uint(v)) << 32) | (0xffffffffu - static_cast<unsigned>(d)));
    s_any = 1;
  }
  __syncthreads();
  for (int l = tid; l < m; l += blockDim.x) {
    const int gc = s_cls[l];
    const u64 key = s_key[l];
    int row = p.nc;  // unmatched label: background false negative
    if (key) {
      const int d = static_cast<int>(0xffffffffu - static_cast<unsigned>(key & 0xffffffffu));
      row = trunc_class(det[static_cast<size_t>(d) * 6 + 5], p.nc);
    }
    if (gc >= 0 && row >= 0)
      atomicAdd(&p.matrix[static_cast<size_t>(row) * stride + gc], 1ull);
    else
      atomicAdd(&p.status[0], 1);
  }
  // pass 2: unmatched kept detections are background false positives — only when the image has a match at all (the
  // reference's `if n:` at utils/metrics.py:175)
  if (!s_any) return;
  for (int d = tid; d < n; d += blockDim.x) {
    if (!kept(d)) continue;
    float v;
    const int bl = best_label(d, &v);
    if (bl >= 0 && static_cast<unsigned>(s_key[bl] & 0xffffffffu) == 0xffffffffu - static_cast<unsigned>(d)) continue;
    const int dc = trunc_class(det[static_cast<size_t>(d) * 6 + 5], p.nc);
    if (dc >= 0)
      atomicAdd(&p.matrix[static_cast<size_t>(dc) * stride + p.nc], 1ull);
    else
      atomicAdd(&p.status[0], 1);
  }
}

}  // namespace
}  // namespace y3

extern "C" int64_t y3_ap_per_class_workspace_bytes(int64_t n, int64_t n_targets, int32_t niou, int32_t nc) {
  if (n < 0 || n_targets < 0 || niou <= 0 || nc <= 0) return -1;
  return static_cast<int64_t>(y3::ap_layout(n, n_targets, niou, nc).total);
}

extern "C" int y3_ap_per_class(const float* conf, int64_t conf_stride, const float* cls, int64_t cls_stride, const uint8_t* tp,
                               int32_t niou, int64_t n, const int32_t* det_count, int64_t rows_per_image,
                               const float* target_cls, int64_t target_stride, int64_t n_targets, int32_t nc, double eps,
                               void* workspace, int64_t workspace_bytes, double* ap, double* p, double* r, double* f1,
                               double* tp_out, double* fp_out, int64_t* nt, uint8_t* present, int32_t* f1_index,
                               int32_t* status, y3_stream_t stream) {
  using namespace y3;
  Y3_REQUIRE(n >= 0 && n <= 0x7fffffffLL - kRadixTile && n_targets >= 0 && n_targets <= 0x7fffffffLL, "ap_per_class: bad size");
  Y3_REQUIRE(niou > 0 && niou <= 64 && nc > 0 && nc <= 65535, "ap_per_class: niou must be in [1, 64], nc in [1, 65535]");
  Y3_REQUIRE(!det_count || rows_per_image > 0, "ap_per_class: rows_per_image must be > 0 with det_count");
  Y3_REQUIRE(ap && p && r && f1 && tp_out && fp_out && nt && present && f1_index && status && workspace, "ap_per_class: null pointer");
  Y3_REQUIRE(n == 0 || (conf && cls && tp), "ap_per_class: null row pointer");
  Y3_REQUIRE(n_targets == 0 || target_cls, "ap_per_class: null target pointer");
  const ApLayout L = ap_layout(n, n_targets, niou, nc);
  Y3_REQUIRE(workspace_bytes >= static_cast<int64_t>(L.total), "ap_per_class: workspace of %lld bytes, %lld needed",
             static_cast<long long>(workspace_bytes), static_cast<long long>(L.total));
  char* ws = static_cast<char*>(workspace);
  ApArgs a;
  a.conf = conf;
  a.conf_stride = conf_stride;
  a.cls = cls;
  a.cls_stride = cls_stride;
  a.tp = tp;
  a.niou = niou;
  a.n = static_cast<int>(n);
  a.det_count = det_count;
  a.rows_per_image = rows_per_image;
  a.tcls = target_cls;
  a.tcls_stride = target_stride;
  a.nt = static_cast<int>(n_targets);
  a.nc = nc;
  a.eps = eps;
  a.key[0] = reinterpret_cast<u64*>(ws + L.key0);
  a.key[1] = reinterpret_cast<u64*>(ws + L.key1);
  a.val[0] = reinterpret_cast<int*>(ws + L.val0);
  a.val[1] = reinterpret_cast<int*>(ws + L.val1);
  a.hist = reinterpret_cast<int*>(ws + L.hist);
  a.nblocks = static_cast<int>((n + kRadixTile - 1) / kRadixTile);
  a.seg = reinterpret_cast<int*>(ws + L.seg);
  a.ntc = reinterpret_cast<int*>(ws + L.ntc);
  a.ntoff = reinterpret_cast<int*>(ws + L.ntoff);
  a.tp_cnt = reinterpret_cast<int*>(ws + L.tp_cnt);
  a.tp_pos = reinterpret_cast<int*>(ws + L.tp_pos);
  a.smax = reinterpret_cast<double*>(ws + L.smax);
  a.pcurve = reinterpret_cast<double*>(ws + L.pcurve);
  a.rcurve = reinterpret_cast<double*>(ws + L.rcurve);
  a.ap = ap;
  a.p = p;
  a.r = r;
  a.f1 = f1;
  a.tp_out = tp_out;
  a.fp_out = fp_out;
  a.nt_out = nt;
  a.present = present;
  a.f1_index = f1_index;
  a.status = status;
  a.skey = a.key[0];
  a.sval = a.val[0];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid_cap = num_sms() * 8;
  Y3_CHECK_CUDA(launch_pdl(ap_init_kernel, dim3(1), dim3(256), 0, st, a));
  Y3_CHECK_CUDA(launch_pdl(ap_targets_kernel, dim3(std::max(1, std::min(grid_cap, (a.nt + 255) / 256))), dim3(256), 0, st, a));
  if (n > 0) {
    Y3_CHECK_CUDA(launch_pdl(ap_keys_kernel, dim3(std::min(grid_cap, (a.n + 255) / 256)), dim3(256), 0, st, a));
    // byte passes: 4 over the confidence bits, then over the class bits (classes 0..nc, nc = sentinel)
    int shifts[6], np_ = 0;
    for (int s = 0; s < 32; s += 8) shifts[np_++] = s;
    shifts[np_++] = 32;
    if (nc >= 256) shifts[np_++] = 40;
    for (int i = 0; i < np_; ++i) {
      const int src = i & 1;
      Y3_CHECK_CUDA(launch_pdl(radix_hist_kernel, dim3(a.nblocks), dim3(kRadixThreads), 0, st,
                               static_cast<const u64*>(a.key[src]), a.n, shifts[i], a.hist, a.nblocks));
      Y3_CHECK_CUDA(launch_pdl(scan_kernel, dim3(1), dim3(kScanThreads), 0, st, a.hist, 256 * a.nblocks));
      Y3_CHECK_CUDA(launch_pdl(radix_scatter_kernel, dim3(a.nblocks), dim3(kRadixThreads), 0, st,
                               static_cast<const u64*>(a.key[src]), static_cast<const int*>(a.val[src]), a.key[src ^ 1],
                               a.val[src ^ 1], a.n, shifts[i], static_cast<const int*>(a.hist), a.nblocks));
    }
    a.skey = a.key[np_ & 1];
    a.sval = a.val[np_ & 1];
  }
  Y3_CHECK_CUDA(launch_pdl(ap_segments_kernel, dim3(1), dim3(kScanThreads), 0, st, a));
  Y3_CHECK_CUDA(launch_pdl(ap_tp_positions_kernel, dim3(niou, nc), dim3(kPosThreads), 0, st, a));
  Y3_CHECK_CUDA(launch_pdl(ap_compute_kernel, dim3(niou + 1, nc), dim3(kApThreads), 0, st, a));
  Y3_CHECK_CUDA(launch_pdl(ap_finalize_kernel, dim3(1), dim3(kScanThreads), 0, st, a));
  return Y3_OK;
}

extern "C" int y3_confusion_update(const float* det, const int32_t* det_count, int32_t bs, int32_t max_det, int32_t det_stride,
                                   const float* labels, int32_t nl, int32_t nc, float conf_thres, float iou_thres, float eps,
                                   int64_t* matrix, int32_t* status, y3_stream_t stream) {
  Y3_REQUIRE(bs >= 0 && max_det >= 0 && nl >= 0 && nc > 0 && det_stride >= max_det, "confusion_update: bad shape");
  if (bs == 0) return Y3_OK;
  Y3_REQUIRE(matrix && status && (max_det == 0 || det) && (nl == 0 || labels), "confusion_update: null pointer");
  y3::ConfArgs a;
  a.det = det;
  a.det_count = det_count;
  a.max_det = max_det;
  a.det_stride = det_stride;
  a.labels = labels;
  a.nl = nl;
  a.nc = nc;
  a.conf = conf_thres;
  a.iou = iou_thres;
  a.eps = eps;
  a.matrix = reinterpret_cast<unsigned long long*>(matrix);
  a.status = status;
  Y3_CHECK_CUDA(y3::launch_pdl(y3::confusion_kernel, dim3(bs), dim3(256), 0, static_cast<cudaStream_t>(stream), a));
  return Y3_OK;
}
