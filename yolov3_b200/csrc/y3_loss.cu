// yolov3_b200 — ComputeLoss forward + backward in four launches, no host synchronisation.
// Replaces ComputeLoss.__call__ and build_targets (reference utils/loss.py:131-244) with ultralytics bbox_iou(CIoU)
// and BCEWithLogitsLoss(pos_weight) inlined, and the autograd graph behind them: the kernels emit dL/dp directly.
//   K1 match    : build_targets — one thread per (level, offset, anchor, target); anchor-ratio test, 5-cell neighbour
//                 expansion, truncation + clamp of grid indices; appends match records (loss.py:183-244)
//   K2 matches  : one warp per match — gather logits, decode box, CIoU (+ analytic gradient by forward-mode duals),
//                 class BCE (+ gradient), IoU -> tobj with last-write-wins in REFERENCE order (loss.py:144-167)
//   K3 obj      : dense objectness BCE over every cell + its gradient (loss.py:169-170)
//   K4 finalize : means, balance, hyp gains, x batch size (loss.py:176-181)
// grads must be zeroed by the caller's stream before K2 (done in y3_loss_fwd_bwd with one memset per level).
// Compiled without fast-math / FMA contraction (see build.py EXACT_SOURCES).
#include <math_constants.h>

#include "y3_common.cuh"
#include "y3_internal.h"

namespace y3 {
namespace {

struct Match {
  unsigned int q;  // position in the reference's enumeration order (offset-major, anchor, target)
  int b, a, gj, gi, cls;
  float tx, ty, tw, th;  // tbox
  float aw, ah;          // anchor (grid units)
};

struct LossArgs {
  y3_loss_desc d;
  Match* matches[Y3_MAX_LEVELS];
  int cap;                            // per-level match capacity = 5*na*nt
  int* count;                         // [nl]
  unsigned long long* tobj_key[Y3_MAX_LEVELS];  // per cell: (q+1) << 32 | float bits of the clamped IoU
  double* acc;                        // [nl][3]: sum(1-iou), sum(cls bce), sum(obj bce)
  float* out;                         // [4]: loss*bs, lbox, lobj, lcls
};

// ---------------------------------------------------------------------------------------------- K1
__global__ void __launch_bounds__(256) loss_match_kernel(const LossArgs p) {
  pdl_entry();
  const y3_loss_desc& d = p.d;
  const int per_level = 5 * d.na * d.nt;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per_level * d.nl) return;
  const int l = i / per_level;
  const int q = i - l * per_level;
  const int oi = q / (d.na * d.nt);
  const int a = (q / d.nt) % d.na;
  const int t = q % d.nt;
  const float* tg = d.targets + static_cast<size_t>(t) * 6;
  const float nx = static_cast<float>(d.nx[l]), ny = static_cast<float>(d.ny[l]);
  const float gx = tg[2] * nx, gy = tg[3] * ny, gw = tg[4] * nx, gh = tg[5] * ny;
  const float aw = d.anchors[l][a][0], ah = d.anchors[l][a][1];
  const float rw = gw / aw, rh = gh / ah;
  const float m = fmaxf(fmaxf(rw, 1.0f / rw), fmaxf(rh, 1.0f / rh));
  if (!(m < d.anchor_t)) return;
  const float g = 0.5f;
  const float ix = nx - gx, iy = ny - gy;
  bool sel;
  float ox = 0.f, oy = 0.f;
  switch (oi) {
    case 0: sel = true; break;
    case 1: sel = (fmodf(gx, 1.0f) < g) && (gx > 1.0f); ox = g; break;
    case 2: sel = (fmodf(gy, 1.0f) < g) && (gy > 1.0f); oy = g; break;
    case 3: sel = (fmodf(ix, 1.0f) < g) && (ix > 1.0f); ox = -g; break;
    default: sel = (fmodf(iy, 1.0f) < g) && (iy > 1.0f); oy = -g; break;
  }
  if (!sel) return;
  const int gi0 = static_cast<int>(truncf(gx - ox)), gj0 = static_cast<int>(truncf(gy - oy));
  Match mt;
  mt.q = static_cast<unsigned int>(q);
  mt.b = static_cast<int>(tg[0]);
  mt.cls = static_cast<int>(tg[1]);
  mt.a = a;
  mt.gi = min(max(gi0, 0), d.nx[l] - 1);
  mt.gj = min(max(gj0, 0), d.ny[l] - 1);
  mt.tx = gx - static_cast<float>(mt.gi);  // tbox uses the CLAMPED indices: the reference clamps gij in place through
  mt.ty = gy - static_cast<float>(mt.gj);  // its gi/gj views one statement before it forms gxy - gij (loss.py:236-240)
  mt.tw = gw;
  mt.th = gh;
  mt.aw = aw;
  mt.ah = ah;
  if (mt.b < 0 || mt.b >= d.bs || mt.cls < 0 || mt.cls >= d.nc) return;  // malformed label row: ignore
  const int slot = atomicAdd(&p.count[l], 1);
  p.matches[l][slot] = mt;
}

// ---------------------------------------------------------------------------------------------- forward-mode duals
struct Dual {
  float v, g[4];
};
__device__ __forceinline__ Dual dconst(float v) { return Dual{v, {0.f, 0.f, 0.f, 0.f}}; }
__device__ __forceinline__ Dual dvar(float v, int k) {
  Dual r = dconst(v);
  r.g[k] = 1.f;
  return r;
}
#define Y3_D4(expr)                 \
  for (int k = 0; k < 4; ++k) {     \
    expr;                           \
  }
__device__ __forceinline__ Dual operator+(Dual a, Dual b) { Dual r; r.v = a.v + b.v; Y3_D4(r.g[k] = a.g[k] + b.g[k]) return r; }
__device__ __forceinline__ Dual operator-(Dual a, Dual b) { Dual r; r.v = a.v - b.v; Y3_D4(r.g[k] = a.g[k] - b.g[k]) return r; }
__device__ __forceinline__ Dual operator*(Dual a, Dual b) { Dual r; r.v = a.v * b.v; Y3_D4(r.g[k] = a.g[k] * b.v + a.v * b.g[k]) return r; }
__device__ __forceinline__ Dual operator/(Dual a, Dual b) {
  Dual r;
  r.v = a.v / b.v;
  Y3_D4(r.g[k] = (a.g[k] - r.v * b.g[k]) / b.v) return r;
}
__device__ __forceinline__ Dual dscale(Dual a, float s) { Dual r; r.v = a.v * s; Y3_D4(r.g[k] = a.g[k] * s) return r; }
__device__ __forceinline__ Dual dadd(Dual a, float s) { a.v += s; return a; }
// torch.minimum / maximum backward: the selected operand gets the gradient, ties split it evenly
__device__ __forceinline__ Dual dmin(Dual a, Dual b) {
  if (a.v < b.v) return a;
  if (b.v < a.v) return b;
  Dual r; r.v = a.v; Y3_D4(r.g[k] = 0.5f * (a.g[k] + b.g[k])) return r;
}
__device__ __forceinline__ Dual dmax(Dual a, Dual b) {
  if (a.v > b.v) return a;
  if (b.v > a.v) return b;
  Dual r; r.v = a.v; Y3_D4(r.g[k] = 0.5f * (a.g[k] + b.g[k])) return r;
}
__device__ __forceinline__ Dual dclamp0(Dual a) {  // clamp(min=0): gradient passes where a >= 0
  if (a.v >= 0.f) return a;
  return dconst(0.f);
}
__device__ __forceinline__ Dual datan(Dual a) {
  Dual r;
  r.v = atanf(a.v);
  const float s = 1.0f / (1.0f + a.v * a.v);
  Y3_D4(r.g[k] = a.g[k] * s) return r;
}

// bbox_iou(box1, box2, xywh=True, CIoU=True, eps=1e-7) with gradient w.r.t. box1 (alpha is a constant: no_grad)
__device__ __forceinline__ Dual ciou_dual(Dual x1, Dual y1, Dual w1, Dual h1, float x2, float y2, float w2, float h2) {
  const float eps = 1e-7f;
  const Dual hw1 = dscale(w1, 0.5f), hh1 = dscale(h1, 0.5f);
  const Dual b1x1 = x1 - hw1, b1x2 = x1 + hw1, b1y1 = y1 - hh1, b1y2 = y1 + hh1;
  const float hw2 = w2 / 2, hh2 = h2 / 2;
  const Dual b2x1 = dconst(x2 - hw2), b2x2 = dconst(x2 + hw2), b2y1 = dconst(y2 - hh2), b2y2 = dconst(y2 + hh2);
  const Dual inter = dclamp0(dmin(b1x2, b2x2) - dmax(b1x1, b2x1)) * dclamp0(dmin(b1y2, b2y2) - dmax(b1y1, b2y1));
  const Dual uni = dadd(w1 * h1 + dconst(w2 * h2) - inter, eps);
  const Dual iou = inter / uni;
  const Dual cw = dmax(b1x2, b2x2) - dmin(b1x1, b2x1);
  const Dual ch = dmax(b1y2, b2y2) - dmin(b1y1, b2y1);
  const Dual c2 = dadd(cw * cw + ch * ch, eps);
  const Dual sx = b2x1 + b2x2 - b1x1 - b1x2, sy = b2y1 + b2y2 - b1y1 - b1y2;
  const Dual rho2 = dscale(sx * sx + sy * sy, 0.25f);
  const Dual dat = dconst(atanf(w2 / h2)) - datan(w1 / h1);
  const Dual v = dscale(dat * dat, 4.0f / (CUDART_PI_F * CUDART_PI_F));
  const float alpha = v.v / (v.v - iou.v + (1.0f + eps));
  return iou - (rho2 / c2 + dscale(v, alpha));
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
// BCEWithLogits(x, t, pos_weight=pw) and d/dx
__device__ __forceinline__ float bce_logits(float x, float t, float pw, float* dx) {
  const float lw = 1.0f + (pw - 1.0f) * t;
  const float sp = fmaxf(-x, 0.0f) + log1pf(expf(-fabsf(x)));  // softplus(-x)
  *dx = (1.0f - t) - lw * (1.0f - sigmoidf_(x));
  return (1.0f - t) * x + lw * sp;
}

// ---------------------------------------------------------------------------------------------- K2
__global__ void __launch_bounds__(256) loss_matches_kernel(const LossArgs p, int l) {
  pdl_entry();
  const y3_loss_desc& d = p.d;
  const int n = p.count[l];
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n) return;
  const Match m = p.matches[l][warp];
  const int no = d.nc + 5;
  const size_t cell = ((static_cast<size_t>(m.b) * d.na + m.a) * d.ny[l] + m.gj) * d.nx[l] + m.gi;
  const float* ps = d.p[l] + cell * no;
  float* gs = d.grad[l] ? d.grad[l] + cell * no : nullptr;
  const float inv_n = 1.0f / static_cast<float>(n);
  // ---- box regression (lane 0)
  if (lane == 0) {
    const float s0 = sigmoidf_(ps[0]), s1 = sigmoidf_(ps[1]), s2 = sigmoidf_(ps[2]), s3 = sigmoidf_(ps[3]);
    const float px = s0 * 2.0f - 0.5f, py = s1 * 2.0f - 0.5f;
    const float t2 = s2 * 2.0f, t3 = s3 * 2.0f;
    const float pw = t2 * t2 * m.aw, ph = t3 * t3 * m.ah;
    const Dual c = ciou_dual(dvar(px, 0), dvar(py, 1), dvar(pw, 2), dvar(ph, 3), m.tx, m.ty, m.tw, m.th);
    atomicAdd(&p.acc[l * 3 + 0], static_cast<double>(1.0f - c.v));
    const float iou_c = fmaxf(c.v, 0.0f);  // iou.detach().clamp(0)
    atomicMax(&p.tobj_key[l][cell], (static_cast<unsigned long long>(m.q + 1u) << 32) | __float_as_uint(iou_c));
    if (gs) {
      const float k = -d.box * static_cast<float>(d.bs) * inv_n * d.grad_scale;  // d(loss)/d(ciou)
      atomicAdd(gs + 0, k * c.g[0] * 2.0f * s0 * (1.0f - s0));
      atomicAdd(gs + 1, k * c.g[1] * 2.0f * s1 * (1.0f - s1));
      atomicAdd(gs + 2, k * c.g[2] * 8.0f * s2 * s2 * (1.0f - s2) * m.aw);
      atomicAdd(gs + 3, k * c.g[3] * 8.0f * s3 * s3 * (1.0f - s3) * m.ah);
    }
  }
  // ---- classification (all lanes), only if nc > 1 (loss.py:164)
  if (d.nc > 1) {
    float sum = 0.f;
    const float k = d.cls * static_cast<float>(d.bs) * inv_n / static_cast<float>(d.nc) * d.grad_scale;
    for (int c = lane; c < d.nc; c += 32) {
      float dx;
      sum += bce_logits(ps[5 + c], c == m.cls ? d.cp : d.cn, d.cls_pw, &dx);
      if (gs) atomicAdd(gs + 5 + c, k * dx);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) atomicAdd(&p.acc[l * 3 + 1], static_cast<double>(sum));
  }
}

// ---------------------------------------------------------------------------------------------- K3
__global__ void __launch_bounds__(256) loss_obj_kernel(const LossArgs p, int l) {
  pdl_entry();
  const y3_loss_desc& d = p.d;
  const int no = d.nc + 5;
  const size_t cells = static_cast<size_t>(d.bs) * d.na * d.ny[l] * d.nx[l];
  const float k = d.obj * static_cast<float>(d.bs) * d.balance[l] / static_cast<float>(cells) * d.grad_scale;
  float sum = 0.f;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < cells;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const unsigned long long key = p.tobj_key[l][i];
    const float t = key ? __uint_as_float(static_cast<unsigned int>(key & 0xFFFFFFFFull)) : 0.0f;
    float dx;
    sum += bce_logits(d.p[l][i * no + 4], t, d.obj_pw, &dx);
    if (d.grad[l]) d.grad[l][i * no + 4] = k * dx;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __shared__ float s[8];
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) tot += s[w];
    atomicAdd(&p.acc[l * 3 + 2], tot);
  }
}

// ---------------------------------------------------------------------------------------------- K4
__global__ void loss_finalize_kernel(const LossArgs p) {
  pdl_entry();
  const y3_loss_desc& d = p.d;
  float lbox = 0.f, lobj = 0.f, lcls = 0.f;
  for (int l = 0; l < d.nl; ++l) {
    const int n = p.count[l];
    const double cells = static_cast<double>(d.bs) * d.na * d.ny[l] * d.nx[l];
    if (n > 0) {
      lbox += static_cast<float>(p.acc[l * 3 + 0] / n);
      if (d.nc > 1) lcls += static_cast<float>(p.acc[l * 3 + 1] / (static_cast<double>(n) * d.nc));
    }
    lobj += static_cast<float>(p.acc[l * 3 + 2] / cells) * d.balance[l];
  }
  lbox *= d.box;
  lobj *= d.obj;
  lcls *= d.cls;
  p.out[0] = (lbox + lobj + lcls) * static_cast<float>(d.bs);
  p.out[1] = lbox;
  p.out[2] = lobj;
  p.out[3] = lcls;
}

size_t al(size_t v) { return (v + 255) / 256 * 256; }

}  // namespace
}  // namespace y3

extern "C" int64_t y3_loss_workspace_bytes(const y3_loss_desc* d) {
  if (!d || d->nl < 1 || d->nl > Y3_MAX_LEVELS) return -1;
  size_t b = y3::al(sizeof(int) * Y3_MAX_LEVELS) + y3::al(sizeof(double) * 3 * Y3_MAX_LEVELS);
  const size_t cap = static_cast<size_t>(5) * d->na * (d->nt > 0 ? d->nt : 1);
  for (int l = 0; l < d->nl; ++l) {
    b += y3::al(sizeof(y3::Match) * cap);
    b += y3::al(sizeof(unsigned long long) * static_cast<size_t>(d->bs) * d->na * d->ny[l] * d->nx[l]);
  }
  return static_cast<int64_t>(b);
}

extern "C" int y3_loss_fwd_bwd(const y3_loss_desc* d, void* workspace, int64_t workspace_bytes, float* out,
                               y3_stream_t stream_) {
  using namespace y3;
  Y3_REQUIRE(d && workspace && out, "loss: null pointer");
  Y3_REQUIRE(d->nl >= 1 && d->nl <= Y3_MAX_LEVELS && d->na >= 1 && d->na <= Y3_MAX_ANCHORS && d->bs > 0 && d->nc >= 1,
             "loss: bad shape");
  Y3_REQUIRE(d->nt >= 0 && (d->nt == 0 || d->targets), "loss: bad targets");
  Y3_REQUIRE(workspace_bytes >= y3_loss_workspace_bytes(d), "loss: workspace too small");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  LossArgs a{};
  a.d = *d;
  a.out = out;
  uint8_t* w = static_cast<uint8_t*>(workspace);
  uint8_t* w0 = w;
  a.count = reinterpret_cast<int*>(w);
  w += al(sizeof(int) * Y3_MAX_LEVELS);
  a.acc = reinterpret_cast<double*>(w);
  w += al(sizeof(double) * 3 * Y3_MAX_LEVELS);
  const size_t head_bytes = static_cast<size_t>(w - w0);
  a.cap = 5 * d->na * (d->nt > 0 ? d->nt : 1);
  for (int l = 0; l < d->nl; ++l) {
    Y3_REQUIRE(d->p[l] && d->ny[l] > 0 && d->nx[l] > 0, "loss: bad level %d", l);
    a.matches[l] = reinterpret_cast<Match*>(w);
    w += al(sizeof(Match) * a.cap);
  }
  Y3_CHECK_CUDA(cudaMemsetAsync(w0, 0, head_bytes, stream));
  const int no = d->nc + 5;
  for (int l = 0; l < d->nl; ++l) {
    const size_t cells = static_cast<size_t>(d->bs) * d->na * d->ny[l] * d->nx[l];
    a.tobj_key[l] = reinterpret_cast<unsigned long long*>(w);
    w += al(sizeof(unsigned long long) * cells);
    Y3_CHECK_CUDA(cudaMemsetAsync(a.tobj_key[l], 0, sizeof(unsigned long long) * cells, stream));
    if (d->grad[l]) Y3_CHECK_CUDA(cudaMemsetAsync(d->grad[l], 0, sizeof(float) * cells * no, stream));
  }
  if (d->nt > 0) {
    const int total = 5 * d->na * d->nt * d->nl;
    Y3_CHECK_CUDA(::y3::launch_pdl(loss_match_kernel, dim3((total + 255) / 256), dim3(256), 0, stream, a));
    for (int l = 0; l < d->nl; ++l) {
      const long long threads = static_cast<long long>(a.cap) * 32;  // one warp per potential match
      Y3_CHECK_CUDA(::y3::launch_pdl(loss_matches_kernel, dim3(static_cast<unsigned>((threads + 255) / 256)), dim3(256), 0, stream, a, l));
    }
  }
  for (int l = 0; l < d->nl; ++l) {
    const size_t cells = static_cast<size_t>(d->bs) * d->na * d->ny[l] * d->nx[l];
    size_t blocks = (cells + 255) / 256;
    const size_t cap = static_cast<size_t>(num_sms()) * 8;
    if (blocks > cap) blocks = cap;
    Y3_CHECK_CUDA(::y3::launch_pdl(loss_obj_kernel, dim3(static_cast<unsigned>(blocks)), dim3(256), 0, stream, a, l));
  }
  Y3_CHECK_CUDA(::y3::launch_pdl(loss_finalize_kernel, dim3(1), dim3(1), 0, stream, a));
  Y3_CHECK_CUDA(cudaGetLastError());
  return Y3_OK;
}
