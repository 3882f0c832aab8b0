// yolov3_b200 — validation matching on the device (SURVEY §8(f) row f2).  Replaces val.process_batch (reference val.py:147-188):
//   iou = box_iou(labels[:, 1:], detections[:, :4]);  for every IoU threshold t:
//     pairs (label l, detection d) with iou >= t and equal class, sorted by iou descending;
//     np.unique over the detection column keeps each detection's FIRST pair  = its best label  l*(d);
//     np.unique over the label column of what is left (now ordered by detection index) keeps each label's first pair
//                                                                            = the lowest-index detection whose best label it is;
//     correct[d, t] = True for the surviving pairs.
// i.e.  correct[d, t]  <=>  l*(d) exists  and  d == min{ d' : l*(d') == l*(d) }.  The reference does this with torch.where,
// a device->host copy, numpy argsort / unique per threshold and per image; here one launch handles a whole batch and all
// thresholds: grid (thresholds, images), one thread per detection, labels of the image staged in shared memory.
// IoU arithmetic is y3_box_iou's (separately rounded fp32, the reference's operand order), so `>= t` decides identically.
// Ties (two same-class labels with bit-equal IoU for one detection): the lower label index wins; numpy's argsort is
// unstable there, like the NMS tie rule (DESIGN.md section 2).
#include "y3_box.cuh"  // iou_ld (a = label box, b = detection box)
#include "y3_common.cuh"
#include "y3_internal.h"

namespace y3 {
namespace {

constexpr int kValMaxLabels = 1024;  // labels of one image staged in shared memory

struct ValArgs {
  const float* det;        // [bs, det_stride, 6] xyxy, conf, cls
  const int* det_count;    // [bs] or null (-> every image has max_det rows)
  int max_det, det_stride;
  const float* labels;     // [nl, 6] = (image, cls, x1, y1, x2, y2)
  int nl;
  const float* iouv;       // [niou]
  int niou;
  float eps;
  uint8_t* correct;        // [bs, max_det, niou]
  int* overflow;           // optional [bs]: labels of the image beyond kValMaxLabels (ignored by the matching)
};

__global__ void __launch_bounds__(256) val_match_kernel(const ValArgs p) {
  __shared__ float4 s_box[kValMaxLabels];
  __shared__ float s_cls[kValMaxLabels];
  __shared__ int s_win[kValMaxLabels];
  __shared__ int s_n;
  __shared__ int s_wcnt[8];
  const int ti = blockIdx.x, img = blockIdx.y;
  const float thr = p.iouv[ti];
  const int n = p.det_count ? min(p.det_count[img], p.max_det) : p.max_det;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  // stage this image's labels (order of appearance = label index inside the image, as labels[targets[:, 0] == si])
  // in index order: a block-wide ordered compaction, 256 labels per round
  for (int base = 0; base < p.nl; base += blockDim.x) {
    const int l = base + threadIdx.x;
    const bool mine = l < p.nl && static_cast<int>(p.labels[static_cast<size_t>(l) * 6]) == img;
    const unsigned bal = __ballot_sync(0xffffffffu, mine);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) s_wcnt[warp] = __popc(bal);
    __syncthreads();
    int off = s_n;
    for (int w = 0; w < warp; ++w) off += s_wcnt[w];
    const int at = off + __popc(bal & ((1u << lane) - 1u));
    if (mine && at < kValMaxLabels) {
      const float* q = p.labels + static_cast<size_t>(l) * 6;
      s_cls[at] = q[1];
      s_box[at] = make_float4(q[2], q[3], q[4], q[5]);
      s_win[at] = 0x7fffffff;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < 8; ++w) tot += s_wcnt[w];
      s_n += tot;
    }
    __syncthreads();
  }
  const int m = min(s_n, kValMaxLabels);
  if (p.overflow && ti == 0 && threadIdx.x == 0) p.overflow[img] = s_n > kValMaxLabels ? s_n - kValMaxLabels : 0;
  const float* det = p.det + static_cast<size_t>(img) * p.det_stride * 6;
  uint8_t* out = p.correct + (static_cast<size_t>(img) * p.max_det) * p.niou + ti;
  auto best_label = [&](int d) -> int {
    const float* q = det + static_cast<size_t>(d) * 6;
    const float4 b = make_float4(q[0], q[1], q[2], q[3]);
    const float cls = q[5];
    float best = -1.0f;
    int bl = -1;
    for (int l = 0; l < m; ++l) {
      if (s_cls[l] != cls) continue;
      const float v = iou_ld(s_box[l], b, p.eps);
      if (v >= thr && v > best) {  // strict >: the lower label index wins a tie
        best = v;
        bl = l;
      }
    }
    return bl;
  };
  // pass 1: every label learns the lowest-index detection whose best label it is
  for (int d = threadIdx.x; d < n; d += blockDim.x) {
    const int bl = best_label(d);
    if (bl >= 0) atomicMin(&s_win[bl], d);
  }
  __syncthreads();
  // pass 2 (the m IoUs per detection are recomputed: cheaper than parking a label index per detection somewhere)
  for (int d = threadIdx.x; d < n; d += blockDim.x) {
    const int bl = best_label(d);
    out[static_cast<size_t>(d) * p.niou] = (bl >= 0 && s_win[bl] == d) ? 1 : 0;
  }
  // rows beyond the image's detection count are defined (zero)
  for (int d = n + threadIdx.x; d < p.max_det; d += blockDim.x) out[static_cast<size_t>(d) * p.niou] = 0;
}

}  // namespace
}  // namespace y3

extern "C" int y3_val_match(const float* det, const int32_t* det_count, int32_t bs, int32_t max_det, int32_t det_stride,
                            const float* labels, int32_t nl, const float* iouv, int32_t niou, float eps, uint8_t* correct,
                            int32_t* overflow, y3_stream_t stream) {
  Y3_REQUIRE(bs >= 0 && max_det >= 0 && nl >= 0 && niou > 0 && niou <= 64 && det_stride >= max_det, "val_match: bad shape");
  if (bs == 0 || max_det == 0) return Y3_OK;
  Y3_REQUIRE(det && iouv && correct && (nl == 0 || labels), "val_match: null pointer");
  y3::ValArgs a;
  a.det = det;
  a.det_count = det_count;
  a.max_det = max_det;
  a.det_stride = det_stride;
  a.labels = labels;
  a.nl = nl;
  a.iouv = iouv;
  a.niou = niou;
  a.eps = eps;
  a.correct = correct;
  a.overflow = overflow;
  y3::val_match_kernel<<<dim3(niou, bs), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  Y3_CHECK_CUDA(cudaGetLastError());
  return Y3_OK;
}
