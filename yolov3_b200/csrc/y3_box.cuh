// yolov3_b200 — box arithmetic shared by the validation kernels (y3_val.cu, y3_metrics.cu).
#pragma once
#include <cuda_runtime.h>

namespace y3 {

// IoU of a label box `a` and a detection box `b` (x1, y1, x2, y2): inter / (a1 + a2 - inter + eps), the operand order of the
// reference's box_iou(labels, detections) (utils/metrics.py:10), every operation separately rounded fp32 (no contraction).
__device__ __forceinline__ float iou_ld(const float4& a, const float4& b, float eps) {
  const float w = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.0f);
  const float h = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.0f);
  const float inter = __fmul_rn(w, h);
  const float a1 = __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y));
  const float a2 = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(a1, a2), inter), eps));
}

}  // namespace y3
