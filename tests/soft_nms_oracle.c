/*
 * soft_nms_oracle.c -- TEST INFRASTRUCTURE ONLY.  The CPU checker of the 3D soft-NMS kernel
 * (3d-multi-resolution-rcnn_b200/csrc/soft_nms3d.cu); the product never links or calls it.
 * tests/soft_nms_oracle.py compiles it with gcc -O2 -ffp-contract=off (no contraction gcc would add
 * of its own) into a temporary directory and binds it with ctypes.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define API __attribute__((visibility("default")))

/* ------------------------------------------------------------------------------------------ */
/* 3D soft-NMS: soft_nms_cpu, mmdet/ops/nms/src/soft_nms_cpu.pyx (mmdet v0.6.0), written with a  */
/* depth axis and the score in column 6, in the reference's own sequential form: argmax by       */
/* `maxscore < s` from position i, swap into i, decay the later rows, and copy the last row over */
/* each row that falls below min_score (N -= 1, redo that position).  Every variable is a C      */
/* float and every operation one fp32 operation in the source's order (-ffp-contract=off); the   */
/* gaussian weight is the reference's np.exp on a Python float: double exp, rounded to float.    */
/* method 1 = linear, 2 = gaussian.  dets [n,7]; out_dets [n,7] (selection order, scores as      */
/* selected) and inds [n]; returns the number of rows left.                                      */
/* ------------------------------------------------------------------------------------------ */
static inline float sn_max(float a, float b) { return a >= b ? a : b; }
static inline float sn_min(float a, float b) { return a <= b ? a : b; }

API int64_t oracle_soft_nms3d(const float *dets, int64_t n, float iou_thr, int method, float sigma, float min_score,
                              float *out_dets, int64_t *inds) {
  float *boxes = out_dets;
  int64_t N = n;
  if (n <= 0) return 0;
  memcpy(boxes, dets, sizeof(float) * 7 * (size_t)n);
  for (int64_t i = 0; i < n; i++) inds[i] = i;
  for (int64_t i = 0; i < n; i++) { /* range(N): the bound is read once */
    float maxscore = boxes[i * 7 + 6];
    int64_t maxpos = i;
    float tb[7];
    for (int c = 0; c < 7; c++) tb[c] = boxes[i * 7 + c];
    int64_t ti = inds[i];
    for (int64_t pos = i + 1; pos < N; pos++) {
      if (maxscore < boxes[pos * 7 + 6]) {
        maxscore = boxes[pos * 7 + 6];
        maxpos = pos;
      }
    }
    for (int c = 0; c < 7; c++) boxes[i * 7 + c] = boxes[maxpos * 7 + c];
    inds[i] = inds[maxpos];
    for (int c = 0; c < 7; c++) boxes[maxpos * 7 + c] = tb[c];
    inds[maxpos] = ti;
    const float tx1 = boxes[i * 7 + 0], ty1 = boxes[i * 7 + 1], tx2 = boxes[i * 7 + 2], ty2 = boxes[i * 7 + 3];
    const float tz1 = boxes[i * 7 + 4], tz2 = boxes[i * 7 + 5];
    int64_t pos = i + 1;
    while (pos < N) {
      float *b = boxes + pos * 7;
      const float x1 = b[0], y1 = b[1], x2 = b[2], y2 = b[3], z1 = b[4], z2 = b[5];
      const float area = ((x2 - x1 + 1) * (y2 - y1 + 1)) * (z2 - z1 + 1);
      const float iw = sn_min(tx2, x2) - sn_max(tx1, x1) + 1;
      if (iw > 0) {
        const float ih = sn_min(ty2, y2) - sn_max(ty1, y1) + 1;
        if (ih > 0) {
          const float id = sn_min(tz2, z2) - sn_max(tz1, z1) + 1;
          if (id > 0) {
            const float tarea = ((tx2 - tx1 + 1) * (ty2 - ty1 + 1)) * (tz2 - tz1 + 1);
            const float inter = (iw * ih) * id;
            const float ua = (tarea + area) - inter;
            const float ov = inter / ua;
            float weight;
            if (method == 1)
              weight = ov > iou_thr ? 1 - ov : 1;
            else
              weight = (float)exp((double)(-(ov * ov) / sigma));
            b[6] = weight * b[6];
            if (b[6] < min_score) {
              for (int c = 0; c < 7; c++) b[c] = boxes[(N - 1) * 7 + c];
              inds[pos] = inds[N - 1];
              N -= 1;
              pos -= 1;
            }
          }
        }
      }
      pos += 1;
    }
  }
  return N;
}
