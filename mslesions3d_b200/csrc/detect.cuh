// Workspace layout of the fused detect_objects and its stages 2-4, shared by detect.cu and windows.cu.
#pragma once
#include "boxes.cuh"

namespace ssd3d {

struct DetectLayout {
  int S, nmax, words;
  long long off_count, off_nkeep, off_keptcnt, off_boxes, off_cand, off_cand2, cand2_stride, off_sboxes, off_sscores, off_sprior, off_mask,
      off_keptpos, off_keptscore, total;
};

// N images (or scans), P candidates per image, C classes (class 0 = background), top_k kept per image.  Segment
// seg = img * (C - 1) + (c - 1) owns count[seg] keys in cand[seg * P ...] and the boxes boxes[(img * P + p) * 6].
DetectLayout detect_layout(int N, long long P, int C, int top_k);

// Stages 2-4 (sort, truncation, NMS, merge, top-k, placeholder) on the candidate lists a stage-1 kernel wrote.
int detect_select(const DetectLayout& L, uint8_t* ws, int N, long long P, int n_classes, float max_overlap, int top_k,
                  float* out_boxes, float* out_scores, int64_t* out_labels, int64_t* out_prior, int32_t* out_count,
                  int32_t* status, cudaStream_t st);

}  // namespace ssd3d
