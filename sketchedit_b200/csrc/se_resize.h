// Pillow-exact BICUBIC resize of ragged uint8 HWC batches (se_resize.cu).
#pragma once
#include <vector>

#include "se_common.cuh"

namespace se {

// Host tables of one in -> out pass (Pillow's precompute_coeffs + normalize_coeffs_8bpc): bounds [out][2] = (first source
// index, tap count), weights [out][ksize] in 22-bit fixed point (zero past the tap count). Returns ksize.
int resize_coeffs(int in, int out, std::vector<int>& bounds, std::vector<int>& weights);

// The same tables on the current device, built and uploaded (on `s`) the first time a pair is seen there and kept for the
// life of the process. Callers must order their uses after that upload (every se_resize_u8 call shares one stream order).
struct ResizeTable { const int* bounds; const int* weights; int ksize; };
int resize_table(int in, int out, cudaStream_t s, ResizeTable* t);

// One image of one pass. Horizontal pass: resample rows (table != null) or copy (table null, same size); vertical pass:
// resample columns. `in` is an [.., in_w, C] plane, `out` an [out_h, out_w, C] plane; `reverse` writes the channels reversed.
struct ResizeJob {
  const unsigned char* in;
  unsigned char* out;
  const int* bounds;
  const int* weights;
  int ksize, in_w, out_h, out_w, reverse;
};

// One launch over `njobs` jobs (device array); max_pix = the largest out_h * out_w among them.
int resize_pass(const ResizeJob* jobs, int njobs, long long max_pix, int C, int vertical, cudaStream_t s);

}  // namespace se
