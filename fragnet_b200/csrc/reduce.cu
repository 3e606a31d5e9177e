// Deterministic second stage of the parameter-gradient reductions that do not finish in their own launch (projection
// and tensor-core weight gradients, finetuning head): per-CTA partial records -> final tensors, in a fixed order.
#include "common.cuh"

namespace {

// One launch handles up to 4 output segments of the record:
//   out_s[(j / row_len_s) * out_stride_s + j % row_len_s] = sum_b partials[b * pstride + rec_off_s + j],  j < width_s
// Block = 8 record lanes x 32 columns: a warp reads one full 128-byte line per record (the first version, 32 record
// lanes x 8 columns, moved 32-byte sectors and ran at ~1 TB/s on the 148 x 64 KB weight-gradient partials); each
// thread sums every 8th record, then a fixed-order smem tree -> run-to-run deterministic.
constexpr int kRedCols = 32, kRedLanes = 8;
__global__ void __launch_bounds__(256) k_reduce_partials(const float *__restrict__ partials, int n_blocks, int pstride,
                                                         ReduceSegments segs) {
  __shared__ float sm[kRedLanes][kRedCols + 1];
  const int tx = threadIdx.x & (kRedCols - 1), ty = threadIdx.x / kRedCols;
  int col = blockIdx.x * kRedCols + tx;          // column in the concatenation of the (32-padded) segments
  int seg = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (seg == i && i + 1 < segs.n && col >= segs.padded_width[i]) {
      col -= segs.padded_width[i];
      seg = i + 1;
    }
  const bool valid = col < segs.width[seg] && (col % segs.row_len[seg]) < segs.valid_len[seg];
  float acc = 0.f;
  pdl_wait();
  if (valid) {
    const float *src = partials + segs.rec_off[seg] + col;
    int b = ty;
    for (; b + 3 * kRedLanes < n_blocks; b += 4 * kRedLanes) {   // four independent loads in flight
      const float v0 = src[(int64_t)b * pstride], v1 = src[(int64_t)(b + kRedLanes) * pstride],
                  v2 = src[(int64_t)(b + 2 * kRedLanes) * pstride], v3 = src[(int64_t)(b + 3 * kRedLanes) * pstride];
      acc += v0; acc += v1; acc += v2; acc += v3;
    }
    for (; b < n_blocks; b += kRedLanes) acc += src[(int64_t)b * pstride];
  }
  sm[ty][tx] = acc;
  __syncthreads();
  if (ty == 0 && valid) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kRedLanes; ++k) s += sm[k][tx];
    const int rl = segs.row_len[seg];
    segs.out[seg][(col / rl) * segs.out_stride[seg] + (col % rl)] = s;
  }
}

}  // namespace

int fnb_launch_reduce_segments(const float *partials, int n_blocks, int pstride, ReduceSegments segs,
                               cudaStream_t stream) {
  int cols = 0;
  for (int i = 0; i < segs.n; ++i) {
    segs.padded_width[i] = (segs.width[i] + kRedCols - 1) & ~(kRedCols - 1);
    if (segs.valid_len[i] <= 0 || segs.valid_len[i] > segs.row_len[i]) segs.valid_len[i] = segs.row_len[i];
    cols += segs.padded_width[i];
  }
  if (cols == 0) return 0;
  if (cudaError_t le = fnb_launch(k_reduce_partials, dim3(cols / kRedCols), dim3(256), 0, stream, partials, n_blocks, pstride, segs))
    return (int)le;
  FNB_CHECK_LAUNCH();
  return 0;
}

extern "C" size_t fnb_scratch_bytes(void) { return (size_t)kScratchFloats * sizeof(float); }
