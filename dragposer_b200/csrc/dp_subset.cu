// dp_subset.cu -- row copies between a batch's per-clip arrays and compact arrays of a subset of its clips.  Per-clip settings on
// the fp32 frame kernel (dp_engine.cu) run each setting's clips as a batch of their own: gather their rows, run the kernel on the
// compact rows, scatter the results back.
#include <algorithm>

#include "dp_internal.h"

namespace {

// scatter == 0: row i of dst <- row ids[i] of src; scatter == 1: row ids[i] of dst <- row i of src.  blockIdx.y picks the copy.
__global__ void dp_copy_rows_kernel(const __grid_constant__ DpRowCopies C, const int32_t* __restrict__ ids, int n, int scatter) {
  const DpRowCopy& c = C.c[blockIdx.y];
  const int total = n * c.width;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < total; k += gridDim.x * blockDim.x) {
    const int i = k / c.width, j = k - i * c.width, r = ids[i];
    const size_t s = (size_t)(scatter ? i : r) * c.src_stride + j, d = (size_t)(scatter ? r : i) * c.dst_stride + j;
    c.dst[d] = c.src[s];
  }
}

}  // namespace

cudaError_t dp_copy_rows_launch(const DpRowCopies& copies, const int32_t* ids, int n, int scatter, cudaStream_t st) {
  if (copies.n == 0 || n == 0) return cudaSuccess;
  int width = 0;
  for (int i = 0; i < copies.n; ++i) width = width > copies.c[i].width ? width : copies.c[i].width;
  const long long total = (long long)n * width;
  const int blocks = (int)std::min<long long>((total + 255) / 256, 1024);
  dp_copy_rows_kernel<<<dim3(blocks, copies.n), 256, 0, st>>>(copies, ids, n, scatter);
  return cudaGetLastError();
}
