// tally_batches.cu - the batch partial tallies of option tally_batches (sm_100a).
//
// A batched bank's history kernel deposits into B partial tallies S_b, one per contiguous range
// of global particle indices (batch_of, nb_bank.cuh). Each S_b * N / n_b is an independent
// estimate of the whole tally, so the spread of the B estimates gives the statistical error of
// their mean, per cell and for the total. The kernels here are the sweeps over the slab that
// the host issues when somebody looks at the tally: the flush into the caller's tally, the
// export of the batches and the statistics. All are memory-bound and run outside a timestep.
#include "transport.cuh"

namespace nb {

namespace {

__device__ __forceinline__ int batch_count(int n, int b, int B) {
  return n / B + (b < n % B ? 1 : 0);  // shard_split (capi.cu)
}

}  // namespace

__global__ void __launch_bounds__(256)
k_batch_flush(double* __restrict__ slab, int B, size_t ncells, double* __restrict__ tally) {
  double* flushed = slab + (size_t)B * ncells;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncells; i += stride) {
    double s = 0.0;
    for (int b = 0; b < B; ++b) s += slab[batch_slot(b, i, B, ncells)];
    tally[i] += s - flushed[i];
    flushed[i] = s;
  }
}

__global__ void __launch_bounds__(256)
k_batch_export(const double* __restrict__ slab, int B, size_t ncells, double* __restrict__ out) {
  const size_t total = (size_t)B * ncells;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += stride) {
    const int b = (int)(j / ncells);
    out[j] = slab[batch_slot(b, j - (size_t)b * ncells, B, ncells)];
  }
}

// x_b = S_b * N / n_b, m = mean of x_b, s^2 = sum (x_b - m)^2 / (B - 1), R = sqrt(s^2 / B) / |m|
// (0 where m == 0), all in batch order.
__global__ void __launch_bounds__(256)
k_batch_relerr(const double* __restrict__ slab, int B, size_t ncells, int n,
               double* __restrict__ relerr) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncells; i += stride) {
    double sum = 0.0;
    for (int b = 0; b < B; ++b)
      sum += slab[batch_slot(b, i, B, ncells)] * (double)n / (double)batch_count(n, b, B);
    const double m = sum / (double)B;
    double ss = 0.0;
    for (int b = 0; b < B; ++b) {
      const double d = slab[batch_slot(b, i, B, ncells)] * (double)n / (double)batch_count(n, b, B) - m;
      ss += d * d;
    }
    const double var = ss / (double)(B - 1);
    relerr[i] = m == 0.0 ? 0.0 : sqrt(var / (double)B) / fabs(m);
  }
}

// One batch per blockIdx.y; a fixed grid, so that the host's sum of the partials is the same
// sum in the same order every time.
__global__ void __launch_bounds__(256)
k_batch_sums(const double* __restrict__ slab, int B, size_t ncells, double* __restrict__ partial) {
  const int b = blockIdx.y;
  double s = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < ncells;
       i += (size_t)gridDim.x * blockDim.x)
    s += slab[batch_slot(b, i, B, ncells)];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double warp_part[8];
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_part[w];
    partial[(size_t)b * gridDim.x + blockIdx.x] = t;
  }
}

int launch_batch_flush(double* slab, int B, size_t ncells, double* tally, cudaStream_t st) {
  k_batch_flush<<<592, 256, 0, st>>>(slab, B, ncells, tally);
  return 1;
}

int launch_batch_export(const double* slab, int B, size_t ncells, double* out, cudaStream_t st) {
  k_batch_export<<<592, 256, 0, st>>>(slab, B, ncells, out);
  return 1;
}

int launch_batch_relerr(const double* slab, int B, size_t ncells, int n, double* relerr,
                        cudaStream_t st) {
  k_batch_relerr<<<592, 256, 0, st>>>(slab, B, ncells, n, relerr);
  return 1;
}

int launch_batch_sums(const double* slab, int B, size_t ncells, double* partial, cudaStream_t st) {
  k_batch_sums<<<dim3(kBatchSumBlocks, B), 256, 0, st>>>(slab, B, ncells, partial);
  return 1;
}

}  // namespace nb
