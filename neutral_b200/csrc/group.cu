// group.cu - kernels of the tally collective (see nb_group.cuh for the protocol).
#include "nb_group.cuh"

namespace nb {

namespace {

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ unsigned long long ld_relaxed_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Spins until *flag >= want. Bounded: after kWaitTimeoutNs the wait gives up and raises
// *fault (the results of this timestep are then wrong and the host says so). The loop polls
// with RELAXED loads and acquires once at the end: an acquire per poll invalidates the SM's L1
// every few hundred nanoseconds, under the history kernel that shares the SM.
__device__ __forceinline__ void wait_at_least(const unsigned long long* flag,
                                              unsigned long long want,
                                              unsigned long long* fault) {
  if (ld_relaxed_sys(flag) < want) {
    const unsigned long long t0 = global_timer_ns();
    while (ld_relaxed_sys(flag) < want) {
      __nanosleep(512);
      if (global_timer_ns() - t0 > kWaitTimeoutNs) {
        atomicExch(fault, 1ull);
        return;
      }
    }
  }
  (void)ld_acquire_sys(flag);
}

// The CTA that finishes last runs `then` (one election counter per kernel kind).
__device__ __forceinline__ bool last_cta(unsigned int* counter) {
  __shared__ bool last;
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  return last;
}

}  // namespace

// ------------------------------------------------------------------------------------
// Reduce-scatter fused with the fold: this rank's slice of every rank's delta, summed in rank
// order, added to the slice of the cumulative tally this rank owns. Peer deltas are read with
// ld.cv: the same addresses held other values three timesteps ago and nothing may serve them
// from a stale line. 32 registers and 128 threads per CTA on purpose: that is what is left on
// an SM whose register file holds six CTAs of the history kernel, so the collective of
// timestep t runs on the SMs while the transport of timestep t+1 owns them.
// ------------------------------------------------------------------------------------
// One warp waits for the flags; the kernels behind it in stream order then find their inputs
// ready without hundreds of CTAs polling (and without any of them sitting on an SM, spinning,
// beside the transport).
__global__ void k_wait_flags(const WaitList w, unsigned long long want) {
  if ((int)threadIdx.x < w.n) wait_at_least(w.flag[threadIdx.x], want, w.fault);
}

__global__ void __launch_bounds__(128, 16)
k_reduce_fold(const GroupView g, double* __restrict__ owned, unsigned long long epoch) {
  SyncBlock* mine = g.sync[g.rank];
  const size_t begin = (size_t)g.rank * g.chunk;
  const size_t end = begin + g.chunk < g.ncells ? begin + g.chunk : g.ncells;
  const size_t count = end > begin ? end - begin : 0;
  const size_t pairs = count >> 1;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  double2* own2 = reinterpret_cast<double2*>(owned);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += stride) {
    double2 s = make_double2(0.0, 0.0);
#pragma unroll 4
    for (int d = 0; d < g.nranks; ++d) {
      const double2 v = __ldcv(reinterpret_cast<const double2*>(g.src[d] + begin) + i);
      s.x += v.x;
      s.y += v.y;
    }
    double2 o = own2[i];
    o.x += s.x;
    o.y += s.y;
    own2[i] = o;
  }
  if ((count & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
    double s = 0.0;
    for (int d = 0; d < g.nranks; ++d) s += __ldcv(g.src[d] + begin + count - 1);
    owned[count - 1] += s;
  }
  if (epoch && last_cta(&mine->cta_done)) {
    if ((int)threadIdx.x < g.nranks)
      st_release_sys(&g.sync[threadIdx.x]->consumed[g.rank], epoch);
    if (threadIdx.x == 0) mine->cta_done = 0;
  }
}


// All-gather fused with the accumulation into the caller-visible tally: slice by slice,
// straight out of the owners' memory. The caller's tally need only be 8-byte aligned; the
// owned slices are 256-byte aligned and every slice starts at an even cell (chunk is even), so
// one test of `tally` picks the 16-byte or the scalar loop for the whole grid.
__global__ void __launch_bounds__(256)
k_gather_owned(const GroupView g, double* __restrict__ tally, unsigned long long epoch) {
  SyncBlock* mine = g.sync[g.rank];
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const bool vec = ((uintptr_t)tally & 15) == 0;
  for (int d = 0; d < g.nranks; ++d) {
    const size_t begin = (size_t)d * g.chunk;
    if (begin >= g.ncells) break;
    const size_t end = begin + g.chunk < g.ncells ? begin + g.chunk : g.ncells;
    const size_t count = end - begin;
    if (!vec) {
      for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        tally[begin + i] += __ldcv(g.src[d] + i);
      continue;
    }
    const size_t pairs = count >> 1;
    double2* t2 = reinterpret_cast<double2*>(tally + begin);
    const double2* s2 = reinterpret_cast<const double2*>(g.src[d]);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < pairs; i += stride) {
      const double2 v = __ldcv(s2 + i);
      double2 t = t2[i];
      t.x += v.x;
      t.y += v.y;
      t2[i] = t;
    }
    if ((count & 1) && blockIdx.x == 0 && threadIdx.x == 0)
      tally[begin + count - 1] += __ldcv(g.src[d] + count - 1);
  }
  if (epoch && last_cta(&mine->cta_done_flush)) {
    if ((int)threadIdx.x < g.nranks)
      st_release_sys(&g.sync[threadIdx.x]->flush_consumed[g.rank], epoch);
    if (threadIdx.x == 0) mine->cta_done_flush = 0;
  }
}

__global__ void k_signal(SyncBlock* mine, int flush, unsigned long long epoch) {
  __threadfence_system();
  st_release_sys(flush ? &mine->flush_ready : &mine->ready, epoch);
}

__global__ void __launch_bounds__(256)
k_fold_plain(double* __restrict__ dst, const double* __restrict__ src, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] += src[i];
}

int launch_reduce_fold(const GroupView& g, double* owned, unsigned long long epoch, int ctas,
                       cudaStream_t st) {
  k_reduce_fold<<<ctas > 0 ? ctas : 592, 128, 0, st>>>(g, owned, epoch);
  return 1;
}

int launch_wait_flags(const WaitList& w, unsigned long long want, cudaStream_t st) {
  k_wait_flags<<<1, 32, 0, st>>>(w, want);
  return 1;
}

int launch_gather_owned(const GroupView& g, double* tally, unsigned long long epoch,
                        cudaStream_t st) {
  k_gather_owned<<<296, 256, 0, st>>>(g, tally, epoch);
  return 1;
}

int launch_signal(SyncBlock* mine, int flush, unsigned long long epoch, cudaStream_t st) {
  k_signal<<<1, 1, 0, st>>>(mine, flush, epoch);
  return 1;
}

int launch_fold_plain(double* dst, const double* src, size_t n, cudaStream_t st) {
  if (n == 0) return 0;
  k_fold_plain<<<296, 256, 0, st>>>(dst, src, n);
  return 1;
}

}  // namespace nb
