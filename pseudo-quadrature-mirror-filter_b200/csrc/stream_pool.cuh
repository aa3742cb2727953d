// Stream pools: device-resident state of P independent streams, any n distinct of which one call steps (include/pqmf_b200.h).
//
// Pool layout (fp32): analysis state [2, P, L], synthesis state [2, P, M, K]; one int32 phase word per stream and direction: bit 0 = the
// half that holds the stream's current history, bit 1 = the parity of its next global frame index.  Row r of a call's block belongs to
// stream ids[r].  The POOL instantiations of the streaming kernels (direct_form.cuh, hankel4_stream.cuh) take their params derived from
// the lockstep ones with this index appended, so the lockstep instantiations keep their parameter layout.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace pqmf {

struct StreamPoolIndex {
  const int* ids;    // [n] stream of each row of the block
  const int* phase;  // [P] phase words (read only by the compute kernels: stream_pool_phase_kernel updates them in a launch of its own)
  int P;
};

// the pool row of stream ids[b] that holds its history (next: the other half) and its frame parity; false: a dead row (id outside
// [0, P)), which gives zeros and touches no state
__device__ __forceinline__ bool pool_row(const StreamPoolIndex& ix, int b, size_t row_floats, size_t& cur, size_t& next, int& parity) {
  const int id = __ldg(ix.ids + b);
  if ((unsigned)id >= (unsigned)ix.P) return false;
  const int ph = __ldg(ix.phase + id);
  cur = ((size_t)(ph & 1) * ix.P + id) * row_floats;
  next = ((size_t)(~ph & 1) * ix.P + id) * row_floats;
  parity = (ph >> 1) & 1;
  return true;
}

// after a call's compute launches: flip the history half of every listed stream and advance its frame parity by the frames it was
// given (xadv for the analysis words, sadv for the synthesis words; a null word array is left alone)
__global__ void stream_pool_phase_kernel(const int* __restrict__ ids, int n, int P, int* xphase, int xadv, int* sphase, int sadv) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int id = ids[r];
  if ((unsigned)id >= (unsigned)P) return;
  if (xphase != nullptr) {
    const int w = xphase[id];
    xphase[id] = ((w & 1) ^ 1) | ((((w >> 1) + xadv) & 1) << 1);
  }
  if (sphase != nullptr) {
    const int w = sphase[id];
    sphase[id] = ((w & 1) ^ 1) | ((((w >> 1) + sadv) & 1) << 1);
  }
}

}  // namespace pqmf
