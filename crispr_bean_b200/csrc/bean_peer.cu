// bean_peer.cu -- exchange buffers in peer GPU memory for the one data-path collective of the path.
//
// With guides sharded over the GPUs of one box the survival step needs R + 1 library-wide sums between consecutive steps
// (include/bean_b200.h, BeanSurvivalState.sums).  Instead of an NCCL all-reduce issued by the host between two launches, each
// rank owns a small buffer that every other rank of the box maps through CUDA IPC: the last CTA of the per-variant kernel
// STORES its rank's partial sums into every peer's buffer over NVLink and raises a per-step flag there; the next step's guide
// kernel waits for the flags of all ranks in its OWN memory and adds the partials in rank order (svi_variant_kernel /
// surv_guide_kernel).  The host is out of the loop: N steps are one C call, as on a single GPU.  Nothing of the reference
// corresponds to this file (the reference is single-process).
#include <string.h>

#include "bean_common.cuh"

extern "C" {

int bean_peer_exchange_bytes(void) { return (int)sizeof(BeanPeerBuffer); }

// cudaMalloc (not torch's caching allocator: IPC handles name whole allocations) + zero + the IPC handle peers open
int bean_peer_alloc(void** ptr, unsigned char* handle64) {
  BEAN_REQUIRE(ptr && handle64, BEAN_EINVAL, "ptr / handle is NULL");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* p = nullptr;
  BEAN_CUDA(cudaMalloc(&p, sizeof(BeanPeerBuffer)));
  BEAN_CUDA(cudaMemset(p, 0, sizeof(BeanPeerBuffer)));
  BEAN_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    BEAN_CUDA(e);
  }
  memcpy(handle64, &h, 64);
  *ptr = p;
  return BEAN_OK;
}

int bean_peer_open(const unsigned char* handle64, void** ptr) {
  BEAN_REQUIRE(ptr && handle64, BEAN_EINVAL, "ptr / handle is NULL");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  BEAN_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return BEAN_OK;
}

int bean_peer_close(void* ptr) {
  if (ptr) BEAN_CUDA(cudaIpcCloseMemHandle(ptr));
  return BEAN_OK;
}

int bean_peer_free(void* ptr) {
  if (ptr) BEAN_CUDA(cudaFree(ptr));
  return BEAN_OK;
}

// zero the step flags of this rank's own buffer, so that the next exchange waits for steps that are run again (a sharded fit
// that is set back to an earlier step).  Synchronises; every rank must have finished writing to it before (host barrier).
int bean_peer_reset_flags(void* own) {
  BEAN_REQUIRE(own, BEAN_EINVAL, "own is NULL");
  BEAN_CUDA(cudaMemset(static_cast<BeanPeerBuffer*>(own)->flag, 0, sizeof(static_cast<BeanPeerBuffer*>(own)->flag)));
  BEAN_CUDA(cudaDeviceSynchronize());
  return BEAN_OK;
}

// number of waits that gave up (a peer did not publish within BEAN_PEER_TIMEOUT_NS): 0 on a healthy run.  Synchronises.
int bean_peer_timeouts(const void* own, unsigned long long* out) {
  BEAN_REQUIRE(own && out, BEAN_EINVAL, "own / out is NULL");
  BEAN_CUDA(cudaMemcpy(out, &static_cast<const BeanPeerBuffer*>(own)->timeouts, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return BEAN_OK;
}

}  // extern "C"
