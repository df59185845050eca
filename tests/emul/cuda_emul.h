// cuda_emul.h — host stand-ins for the CUDA runtime calls and the kernel-launch syntax used by
// mjlab_b200/csrc/b2sim.cu (tests/emul/build.py rewrites `k<<<g, b, s, st>>>(args)` into EMUL_LAUNCH).
// "Device" memory is host memory, streams and events do nothing, CTAs of a launch run one after the other, each on
// blockDim.x fibers (warp_emul.h).  Test infrastructure only.
#pragma once
#include "warp_emul.h"

#include <functional>
#include <vector>

typedef int cudaError_t;
enum { cudaSuccess = 0 };
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice };
enum { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };

inline cudaError_t cudaMalloc(void** p, size_t n) {
  size_t r = (n + 255) & ~(size_t)255;
  *p = aligned_alloc(256, r ? r : 256);
  return *p ? 0 : 2;
}
template <class T> inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc((void**)p, n); }
inline cudaError_t cudaFree(void* p) { free(p); return 0; }
inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, int) { memcpy(d, s, n); return 0; }
inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, int, cudaStream_t = nullptr) { memcpy(d, s, n); return 0; }
inline cudaError_t cudaMemcpy2DAsync(void* d, size_t dpitch, const void* s, size_t spitch, size_t width, size_t height, int,
                                     cudaStream_t = nullptr) {
  for (size_t r = 0; r < height; r++) memcpy((char*)d + r * dpitch, (const char*)s + r * spitch, width);
  return 0;
}
inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return 0; }
template <class S> inline cudaError_t cudaMemcpyToSymbol(S& sym, const void* s, size_t n) { memcpy(&sym, s, n); return 0; }
template <class S> inline cudaError_t cudaMemcpyFromSymbol(void* d, const S& sym, size_t n) { memcpy(d, &sym, n); return 0; }
inline cudaError_t cudaGetLastError() { return 0; }
inline const char* cudaGetErrorString(cudaError_t) { return "emulated CUDA runtime"; }
inline cudaError_t cudaDeviceSynchronize() { return 0; }
inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
inline cudaError_t cudaSetDevice(int) { return 0; }
inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return 0; }
template <class F> inline cudaError_t cudaFuncSetAttribute(F, int, int) { return 0; }
inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (void*)1; return 0; }
inline cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = (void*)1; return 0; }
inline cudaError_t cudaEventDestroy(cudaEvent_t) { return 0; }
inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = nullptr) { return 0; }
inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return 0; }

namespace cuda_emul {
// run `kernel(args...)` for every CTA of the grid, one CTA at a time, on block.x fibers
template <class K, class... A>
inline void launch(K kernel, dim3 grid, dim3 block, size_t smem, A... args) {
  warp_emul::Ctx& c = warp_emul::ctx();
  const int nt = (int)block.x, nw = (nt + 31) / 32;
  emul_blockDim() = block;
  emul_gridDim() = grid;
  for (int w = 0; w < nw; w++) c.w[w].bar = warp_emul::Bar{0, (w + 1) * 32 <= nt ? 32 : nt - w * 32, 0};
  c.cta = warp_emul::Bar{0, nt, 0};
  c.dyn_smem = aligned_alloc(128, ((smem + 127) & ~(size_t)127) + 128);
  for (unsigned b = 0; b < grid.x; b++) {
    emul_blockIdx() = {b, 0, 0};
    warp_emul::run_fibers(nt, [&]() { kernel(args...); });
  }
  free(c.dyn_smem);
  c.dyn_smem = nullptr;
}
}  // namespace cuda_emul
#define EMUL_LAUNCH(kernel, grid, block, smem, stream, ...) cuda_emul::launch(kernel, dim3(grid), dim3(block), (size_t)(smem), __VA_ARGS__)
