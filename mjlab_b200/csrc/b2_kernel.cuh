// b2_kernel.cuh — fused batched forward-dynamics step, one warp per environment (sm_100a).
//
// Replaces mjwarp.step / mjwarp.forward (reference call sites src/mjlab/sim/sim.py:136,139,187,195;
// pipeline order per SURVEY.md Appendix A.1).  Design (DESIGN.md):
//   * one warp owns one environment for the whole step; 4 warps per CTA, no block-level barriers;
//   * the environment's state vectors are bulk-copied global->shared with cp.async.bulk + mbarrier
//     (TMA 1-D) and every intermediate (poses, spatial inertias, joint-space inertia, contacts,
//     solver scratch) lives in that warp's shared-memory block — nothing but inputs/outputs touches HBM;
//   * the constraint Jacobian is never materialised: contacts of one body pair share a 6x6 block
//     A_g = sum_c S_c W_c S_c^T that is projected through the motion vectors (cdof) of the dofs
//     between the two bodies, so H = M + J^T D J, J v and J^T f cost O(ndof_chain^2) per body pair;
//   * Newton with exact 1-D line search; packed blocked L^T D L, eliminated bottom-up with dof-tree schedules.
// With -DB2_HOST_EMULATION the warp-level helpers (everything above the kernel) compile as plain C++ against
// tests/emul/warp_emul.h (32 host threads in lock step), so they are unit-tested without a GPU.
#pragma once
#ifdef B2_HOST_EMULATION
#include "cuda_emul.h"
#else
#include <cuda_runtime.h>
#endif
#include <math.h>
#include <stdint.h>

#include "b2_types.h"

#define FULL 0xffffffffu
#define MINVAL 1e-15f
#define MINIMP 0.0001f
#define MAXIMP 0.9999f
#define MINMU 1e-5f
// shared-memory record strides chosen odd so lane-per-record accesses are bank-conflict free
#define SD 7   // 6-float records: cdof, cdofdot, cvel, cacc / wrenches
#define SI 11  // 10-float records: cinert, crb


namespace b2 {

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
__device__ __forceinline__ float dot3(const float* a, const float* b) {
  return a[0] * b[0] + a[1] * b[1] + a[2] * b[2];
}
__device__ __forceinline__ void cross3(float* r, const float* a, const float* b) {
  float x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  r[0] = x; r[1] = y; r[2] = z;
}
__device__ __forceinline__ float normalize3(float* a) {
  float n = sqrtf(dot3(a, a));
  if (n < MINVAL) { a[0] = 1.f; a[1] = 0.f; a[2] = 0.f; return n; }
  float inv = 1.f / n;
  a[0] *= inv; a[1] *= inv; a[2] *= inv;
  return n;
}
__device__ __forceinline__ void normalize4(float* q) {
  float n = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1.f; q[1] = q[2] = q[3] = 0.f; return; }
  float inv = 1.f / n;
  q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}
__device__ __forceinline__ void mulquat(float* r, const float* a, const float* b) {
  float w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3];
  float x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2];
  float y = a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1];
  float z = a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0];
  r[0] = w; r[1] = x; r[2] = y; r[3] = z;
}
// r = R(q) v
__device__ __forceinline__ void rotq(float* r, const float* q, const float* v) {
  float t[3], u[3];
  cross3(t, q + 1, v);
  t[0] *= 2.f; t[1] *= 2.f; t[2] *= 2.f;
  cross3(u, q + 1, t);
  r[0] = v[0] + q[0] * t[0] + u[0];
  r[1] = v[1] + q[0] * t[1] + u[1];
  r[2] = v[2] + q[0] * t[2] + u[2];
}
__device__ __forceinline__ void quat2mat(float* m, const float* q) {
  float q00 = q[0] * q[0], q11 = q[1] * q[1], q22 = q[2] * q[2], q33 = q[3] * q[3];
  float q01 = q[0] * q[1], q02 = q[0] * q[2], q03 = q[0] * q[3];
  float q12 = q[1] * q[2], q13 = q[1] * q[3], q23 = q[2] * q[3];
  m[0] = q00 + q11 - q22 - q33; m[4] = q00 - q11 + q22 - q33; m[8] = q00 - q11 - q22 + q33;
  m[1] = 2.f * (q12 - q03); m[2] = 2.f * (q13 + q02);
  m[3] = 2.f * (q12 + q03); m[5] = 2.f * (q23 - q01);
  m[6] = 2.f * (q13 - q02); m[7] = 2.f * (q23 + q01);
}
__device__ __forceinline__ void mul_inert_vec(float* r, const float* i, const float* v) {
  r[0] = i[0] * v[0] + i[3] * v[1] + i[4] * v[2] - i[8] * v[4] + i[7] * v[5];
  r[1] = i[3] * v[0] + i[1] * v[1] + i[5] * v[2] + i[8] * v[3] - i[6] * v[5];
  r[2] = i[4] * v[0] + i[5] * v[1] + i[2] * v[2] - i[7] * v[3] + i[6] * v[4];
  r[3] = i[8] * v[1] - i[7] * v[2] + i[9] * v[3];
  r[4] = i[6] * v[2] - i[8] * v[0] + i[9] * v[4];
  r[5] = i[7] * v[0] - i[6] * v[1] + i[9] * v[5];
}
__device__ __forceinline__ void cross_motion(float* r, const float* vel, const float* v) {
  r[0] = -vel[2] * v[1] + vel[1] * v[2];
  r[1] = vel[2] * v[0] - vel[0] * v[2];
  r[2] = -vel[1] * v[0] + vel[0] * v[1];
  r[3] = -vel[2] * v[4] + vel[1] * v[5] - vel[5] * v[1] + vel[4] * v[2];
  r[4] = vel[2] * v[3] - vel[0] * v[5] + vel[5] * v[0] - vel[3] * v[2];
  r[5] = -vel[1] * v[3] + vel[0] * v[4] - vel[4] * v[0] + vel[3] * v[1];
}
__device__ __forceinline__ void cross_force(float* r, const float* vel, const float* f) {
  r[0] = -vel[2] * f[1] + vel[1] * f[2] - vel[5] * f[4] + vel[4] * f[5];
  r[1] = vel[2] * f[0] - vel[0] * f[2] + vel[5] * f[3] - vel[3] * f[5];
  r[2] = -vel[1] * f[0] + vel[0] * f[1] - vel[4] * f[3] + vel[3] * f[4];
  r[3] = -vel[2] * f[4] + vel[1] * f[5];
  r[4] = vel[2] * f[3] - vel[0] * f[5];
  r[5] = -vel[1] * f[3] + vel[0] * f[4];
}
__device__ __forceinline__ float dot6(const float* a, const float* b) {
  return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3] + a[4] * b[4] + a[5] * b[5];
}
__device__ __forceinline__ int tri(int i, int j) { return (i * (i + 1) >> 1) + j; }  // j <= i
__device__ __forceinline__ int pad4i(int n) { return (n + 3) & ~3; }

#ifndef B2_HOST_EMULATION
// ---- TMA 1-D bulk copy + mbarrier (PTX) -------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes,
                                         unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
               "r"(smem_u32(src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
#else
// host emulation: the bulk copies are plain memcpy by the issuing lane; the warp barrier that precedes
// mbar_wait in the kernel orders them
inline void mbar_init(unsigned long long*, int) {}
inline void mbar_expect(unsigned long long*, uint32_t) {}
inline void bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long*) { memcpy(dst, src, bytes); }
inline void mbar_wait(unsigned long long*, uint32_t) {}
inline void bulk_s2g(void* dst, const void* src, uint32_t bytes) { memcpy(dst, src, bytes); }
inline void bulk_commit_wait() {}
inline void fence_async_smem() {}
#endif  // B2_HOST_EMULATION

#define MP(arr) (m.arr.p + (size_t)w * m.arr.stride)
// Visit the set bits of a 64-bit mask in ascending order, one 32-bit half at a time (64-bit find-first-set,
// clear-lowest and shifts cost twice the instructions; the halves share one copy of the loop body).
#define FOR_BITS64(mask64, d)                                                        \
  _Pragma("unroll 1") for (int h_ = 0; h_ < 2; h_++)                                 \
    for (unsigned w_ = h_ ? (unsigned)((mask64) >> 32) : (unsigned)(mask64), d_ = 0; \
         w_ != 0u && ((d_ = 32u * h_ + (unsigned)__ffs((int)w_) - 1u), true); w_ &= w_ - 1u) \
      for (int d = (int)d_, once_ = 1; once_; once_ = 0)

#ifdef B2_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[32];
#define PHASE_MARK(id)                                                        \
  do {                                                                        \
    __syncwarp();                                                             \
    long long now_ = clock64();                                               \
    if (lane == 0) atomicAdd(&g_phase_cycles[id], (unsigned long long)(now_ - tphase_)); \
    tphase_ = now_;                                                           \
  } while (0)
#else
#define PHASE_MARK(id)
#endif

// approximate reciprocal (MUFU.RCP): the IEEE-rounded __frcp_rn costs ~13 instructions per call
__device__ __forceinline__ float b2_rcp(float x) {
#if defined(B2_HOST_EMULATION) || defined(B2_PRECISE_RCP)
  return __frcp_rn(x);
#else
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#endif
}
// ---- bottom-up blocked L^T D L (leaves first) -----------------------------------------------------------
// Pivots are eliminated from the last dof to the first, four per block step, so the dof tree's zero pattern
// survives (no fill between branches) and the trailing update visits only the entries the tree can make
// non-zero (G1: 437 instead of 1560 pair-visits per factorisation).  In place: A[k,k] = d_k,
// A[k,j] = L_kj d_k (j < k), invdiag[k] = 1/d_k, M = L^T D L with L unit lower.  `list`/`start`: per-block
// schedules (words p | i << 12 | j << 18); with sparse == false (a contact couples two branches) the block
// with m leading rows takes the first tri(m) words of the dense list instead.
// `blk0`: index of the first block's schedule when only the leading n x n part of an nv x nv matrix is factorised
// (n = nv - 4 * blk0).  `snap_n` / `snap`: when the elimination reaches the leading snap_n x snap_n block (all
// pivots >= snap_n done) that block - the Schur complement onto the first snap_n dofs - is copied to `snap`.
__device__ __noinline__ void ldl_factor(float* A, float* invdiag, int n, const unsigned* slist, const int* start,
                                        const unsigned* __restrict__ dense, bool sparse, int lane, int blk0 = 0,
                                        int snap_n = 0, float* snap = nullptr) {
  int blk = blk0;
#pragma unroll 1
  for (int kt = n - 1; kt >= 0; kt -= 4, blk++) {
    if (kt + 1 == snap_n) {
#pragma unroll 1
      for (int i = lane; i < (snap_n * (snap_n + 1) >> 1); i += 32) snap[i] = A[i];
      __syncwarp();
    }
    const int nb = min(4, kt + 1), lead = kt - nb + 1;
    const int rb0 = kt * (kt + 1) >> 1, rb1 = rb0 - kt, rb2 = rb1 - (kt - 1), rb3 = rb2 - (kt - 2);
    float dv[4], Lb[6];
    {
      // 4x4 diagonal block (pivot order kt, kt-1, kt-2, kt-3), factorised redundantly by every lane
      float a10 = 0.f, a11 = 1.f, a20 = 0.f, a21 = 0.f, a22 = 1.f, a30 = 0.f, a31 = 0.f, a32 = 0.f, a33 = 1.f;
      float a00 = A[rb0 + kt];
      if (nb == 4) {  // (every block but possibly the last: one uniform branch instead of three predicated groups)
        a10 = A[rb0 + kt - 1]; a11 = A[rb1 + kt - 1];
        a20 = A[rb0 + kt - 2]; a21 = A[rb1 + kt - 2]; a22 = A[rb2 + kt - 2];
        a30 = A[rb0 + kt - 3]; a31 = A[rb1 + kt - 3]; a32 = A[rb2 + kt - 3]; a33 = A[rb3 + kt - 3];
      } else {
        if (nb > 1) { a10 = A[rb0 + kt - 1]; a11 = A[rb1 + kt - 1]; }
        if (nb > 2) { a20 = A[rb0 + kt - 2]; a21 = A[rb1 + kt - 2]; a22 = A[rb2 + kt - 2]; }
      }
      __syncwarp();  // every lane holds the block before any panel store touches it
      dv[0] = b2_rcp(fmaxf(a00, MINVAL));
      Lb[0] = a10 * dv[0];
      dv[1] = b2_rcp(fmaxf(a11 - a10 * Lb[0], MINVAL));
      Lb[1] = a20 * dv[0];
      float t21 = a21 - a20 * Lb[0];
      Lb[2] = t21 * dv[1];
      dv[2] = b2_rcp(fmaxf(a22 - a20 * Lb[1] - t21 * Lb[2], MINVAL));
      Lb[3] = a30 * dv[0];
      float t31 = a31 - a30 * Lb[0];
      Lb[4] = t31 * dv[1];
      float t32 = a32 - a30 * Lb[1] - t31 * Lb[2];
      Lb[5] = t32 * dv[2];
      dv[3] = b2_rcp(fmaxf(a33 - a30 * Lb[3] - t31 * Lb[4] - t32 * Lb[5], MINVAL));
      invdiag[kt] = dv[0];
      if (nb > 1) invdiag[kt - 1] = dv[1];
      if (nb > 2) invdiag[kt - 2] = dv[2];
      if (nb > 3) invdiag[kt - 3] = dv[3];
    }
    // panel: the pivot rows kt-t at every column q < kt (lane = column); entry (kt-t, q) exists for q <= kt-t
#pragma unroll 1
    for (int base = 0; base < kt; base += 32) {
      const int q = base + lane;
      const bool ok = q < kt;
      float r0 = ok ? A[rb0 + q] : 0.f;
      float r1 = (ok && nb > 1 && q <= kt - 1) ? A[rb1 + q] : 0.f;
      float r2 = (ok && nb > 2 && q <= kt - 2) ? A[rb2 + q] : 0.f;
      float r3 = (ok && nb > 3 && q <= kt - 3) ? A[rb3 + q] : 0.f;
      r1 -= r0 * Lb[0];
      r2 -= r0 * Lb[1] + r1 * Lb[2];
      r3 -= r0 * Lb[3] + r1 * Lb[4] + r2 * Lb[5];
      if (ok && nb > 1 && q <= kt - 1) A[rb1 + q] = r1;
      if (ok && nb > 2 && q <= kt - 2) A[rb2 + q] = r2;
      if (ok && nb > 3 && q <= kt - 3) A[rb3 + q] = r3;
    }
    __syncwarp();
    if (lead <= 0) break;  // (only the last block can be partial, and it has nothing left to update)
    // trailing update: A[i,j] -= sum_t c_t,i c_t,j / d_t over the scheduled entries, c_t,q = A[kt-t, q]
    const unsigned* lst = sparse ? slist + start[blk] : dense;
    const int np = sparse ? start[blk + 1] - start[blk] : (lead * (lead + 1) >> 1);
    // The pivot rows are addressed from row 3's base: rows 2, 1, 0 start kt-2, 2kt-3 and 3kt-3 floats further on,
    // so one index register per operand serves all four loads (offsets folded into the block's row pointers).
    const float* R3 = A + rb3; const float* R2 = A + rb2; const float* R1 = A + rb1; const float* R0 = A + rb0;
    int p = lane;
#pragma unroll 1
    for (; p + 32 < np; p += 64) {
      unsigned e0 = lst[p], e1 = lst[p + 32];
      int i0 = (e0 >> 12) & 63, j0 = e0 >> 18, i1 = (e1 >> 12) & 63, j1 = e1 >> 18;
      float acc0 = A[e0 & 0xfff], acc1 = A[e1 & 0xfff];
      acc0 = fmaf(-R0[i0], R0[j0] * dv[0], acc0); acc1 = fmaf(-R0[i1], R0[j1] * dv[0], acc1);
      acc0 = fmaf(-R1[i0], R1[j0] * dv[1], acc0); acc1 = fmaf(-R1[i1], R1[j1] * dv[1], acc1);
      acc0 = fmaf(-R2[i0], R2[j0] * dv[2], acc0); acc1 = fmaf(-R2[i1], R2[j1] * dv[2], acc1);
      acc0 = fmaf(-R3[i0], R3[j0] * dv[3], acc0); acc1 = fmaf(-R3[i1], R3[j1] * dv[3], acc1);
      A[e0 & 0xfff] = acc0;
      A[e1 & 0xfff] = acc1;
    }
#pragma unroll 1
    for (; p < np; p += 32) {
      unsigned e0 = lst[p];
      int i0 = (e0 >> 12) & 63, j0 = e0 >> 18;
      float acc0 = A[e0 & 0xfff];
      acc0 = fmaf(-R0[i0], R0[j0] * dv[0], acc0);
      acc0 = fmaf(-R1[i0], R1[j0] * dv[1], acc0);
      acc0 = fmaf(-R2[i0], R2[j0] * dv[2], acc0);
      acc0 = fmaf(-R3[i0], R3[j0] * dv[3], acc0);
      A[e0 & 0xfff] = acc0;
    }
    __syncwarp();
  }
}
// x <- (L^T D L)^-1 x for the factor above.  Rows >= 32 are kept out of the two 32-row sweeps (broadcasts in
// the first sweep, warp reductions in the second).
__device__ __noinline__ void ldl_solve(const float* L, const float* invdiag, float* x, int n, int lane) {
  const int n0 = min(n, 32), nh = n - n0;
  float x0 = lane < n0 ? x[lane] : 0.f;
  float x1 = lane < nh ? x[lane + 32] : 0.f;
  const float d0 = lane < n0 ? invdiag[lane] : 0.f, d1 = lane < nh ? invdiag[lane + 32] : 0.f;
  const int r0 = lane * (lane + 1) >> 1;
  // L^T y = b: pivots from the last row up; row k is contiguous (lane = column)
#pragma unroll 1
  for (int j = nh - 1; j >= 0; j--) {
    const int rk = (32 + j) * (33 + j) >> 1;
    float yk = __shfl_sync(FULL, x1, j) * invdiag[32 + j];
    if (lane < j) x1 -= L[rk + 32 + lane] * yk;
    x0 -= L[rk + lane] * yk;
  }
  int rk = n0 * (n0 - 1) >> 1;  // tri(n0 - 1, 0)
  // Pivot k's contribution is A[k,lane] * (u_k / d_k): lane k holds 1/d_k in a register and its u_k is final once
  // the pivots above it are done, so the product is formed there and shuffled (no load of invdiag[k] per step).
  // Unrolled by four: the kernel is issue bound and the loop control was a third of the sweep's instructions.
#pragma unroll 4
  for (int k = n0 - 1; k >= 0; k--) {
    const float yk = __shfl_sync(FULL, x0 * d0, k);
    const float l = lane < k ? L[rk + lane] : 0.f;
    x0 = fmaf(-l, yk, x0);
    rk -= k;
  }
  x0 *= d0; x1 *= d1;  // D z = y
  // L x = z: x_k = z_k - (1/d_k) sum_{j<k} A[k,j] x_j, columns in ascending order (lane = row)
#pragma unroll 4
  for (int j = 0; j < n0; j++) {
    float t = (lane > j && lane < n0) ? L[r0 + j] * d0 : 0.f;
    x0 = fmaf(-t, __shfl_sync(FULL, x0, j), x0);
  }
#pragma unroll 1
  for (int r = 0; r < nh; r++) {
    const int rr = (32 + r) * (33 + r) >> 1;
    float part = L[rr + lane] * x0;  // nh > 0 implies n0 == 32: every lane owns a row < 32
    if (lane < r) part += L[rr + 32 + lane] * x1;
    part = wsum(part);
    if (lane == r) x1 -= d1 * part;
  }
  if (lane < n0) x[lane] = x0;
  if (lane < nh) x[lane + 32] = x1;
  __syncwarp();
}
// y = M x for packed symmetric M (both in shared memory).  One column loop for all lanes (entry (i,j) lives
// at tri(max)+min), four independent accumulators so the loads of four columns are in flight together.
__device__ __noinline__ void symv(const float* M, const float* x, float* y, int n, int lane) {
  #pragma unroll 1
  for (int i = lane; i < n; i += 32) {
    const int ri = i * (i + 1) >> 1;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
    int j = 0, tj = 0;  // tj = tri(j, 0)
    #pragma unroll 1
    for (; j + 4 <= n; j += 4) {
      int a0 = j <= i ? ri + j : tj + i;
      int u1 = tj + j + 1, u2 = u1 + j + 2, u3 = u2 + j + 3;
      int a1 = j + 1 <= i ? ri + j + 1 : u1 + i;
      int a2 = j + 2 <= i ? ri + j + 2 : u2 + i;
      int a3 = j + 3 <= i ? ri + j + 3 : u3 + i;
      t0 += M[a0] * x[j]; t1 += M[a1] * x[j + 1]; t2 += M[a2] * x[j + 2]; t3 += M[a3] * x[j + 3];
      tj = u3 + j + 4;
    }
    #pragma unroll 1
    for (; j < n; j++) {
      t0 += M[j <= i ? ri + j : tj + i] * x[j];
      tj += j + 1;
    }
    y[i] = (t0 + t1) + (t2 + t3);
  }
  __syncwarp();
}

// ---- narrowphase primitives (engine_collision_primitive.c semantics; SURVEY.md Appendix A.9) ----
struct RawCon {
  float dist, pos[3], n[3], yh[3];
};
__device__ __forceinline__ int sphere_sphere(RawCon& c, float margin, const float* p1, float r1,
                                             const float* p2, float r2) {
  float dif[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]};
  float cd = sqrtf(dot3(dif, dif));
  if (cd > margin + r1 + r2) return 0;
  c.dist = cd - r1 - r2;
  normalize3(dif);
  for (int k = 0; k < 3; k++) {
    c.n[k] = dif[k];
    c.pos[k] = p1[k] + dif[k] * (r1 + 0.5f * c.dist);
    c.yh[k] = 0.f;
  }
  return 1;
}
__device__ __forceinline__ int plane_sphere(RawCon& c, float margin, const float* pp, const float* pn,
                                            const float* sp, float r) {
  float dif[3] = {sp[0] - pp[0], sp[1] - pp[1], sp[2] - pp[2]};
  float cd = dot3(dif, pn);
  if (cd > margin + r) return 0;
  c.dist = cd - r;
  for (int k = 0; k < 3; k++) {
    c.n[k] = pn[k];
    c.pos[k] = sp[k] - pn[k] * (r + 0.5f * c.dist);
    c.yh[k] = 0.f;
  }
  return 1;
}
// ---- box primitives (own definitions, identical to oracle/b2_oracle.c: sphere_box, capsule_box, box_box) ----
// poses are 12 floats: pos[3], row-major mat[9]
__device__ __forceinline__ float point_box_dist2(const float* pt, const float* bx, const float* h) {
  float d[3] = {pt[0] - bx[0], pt[1] - bx[1], pt[2] - bx[2]}, sum = 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    float l = bx[3 + k] * d[0] + bx[6 + k] * d[1] + bx[9 + k] * d[2];
    float e = l > h[k] ? l - h[k] : (l < -h[k] ? l + h[k] : 0.f);
    sum += e * e;
  }
  return sum;
}
__device__ __noinline__ int sphere_box(RawCon& c, float margin, const float* sp, float r, const float* bx,
                                       const float* h) {
  float d[3] = {sp[0] - bx[0], sp[1] - bx[1], sp[2] - bx[2]}, l[3], cl[3], nl[3];
  bool inside = true;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    l[k] = bx[3 + k] * d[0] + bx[6 + k] * d[1] + bx[9 + k] * d[2];
    cl[k] = fminf(fmaxf(l[k], -h[k]), h[k]);
    if (cl[k] != l[k]) inside = false;
  }
  float dist;
  if (!inside) {
    float e[3] = {l[0] - cl[0], l[1] - cl[1], l[2] - cl[2]};
    float dc = sqrtf(dot3(e, e));
    if (dc > r + margin) return 0;
    dist = dc - r;
    float inv = 1.f / dc;
    nl[0] = -e[0] * inv; nl[1] = -e[1] * inv; nl[2] = -e[2] * inv;
  } else {
    int best = 0; float depth = h[0] - fabsf(l[0]);
#pragma unroll
    for (int k = 1; k < 3; k++) { float t = h[k] - fabsf(l[k]); if (t < depth) { depth = t; best = k; } }
    nl[0] = nl[1] = nl[2] = 0.f;
    float sg = l[best] >= 0.f ? -1.f : 1.f;
    if (best == 0) nl[0] = sg; else if (best == 1) nl[1] = sg; else nl[2] = sg;
    dist = -(depth + r);
  }
  c.dist = dist;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    float nk = bx[3 + 3 * k] * nl[0] + bx[4 + 3 * k] * nl[1] + bx[5 + 3 * k] * nl[2];
    c.n[k] = nk; c.pos[k] = sp[k] + nk * (r + 0.5f * dist); c.yh[k] = 0.f;
  }
  return 1;
}
// distance from the axis point l0 + t*al (box frame) to the box
__device__ __forceinline__ float axis_box_dist(const float* l0, const float* al, float t, const float* h) {
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    float l = l0[k] + al[k] * t;
    float e = l > h[k] ? l - h[k] : (l < -h[k] ? l + h[k] : 0.f);
    sum += e * e;
  }
  return sqrtf(sum);
}
__device__ __noinline__ int capsule_box(RawCon* c, float margin, const float* cp, const float* cs, const float* bx,
                                        const float* h) {
  float ax[3] = {cp[3 + 2], cp[3 + 5], cp[3 + 8]}, len = cs[1], r = cs[0];
  float d0[3] = {cp[0] - bx[0], cp[1] - bx[1], cp[2] - bx[2]}, l0[3], al[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    l0[k] = bx[3 + k] * d0[0] + bx[6 + k] * d0[1] + bx[9 + k] * d0[2];
    al[k] = bx[3 + k] * ax[0] + bx[6 + k] * ax[1] + bx[9 + k] * ax[2];
  }
  float lo = -len, hi = len;
  const float gr = 0.6180339887498949f;
  float x1 = hi - gr * (hi - lo), x2 = lo + gr * (hi - lo);
  float f1 = axis_box_dist(l0, al, x1, h), f2 = axis_box_dist(l0, al, x2, h);
  #pragma unroll 1
  for (int it = 0; it < 24; it++) {
    if (f1 <= f2) { hi = x2; x2 = x1; f2 = f1; x1 = hi - gr * (hi - lo); f1 = axis_box_dist(l0, al, x1, h); }
    else { lo = x1; x1 = x2; f1 = f2; x2 = lo + gr * (hi - lo); f2 = axis_box_dist(l0, al, x2, h); }
  }
  float ts = 0.5f * (lo + hi);
  float dmin = axis_box_dist(l0, al, ts, h);
  if (dmin > r + margin) return 0;
  float level = dmin + 1e-3f * r;
  float ta = -len, tb = len;
  if (axis_box_dist(l0, al, -len, h) > level) {
    float a = -len, b = ts;   // d(a) > level >= d(b)
    #pragma unroll 1
    for (int it = 0; it < 16; it++) {
      float mid = 0.5f * (a + b);
      if (axis_box_dist(l0, al, mid, h) > level) a = mid; else b = mid;
    }
    ta = b;
  }
  if (axis_box_dist(l0, al, len, h) > level) {
    float a = ts, b = len;    // d(a) <= level < d(b)
    #pragma unroll 1
    for (int it = 0; it < 16; it++) {
      float mid = 0.5f * (a + b);
      if (axis_box_dist(l0, al, mid, h) > level) b = mid; else a = mid;
    }
    tb = a;
  }
  int n = 0;
  float p[3];
  if (tb - ta < 0.02f * len) {
    float tm = 0.5f * (ta + tb);
    p[0] = cp[0] + ax[0] * tm; p[1] = cp[1] + ax[1] * tm; p[2] = cp[2] + ax[2] * tm;
    n += sphere_box(c[n], margin, p, r, bx, h);
  } else {
    p[0] = cp[0] + ax[0] * ta; p[1] = cp[1] + ax[1] * ta; p[2] = cp[2] + ax[2] * ta;
    n += sphere_box(c[n], margin, p, r, bx, h);
    p[0] = cp[0] + ax[0] * tb; p[1] = cp[1] + ax[1] * tb; p[2] = cp[2] + ax[2] * tb;
    n += sphere_box(c[n], margin, p, r, bx, h);
  }
  return n;
}
// box - box: separating-axis test (15 axes), then either the incident face clipped against the reference face
// (<= 8 contacts) or one edge-edge contact; the same statement as oracle/b2_oracle.c: box_box (see there).
__device__ __noinline__ int box_box(RawCon* c, float margin, const float* x1, const float* h1, const float* x2,
                                    const float* h2) {
  const float *p1 = x1, *m1 = x1 + 3, *p2 = x2, *m2 = x2 + 3;
  float A[3][3], B[3][3], R[3][3], Q[3][3], t[3] = {p2[0] - p1[0], p2[1] - p1[1], p2[2] - p1[2]}, tA[3], tB[3];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int k = 0; k < 3; k++) { A[i][k] = m1[3 * k + i]; B[i][k] = m2[3 * k + i]; }  // axes = columns
#pragma unroll
  for (int i = 0; i < 3; i++) {
    tA[i] = dot3(t, A[i]); tB[i] = dot3(t, B[i]);
#pragma unroll
    for (int j = 0; j < 3; j++) { R[i][j] = dot3(A[i], B[j]); Q[i][j] = fabsf(R[i][j]) + 1e-6f; }
  }
  int best = -1; float bdepth = 0.f;
#pragma unroll
  for (int i = 0; i < 3; i++) {  // face axes of box 1
    float depth = h1[i] + h2[0] * Q[i][0] + h2[1] * Q[i][1] + h2[2] * Q[i][2] - fabsf(tA[i]);
    if (depth < -margin) return 0;
    if (best < 0 || depth < bdepth - 1e-5f * (1.f + fabsf(bdepth))) { best = i; bdepth = depth; }
  }
#pragma unroll
  for (int j = 0; j < 3; j++) {  // face axes of box 2
    float depth = h2[j] + h1[0] * Q[0][j] + h1[1] * Q[1][j] + h1[2] * Q[2][j] - fabsf(tB[j]);
    if (depth < -margin) return 0;
    if (depth < bdepth - 1e-5f * (1.f + fabsf(bdepth))) { best = 3 + j; bdepth = depth; }
  }
  #pragma unroll 1
  for (int e = 0; e < 9; e++) {  // edge axes a_i x b_j
    const int i = e / 3, j = e - 3 * i;
    float l2 = 1.f - R[i][j] * R[i][j];
    if (l2 < 1e-6f) continue;  // (nearly) parallel edges: covered by the face axes
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
    float il = 1.f / sqrtf(l2);
    float depth = (h1[i1] * Q[i2][j] + h1[i2] * Q[i1][j] + h2[j1] * Q[i][j2] + h2[j2] * Q[i][j1] -
                   fabsf(tA[i2] * R[i1][j] - tA[i1] * R[i2][j])) * il;
    if (depth < -margin) return 0;
    if (depth + 0.05f * fabsf(depth) + 1e-6f < bdepth) { best = 6 + e; bdepth = depth; }
  }
  if (best >= 6) {
    const int i = (best - 6) / 3, j = (best - 6) % 3;
    float L[3];
    cross3(L, A[i], B[j]);
    normalize3(L);
    if (dot3(L, t) < 0.f) { L[0] = -L[0]; L[1] = -L[1]; L[2] = -L[2]; }
    float pa[3] = {p1[0], p1[1], p1[2]}, pb[3] = {p2[0], p2[1], p2[2]};
    for (int k = 0; k < 3; k++) {
      if (k != i) { float sg = dot3(A[k], L) >= 0.f ? h1[k] : -h1[k]; for (int x = 0; x < 3; x++) pa[x] += sg * A[k][x]; }
      if (k != j) { float sg = dot3(B[k], L) >= 0.f ? -h2[k] : h2[k]; for (int x = 0; x < 3; x++) pb[x] += sg * B[k][x]; }
    }
    float d[3] = {pb[0] - pa[0], pb[1] - pa[1], pb[2] - pa[2]}, r = R[i][j], da = dot3(d, A[i]), db = dot3(d, B[j]);
    float den = 1.f - r * r;
    float sA = (da - r * db) / den, sB = (r * da - db) / den;
    sA = fminf(fmaxf(sA, -h1[i]), h1[i]);
    sB = fminf(fmaxf(sB, -h2[j]), h2[j]);
    c[0].dist = -bdepth;
    for (int x = 0; x < 3; x++) {
      c[0].pos[x] = 0.5f * (pa[x] + sA * A[i][x] + pb[x] + sB * B[j][x]);
      c[0].n[x] = L[x]; c[0].yh[x] = 0.f;
    }
    return 1;
  }
  const int ref = best >= 3, ax = ref ? best - 3 : best;
  float (*Ar)[3] = ref ? B : A; float (*Ai)[3] = ref ? A : B;
  const float *pr = ref ? p2 : p1, *pi = ref ? p1 : p2, *hr = ref ? h2 : h1, *hi = ref ? h1 : h2;
  float sgn = (ref ? -tB[ax] : tA[ax]) >= 0.f ? 1.f : -1.f;
  float n[3] = {sgn * Ar[ax][0], sgn * Ar[ax][1], sgn * Ar[ax][2]};
  int inc = 0; float bd = fabsf(dot3(n, Ai[0]));
  for (int k = 1; k < 3; k++) { float v = fabsf(dot3(n, Ai[k])); if (v > bd + 1e-6f) { bd = v; inc = k; } }
  float si = dot3(n, Ai[inc]) > 0.f ? -1.f : 1.f;
  const int k1 = (inc + 1) % 3, k2 = (inc + 2) % 3, u1 = (ax + 1) % 3, u2 = (ax + 2) % 3;
  float poly[16][3], tmp[16][3]; int np_ = 4;
  for (int v = 0; v < 4; v++) {
    float s1 = (v == 0 || v == 3) ? hi[k1] : -hi[k1], s2 = (v < 2) ? hi[k2] : -hi[k2];
    for (int x = 0; x < 3; x++) poly[v][x] = pi[x] + si * hi[inc] * Ai[inc][x] + s1 * Ai[k1][x] + s2 * Ai[k2][x];
  }
  #pragma unroll 1
  for (int pl = 0; pl < 4 && np_ > 0; pl++) {  // the four side planes of the reference face
    const float* u = Ar[pl < 2 ? u1 : u2]; float lim = hr[pl < 2 ? u1 : u2] + 1e-6f, sg = (pl & 1) ? -1.f : 1.f;
    int nt = 0;
    #pragma unroll 1
    for (int v = 0; v < np_; v++) {
      const float *P = poly[v], *Qv = poly[(v + 1) % np_];
      float dP = sg * ((P[0] - pr[0]) * u[0] + (P[1] - pr[1]) * u[1] + (P[2] - pr[2]) * u[2]) - lim;
      float dQ = sg * ((Qv[0] - pr[0]) * u[0] + (Qv[1] - pr[1]) * u[1] + (Qv[2] - pr[2]) * u[2]) - lim;
      if (dP <= 0.f) { for (int x = 0; x < 3; x++) tmp[nt][x] = P[x]; nt++; }
      if ((dP <= 0.f) != (dQ <= 0.f)) { float f = dP / (dP - dQ); for (int x = 0; x < 3; x++) tmp[nt][x] = P[x] + f * (Qv[x] - P[x]); nt++; }
    }
    np_ = nt > 8 ? 8 : nt;
    for (int v = 0; v < np_; v++) for (int x = 0; x < 3; x++) poly[v][x] = tmp[v][x];
  }
  int nc = 0;
  #pragma unroll 1
  for (int v = 0; v < np_ && nc < 8; v++) {
    float depth = hr[ax] - ((poly[v][0] - pr[0]) * n[0] + (poly[v][1] - pr[1]) * n[1] + (poly[v][2] - pr[2]) * n[2]);
    if (depth < -margin) continue;
    c[nc].dist = -depth;
    for (int x = 0; x < 3; x++) {
      c[nc].pos[x] = poly[v][x] + 0.5f * depth * n[x];
      c[nc].n[x] = ref ? -n[x] : n[x];  // from box 1 to box 2
      c[nc].yh[x] = 0.f;
    }
    nc++;
  }
  return nc;
}
// ---- mesh / height-field pairs: convex routines of b2_convex.h (GJK / EPA, single source with the oracle) ----
#define B2C_REAL float
#define B2C_FN __device__ __noinline__
#define B2C_INL __device__ __forceinline__
#define B2C_SQRT sqrtf
#include "b2_convex.h"
// a, b: pose records (pos[3], mat[9], rbound, margin) of geoms g1, g2 with type(g1) <= type(g2)
__device__ __noinline__ int convex_narrowphase(RawCon* rc, float margin, const DevModel& m, int g1, int g2,
                                               const float* a, const float* b, const float* s1, const float* s2) {
  const int t1 = m.geom_type[g1], t2 = m.geom_type[g2];
  B2CCon cc[B2C_MAXOUT];
  B2CShape A, B;
  const float* v2 = nullptr; int n2 = 0;
  if (t2 == G_MESH) { int id = m.geom_dataid[g2]; v2 = m.mesh_vert + 3 * m.mesh_vertadr[id]; n2 = m.mesh_vertnum[id]; }
  const float r2 = b2c_shape(&B, t2, b, b + 3, s2, v2, n2);
  int n = 0;
  if (t1 == G_PLANE) {
    float pn[3] = {a[3 + 2], a[3 + 5], a[3 + 8]};
    if (t2 == G_CYLINDER) n = b2c_plane_cylinder(cc, margin, a, pn, b, b + 3, s2);
    else if (t2 == G_ELLIPSOID) n = b2c_plane_ellipsoid(cc, margin, a, pn, &B);
    else n = b2c_plane_mesh(cc, margin, a, pn, &B);
  } else if (t1 == G_HFIELD) {
    n = 0;  // height-field pairs go through hfield_lanes
  } else {
    const float* v1 = nullptr; int n1 = 0;
    if (t1 == G_MESH) { int id = m.geom_dataid[g1]; v1 = m.mesh_vert + 3 * m.mesh_vertadr[id]; n1 = m.mesh_vertnum[id]; }
    const float r1 = b2c_shape(&A, t1, a, a + 3, s1, v1, n1);
    n = b2c_pair(cc, margin, &A, r1, &B, r2, a, b, a[12] + b[12]);
  }
  for (int i = 0; i < n; i++) {
    rc[i].dist = cc[i].dist;
    for (int k = 0; k < 3; k++) { rc[i].pos[k] = cc[i].pos[k]; rc[i].n[k] = cc[i].n[k]; rc[i].yh[k] = 0.f; }
  }
  return n;
}

// Pose record (pos[3], mat[9], rbound, ...) of a collision geom from its slot code: a shared-memory slot, or
// -2 - index of a height field welded to the world (posed once at create, global memory)
__device__ __forceinline__ const float* cpose(const float* gpose, const DevModel& m, int cs) {
  return cs >= 0 ? gpose + GP * cs : m.fixed_pose + 16 * (size_t)(-2 - cs);
}
// Height-field pairs of one batch of 32 candidates, with the prisms of all pairs spread over the lanes.
// Called by the whole warp; lane `lane` owns the pair (g1 = height field, g2, poses a / b) when `hf`.
// Per pair the work is a list of items (cell, triangle) under the geom's footprint (b2c_hfield_range); most
// are rejected by two cheap tests (b2c_hfield_cull) and the rest need GJK / EPA on a prism (b2c_hfield_prism).
// One lane per pair leaves the warp waiting for the limb with the most prisms (3.4 GJK calls on the slowest
// lane of 7.7 per environment on the rough-terrain workload): here every lane culls one item per round, the
// survivors queue up in shared memory and are solved 32 at a time.  Contacts are merged by the owning lane in
// ascending item order, which is the order of the sequential driver b2c_hfield (same contacts, same order).
// scratch: HF_SCRATCH words of shared memory (records of the 32 owners + the queue).
#define HF_REC 12
#define HF_SCRATCH (32 * HF_REC + 64)
__device__ __forceinline__ const float* hf_ptr(const int* rec) {
  return (const float*)(((unsigned long long)(unsigned)rec[1] << 32) | (unsigned long long)(unsigned)rec[0]);
}
__device__ __noinline__ int hfield_lanes(RawCon* rc, bool hf, float margin, const DevModel& m, const float* gsize,
                                         int g1, int g2, const float* a, const float* b, int* scratch, int lane) {
  int* rec = scratch + HF_REC * lane;
  int* queue = scratch + 32 * HF_REC;
#ifdef B2_PHASE_TIMING
  long long tphase_ = clock64();
#endif
  B2CHfRange R;
  R.count = 0;
  if (hf) {
    const int t2 = m.geom_type[g2];
    B2CShape B;
    const float* v2 = nullptr; int n2 = 0;
    if (t2 == G_MESH) { int id = m.geom_dataid[g2]; v2 = m.mesh_vert + 3 * m.mesh_vertadr[id]; n2 = m.mesh_vertnum[id]; }
    const float r2 = b2c_shape(&B, t2, b, b + 3, gsize + 3 * g2, v2, n2);
    const int id = m.geom_dataid[g1];
    b2c_hfield_range(&R, margin, a, a + 3, m.hfield_size + 4 * id, m.hfield_nrow[id], m.hfield_ncol[id], &B, r2, b, b[12]);
    rec[0] = (int)(unsigned)(unsigned long long)a; rec[1] = (int)(unsigned)((unsigned long long)a >> 32);
    rec[2] = (int)(unsigned)(unsigned long long)b; rec[3] = (int)(unsigned)((unsigned long long)b >> 32);
    rec[4] = g1; rec[5] = g2; rec[6] = __float_as_int(margin);
    rec[7] = R.r0; rec[8] = R.c0; rec[9] = R.ncc; rec[10] = __float_as_int(R.lo2);
  }
  int incl = R.count;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(FULL, incl, 31);
  PHASE_MARK(21);  // footprints
  if (total == 0) return 0;
  __syncwarp();
  B2CCon out[B2C_MAXOUT];
  int order[B2C_MAXOUT], n = 0;
  float tie = 0.f;
  if (hf) { const int id = m.geom_dataid[g1]; tie = b2c_hfield_tie(m.hfield_size + 4 * id, m.hfield_nrow[id], m.hfield_ncol[id], b[12]); }
  int qn = 0;
  #pragma unroll 1
  for (int i0 = 0; i0 < total || qn > 0;) {
    if (i0 < total) {
      // cull: item i of the concatenated lists; its owner is the first lane whose inclusive count exceeds i
      const int i = min(i0 + lane, total - 1);
      int ow = 0;
#pragma unroll
      for (int st = 16; st > 0; st >>= 1) {
        int v = __shfl_sync(FULL, incl, ow + st - 1);
        if (v <= i) ow += st;
      }
      const int first = __shfl_sync(FULL, incl - R.count, ow);
      bool keep = false;
      if (i0 + lane < total) {
        const int* q = scratch + HF_REC * ow;
        const float *qa = hf_ptr(q), *qb = hf_ptr(q + 2);
        const int h1 = q[4], h2 = q[5], t2 = m.geom_type[h2], id = m.geom_dataid[h1];
        B2CHfRange Q;
        Q.r0 = q[7]; Q.c0 = q[8]; Q.ncc = q[9]; Q.lo2 = __int_as_float(q[10]); Q.count = 0;
        B2CShape B;
        const float* v2 = nullptr; int n2 = 0;
        if (t2 == G_MESH) { int mid = m.geom_dataid[h2]; v2 = m.mesh_vert + 3 * m.mesh_vertadr[mid]; n2 = m.mesh_vertnum[mid]; }
        const float r2 = b2c_shape(&B, t2, qb, qb + 3, gsize + 3 * h2, v2, n2);
        keep = b2c_hfield_cull(&Q, i - first, __int_as_float(q[6]), qa, qa + 3, m.hfield_size + 4 * id, m.hfield_nrow[id],
                               m.hfield_ncol[id], m.hfield_data + m.hfield_adr[id], &B, r2) != 0;
      }
      const unsigned km = __ballot_sync(FULL, keep);
      if (keep) queue[qn + __popc(km & ((1u << lane) - 1u))] = (ow << 24) | (i - first);
      qn += __popc(km);
      i0 += 32;
      __syncwarp();
      PHASE_MARK(22);  // cull
    }
    if (qn >= 32 || (i0 >= total && qn > 0)) {
      const int take = min(qn, 32);
      const bool act = lane < take;
      const int code = act ? queue[lane] : 0;
      const int ow = code >> 24, j = code & 0xffffff;
      bool hit = false;
      B2CCon cn;
      cn.dist = 0.f; cn.pos[0] = cn.pos[1] = cn.pos[2] = 0.f; cn.n[0] = cn.n[1] = cn.n[2] = 0.f;
      if (act) {
        const int* q = scratch + HF_REC * ow;
        const float *qa = hf_ptr(q), *qb = hf_ptr(q + 2);
        const int h1 = q[4], h2 = q[5], t2 = m.geom_type[h2], id = m.geom_dataid[h1];
        B2CHfRange Q;
        Q.r0 = q[7]; Q.c0 = q[8]; Q.ncc = q[9]; Q.lo2 = __int_as_float(q[10]); Q.count = 0;
        B2CShape B;
        const float* v2 = nullptr; int n2 = 0;
        if (t2 == G_MESH) { int mid = m.geom_dataid[h2]; v2 = m.mesh_vert + 3 * m.mesh_vertadr[mid]; n2 = m.mesh_vertnum[mid]; }
        const float r2 = b2c_shape(&B, t2, qb, qb + 3, gsize + 3 * h2, v2, n2);
        hit = b2c_hfield_prism(&cn, &Q, j, __int_as_float(q[6]), qa, qa + 3, m.hfield_size + 4 * id, m.hfield_nrow[id],
                               m.hfield_ncol[id], m.hfield_data + m.hfield_adr[id], &B, r2, qb, qb[12]) != 0;
      }
      unsigned hm = __ballot_sync(FULL, hit);
      #pragma unroll 1
      while (hm) {
        const int sl = __ffs((int)hm) - 1;
        hm &= hm - 1u;
        const int dst = __shfl_sync(FULL, ow, sl), jj = __shfl_sync(FULL, j, sl);
        B2CCon c2;
        c2.dist = __shfl_sync(FULL, cn.dist, sl);
#pragma unroll
        for (int k = 0; k < 3; k++) { c2.pos[k] = __shfl_sync(FULL, cn.pos[k], sl); c2.n[k] = __shfl_sync(FULL, cn.n[k], sl); }
        if (lane == dst) b2c_hfield_keep(out, order, &n, &c2, jj, tie);
      }
      const int rest = qn - take;
      const int mv = lane < rest ? queue[32 + lane] : 0;
      __syncwarp();
      if (lane < rest) queue[lane] = mv;
      __syncwarp();
      qn = rest;
      PHASE_MARK(23);  // prisms (GJK / EPA) + merge
    }
  }
  b2c_hfield_sort(out, order, n);
  for (int i = 0; i < n; i++) {
    rc[i].dist = out[i].dist;
    for (int k = 0; k < 3; k++) { rc[i].pos[k] = out[i].pos[k]; rc[i].n[k] = out[i].n[k]; rc[i].yh[k] = 0.f; }
  }
  return n;
}

__device__ __forceinline__ void make_frame(float* f /*9: n, yhint -> n,t1,t2*/) {
  normalize3(f);
  if (sqrtf(dot3(f + 3, f + 3)) < 0.5f) {
    f[3] = f[4] = f[5] = 0.f;
    if (f[1] < 0.5f && f[1] > -0.5f) f[4] = 1.f; else f[5] = 1.f;
  }
  float t = dot3(f, f + 3);
  f[3] -= t * f[0]; f[4] -= t * f[1]; f[5] -= t * f[2];
  normalize3(f + 3);
  cross3(f + 6, f, f + 3);
}

// dst rows (+)= J x for every constraint row: contacts (4 pyramid rows, or row 0 for condim 1) and
// joint limits.  J is never formed: per body-pair group g the relative spatial velocity
// V_g = sum_{d in chain(b2) xor chain(b1)} (+-) cdof_d x_d is shared by all contacts of the group.
__device__ __noinline__ void mulJ(const float* x, int dstc, int dstl, bool accumulate, float* con,
                                  float* lim, const int* gstart, float* gV, const float* cdof,
                                  const unsigned long long* __restrict__ dofmask, int ncon, int nlim,
                                  int ngroup, int MC, int NLC, int lane) {
  #pragma unroll 1
  for (int g0 = 0; g0 < ngroup; g0 += 5) {
    int gi = lane / 6, comp = lane - 6 * gi, g = g0 + gi;
    if (gi < 5 && g < ngroup) {
      int key = ((int*)con)[CINFO * MC + gstart[g]] & 0xffff;
      unsigned long long m2 = dofmask[key >> 8];
      unsigned long long mk = dofmask[key & 0xff] ^ m2;
      float acc = 0.f;
      // (the two 32-bit halves separately: 64-bit find-first-set / shifts cost twice the instructions)
#pragma unroll
      for (int h = 0; h < 2; h++) {
        unsigned wd = h ? (unsigned)(mk >> 32) : (unsigned)mk;
        const unsigned sg = h ? (unsigned)(m2 >> 32) : (unsigned)m2;
        const float* cd = cdof + SD * 32 * h + comp;
        const float* xx = x + 32 * h;
        while (wd) {
          int d = __ffs((int)wd) - 1;
          wd &= wd - 1u;
          float v = cd[SD * d] * xx[d];
          acc += (sg >> d & 1u) ? v : -v;
        }
      }
      gV[6 * g + comp] = acc;
    }
  }
  __syncwarp();
  #pragma unroll 1
  for (int c = lane; c < ncon; c += 32) {
    const float* V = gV + 6 * (((int*)con)[CINFO * MC + c] >> 24 & 0xff);
    float a3[3];
#pragma unroll
    for (int mm = 0; mm < 3; mm++) {
      float t = 0.f;
#pragma unroll
      for (int a = 0; a < 6; a++) t += con[(CS0 + 6 * mm + a) * MC + c] * V[a];
      a3[mm] = t;
    }
    float mu = con[CMU * MC + c];
    int dim = ((int*)con)[CINFO * MC + c] >> 16 & 0xf;
    float r0, r1, r2, r3;
    if (dim == 1) { r0 = a3[0]; r1 = r2 = r3 = 0.f; }
    else if (dim == 0) { r0 = r1 = r2 = r3 = 0.f; }
    else { r0 = a3[0] + mu * a3[1]; r1 = a3[0] - mu * a3[1]; r2 = a3[0] + mu * a3[2]; r3 = a3[0] - mu * a3[2]; }
    if (accumulate) {
      con[(dstc + 0) * MC + c] += r0; con[(dstc + 1) * MC + c] += r1;
      con[(dstc + 2) * MC + c] += r2; con[(dstc + 3) * MC + c] += r3;
    } else {
      con[(dstc + 0) * MC + c] = r0; con[(dstc + 1) * MC + c] = r1;
      con[(dstc + 2) * MC + c] = r2; con[(dstc + 3) * MC + c] = r3;
    }
  }
  #pragma unroll 1
  for (int r = lane; r < nlim; r += 32) {
    int info = ((int*)lim)[LINFO * NLC + r];
    float v = ((info >> 16 & 1) ? -1.f : 1.f) * x[info & 0xffff];
    if (accumulate) lim[dstl * NLC + r] += v; else lim[dstl * NLC + r] = v;
  }
  __syncwarp();
}
// sum over rows of 0.5*D*min(r,0)^2 for the residuals stored in field (fc, fl)
__device__ __noinline__ float rows_cost(int fc, int fl, const float* con, const float* lim, int ncon,
                                        int nlim, int MC, int NLC, int lane) {
  float cost = 0.f;
  #pragma unroll 1
  for (int c = lane; c < ncon; c += 32) {
    float D = con[CD * MC + c];
#pragma unroll
    for (int r = 0; r < 4; r++) {
      float v = con[(fc + r) * MC + c];
      if (v < 0.f) cost += 0.5f * D * v * v;
    }
  }
  #pragma unroll 1
  for (int r = lane; r < nlim; r += 32) {
    float v = lim[fl * NLC + r];
    if (v < 0.f) cost += 0.5f * lim[LD * NLC + r] * v * v;
  }
  return wsum(cost);
}

}  // namespace b2

// ==================================================================================================
// The kernel
// ==================================================================================================
// MODE bit 0: integrate (step) or not (forward); bit 1: the model has mesh / height-field collision pairs.  The
// convex routines are ~120 KB of code: models without such pairs (BASELINE configs A-E) run the instantiation
// that does not contain them (measured: their presence alone costs 2 % of the G1 step through code layout).
template <int MODE>
__global__ void __launch_bounds__(32 * B2_WARPS_PER_CTA, B2_MIN_CTAS)
b2_step_kernel(const __grid_constant__ DevModel m, const __grid_constant__ DevData dd) {
  using namespace b2;
  constexpr bool STEP = (MODE & 1) != 0, CVX = (MODE & 2) != 0;
#ifdef B2_HOST_EMULATION
  float* smem_all = (float*)warp_emul::ctx().dyn_smem;
#else
  extern __shared__ __align__(16) float smem_all[];
#endif
  __shared__ __align__(8) unsigned long long bars[B2_WARPS_PER_CTA];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per-CTA copy of the factorisation pair schedule (shared by the CTA's warps)
  unsigned* s_sched = (unsigned*)(smem_all + (size_t)B2_WARPS_PER_CTA * m.lay.total);
#define SCHED s_sched, (const int*)s_sched + m.ldl_nsparse, m.ldl_dense
#define FACTOR(sp) ldl_factor(H, invdiag, nv, SCHED, sp, lane)
#define SOLVE(v, tree) ldl_solve(H, invdiag, v, nv, lane)
  // Phase-synchronous execution (dd.phase_sync): the kernel's code is ~200 KB against a 32 KB instruction cache,
  // so the CTA's warps are re-aligned at every phase boundary, at one vote per Newton iteration and between the
  // three segments of an iteration, and they fetch the same code together.
  const bool psync = dd.phase_sync != 0;
#define PSYNC() do { if (psync) __syncthreads(); } while (0)
#pragma unroll 1
  for (int i = threadIdx.x; i < m.ldl_nsparse; i += 32 * B2_WARPS_PER_CTA) s_sched[i] = m.ldl_sparse[i];
  if (threadIdx.x < 18) s_sched[m.ldl_nsparse + threadIdx.x] = (unsigned)m.ldl_start[threadIdx.x];
  if (lane == 0) mbar_init(&bars[warp], 1);
  __syncthreads();  // the only block barrier; nothing below synchronises across warps
  const Layout& L = m.lay;
  float* s = smem_all + (size_t)warp * L.total;
  const int nq = m.nq, nv = m.nv, nu = m.nu, nb = m.nbody, njnt = m.njnt;
  const int MC = L.maxcon, NLC = L.nlimcap;
  // One warp per launch slot; environments are handed out heavy-first (dd.world_order).
  const int slot = blockIdx.x * B2_WARPS_PER_CTA + warp;
  if (slot >= dd.world_count) return;
  const int w = dd.world_order != nullptr ? dd.world_order[dd.world_base + slot] : dd.world_base + slot;
  if (dd.world_mask != nullptr && dd.world_mask[w] == 0) return;
#ifdef B2_PHASE_TIMING
  long long tphase_ = clock64();
#endif

  // ---------------- phase 0: TMA bulk load of this environment's state -------------------------
  float* qpos = s + L.qpos; float* qvel = s + L.qvel; float* qacc_ws = s + L.qacc_ws;
  // inputs with a single use (phase 4) are read from global memory in place
  const float* ctrl = dd.ctrl.p + (size_t)w * dd.ctrl.stride;
  const float* qfrc_applied = dd.qfrc_applied.p + (size_t)w * dd.qfrc_applied.stride;
  const float* xfrc = dd.xfrc_applied.p + (size_t)w * dd.xfrc_applied.stride;
  {
    unsigned long long* bar = &bars[warp];
    fence_async_smem();  // the barrier's initialisation precedes the bulk writes that complete on it
    __syncwarp();
    if (lane == 0) {
      uint32_t bytes = 4u * (dd.qpos.stride + dd.qvel.stride + dd.qacc_warmstart.stride);
      mbar_expect(bar, bytes);
      bulk_g2s(qpos, dd.qpos.p + (size_t)w * dd.qpos.stride, 4u * dd.qpos.stride, bar);
      bulk_g2s(qvel, dd.qvel.p + (size_t)w * dd.qvel.stride, 4u * dd.qvel.stride, bar);
      bulk_g2s(qacc_ws, dd.qacc_warmstart.p + (size_t)w * dd.qacc_warmstart.stride, 4u * dd.qacc_warmstart.stride, bar);
    }
    __syncwarp();
    mbar_wait(bar, 0);
  }

  PHASE_MARK(0);
  PSYNC();
  float* xpos = s + L.xpos; float* xquat = s + L.xquat; float* xipos = s + L.xipos;
  float* scom = s + L.scom; float* xanchor = s + L.xanchor; float* xaxis = s + L.xaxis;
  float* cinert = s + L.cinert; float* crb = s + L.crb; float* cdof = s + L.cdof;
  float* cdofdot = s + L.cdofdot; float* cvel = s + L.cvel; float* cacc = s + L.cacc;
  float* H = s + L.H; float* invdiag = s + L.invdiag;
  // the joint-space inertia lives in global memory (2.5 KB per env, L2-resident): it is written once, copied
  // into H before each factorisation and read by symv only when the solver runs on all dofs
  float* Mq = dd.qM_packed.p + (size_t)w * dd.qM_packed.stride;
  float* qfrc_smooth = s + L.qfrc_smooth; float* qacc_smooth = s + L.qacc_smooth;
  float* qacc = s + L.qacc; float* Ma = s + L.Ma; float* grad = s + L.grad;
  float* Mv = s + L.Mv; float* qfrc_c = s + L.qfrc_c;
  float* tmpv = s + L.tmpv; float* actf = s + L.actf;

  // Consumer-visible kinematics (poses, cvel, derived velocities) are observable only after the last sub-step
  // of a decimation loop: the launches before it skip those stores (and the poses of non-colliding geoms).
  const bool emit = dd.emit != 0;
  bool ctrl_changed = false;
  // ---------------- phase 1: kinematics (lane per body, private walk down its ancestor chain) ----
  {
    const float* body_pos = MP(body_pos); const float* body_quat = MP(body_quat);
    const float* jnt_pos = MP(jnt_pos); const float* jnt_axis = MP(jnt_axis);
    const float* qpos0 = MP(qpos0);
    const float* body_ipos = MP(body_ipos);
    #pragma unroll 1
    for (int b = lane; b < nb; b += 32) {
      float pos[3] = {0.f, 0.f, 0.f}, quat[4] = {1.f, 0.f, 0.f, 0.f};
      int depth = m.body_depth[b];
      if (m.fastkin) {
        // one dependent load level per chain step: chain id -> 64-byte record (prefetched one ahead)
        const int* chain = m.body_chain + b * m.maxdepth;
        int c = depth > 0 ? chain[0] : 0;
        int cn = depth > 1 ? chain[1] : 0;
        float4 p0 = m.kinrec[4 * c], p1 = m.kinrec[4 * c + 1], p2 = m.kinrec[4 * c + 2], p3 = m.kinrec[4 * c + 3];
        #pragma unroll 1
        for (int k = 0; k < depth; k++) {
          const float4 r0 = p0, r1 = p1, r2 = p2, r3 = p3;
          c = cn;  // the next step's record and the id after it are in flight while this step computes
          cn = k + 2 < depth ? chain[k + 2] : 0;
          p0 = m.kinrec[4 * c]; p1 = m.kinrec[4 * c + 1]; p2 = m.kinrec[4 * c + 2]; p3 = m.kinrec[4 * c + 3];
          int tj = __float_as_int(r2.w), qa = __float_as_int(r3.w);
          int type = tj & 0xff, ja = tj >> 8;
          bool last = (k == depth - 1);
          if (type == JNT_FREE) {
            pos[0] = qpos[qa]; pos[1] = qpos[qa + 1]; pos[2] = qpos[qa + 2];
            quat[0] = qpos[qa + 3]; quat[1] = qpos[qa + 4]; quat[2] = qpos[qa + 5]; quat[3] = qpos[qa + 6];
            normalize4(quat);
            if (last) {
              xanchor[3 * ja] = pos[0]; xanchor[3 * ja + 1] = pos[1]; xanchor[3 * ja + 2] = pos[2];
              float ax0[3] = {r3.x, r3.y, r3.z}, ax[3];
              rotq(ax, quat, ax0);
              xaxis[3 * ja] = ax[0]; xaxis[3 * ja + 1] = ax[1]; xaxis[3 * ja + 2] = ax[2];
            }
          } else {
            float bp[3] = {r0.x, r0.y, r0.z}, bq[4] = {r1.x, r1.y, r1.z, r1.w}, t[3], q2[4];
            rotq(t, quat, bp);
            pos[0] += t[0]; pos[1] += t[1]; pos[2] += t[2];
            mulquat(q2, quat, bq);
            quat[0] = q2[0]; quat[1] = q2[1]; quat[2] = q2[2]; quat[3] = q2[3];
            if (type != 0xff) {
              float jp[3] = {r2.x, r2.y, r2.z}, jax[3] = {r3.x, r3.y, r3.z}, anchor[3], axis[3];
              rotq(anchor, quat, jp);
              anchor[0] += pos[0]; anchor[1] += pos[1]; anchor[2] += pos[2];
              rotq(axis, quat, jax);
              if (last) {
                xanchor[3 * ja] = anchor[0]; xanchor[3 * ja + 1] = anchor[1]; xanchor[3 * ja + 2] = anchor[2];
                xaxis[3 * ja] = axis[0]; xaxis[3 * ja + 1] = axis[1]; xaxis[3 * ja + 2] = axis[2];
              }
              float dq = qpos[qa] - r0.w;
              if (type == JNT_SLIDE) {
                pos[0] += axis[0] * dq; pos[1] += axis[1] * dq; pos[2] += axis[2] * dq;
              } else {
                float sn, cs;
                sincosf(0.5f * dq, &sn, &cs);
                float ql[4] = {cs, jax[0] * sn, jax[1] * sn, jax[2] * sn};
                mulquat(q2, quat, ql);
                quat[0] = q2[0]; quat[1] = q2[1]; quat[2] = q2[2]; quat[3] = q2[3];
                rotq(t, quat, jp);
                pos[0] = anchor[0] - t[0]; pos[1] = anchor[1] - t[1]; pos[2] = anchor[2] - t[2];
              }
            }
          }
          normalize4(quat);
        }
        depth = 0;  // generic walk below is skipped
      }
      #pragma unroll 1
      for (int k = 0; k < depth; k++) {
        int c = m.body_chain[b * m.maxdepth + k];
        int jn = m.body_jntnum[c], ja = m.body_jntadr[c];
        bool last = (k == depth - 1);
        if (jn == 1 && m.jnt_type[ja] == JNT_FREE) {
          int a = m.jnt_qposadr[ja];
          pos[0] = qpos[a]; pos[1] = qpos[a + 1]; pos[2] = qpos[a + 2];
          quat[0] = qpos[a + 3]; quat[1] = qpos[a + 4]; quat[2] = qpos[a + 5]; quat[3] = qpos[a + 6];
          normalize4(quat);
          if (last) {
            xanchor[3 * ja] = pos[0]; xanchor[3 * ja + 1] = pos[1]; xanchor[3 * ja + 2] = pos[2];
            float ax[3]; rotq(ax, quat, jnt_axis + 3 * ja);
            xaxis[3 * ja] = ax[0]; xaxis[3 * ja + 1] = ax[1]; xaxis[3 * ja + 2] = ax[2];
          }
        } else {
          float t[3], q2[4];
          rotq(t, quat, body_pos + 3 * c);
          pos[0] += t[0]; pos[1] += t[1]; pos[2] += t[2];
          mulquat(q2, quat, body_quat + 4 * c);
          quat[0] = q2[0]; quat[1] = q2[1]; quat[2] = q2[2]; quat[3] = q2[3];
          for (int j = ja; j < ja + jn; j++) {
            float anchor[3], axis[3];
            rotq(anchor, quat, jnt_pos + 3 * j);
            anchor[0] += pos[0]; anchor[1] += pos[1]; anchor[2] += pos[2];
            rotq(axis, quat, jnt_axis + 3 * j);
            if (last) {
              xanchor[3 * j] = anchor[0]; xanchor[3 * j + 1] = anchor[1]; xanchor[3 * j + 2] = anchor[2];
              xaxis[3 * j] = axis[0]; xaxis[3 * j + 1] = axis[1]; xaxis[3 * j + 2] = axis[2];
            }
            int qa = m.jnt_qposadr[j];
            float dq = qpos[qa] - qpos0[qa];
            if (m.jnt_type[j] == JNT_SLIDE) {
              pos[0] += axis[0] * dq; pos[1] += axis[1] * dq; pos[2] += axis[2] * dq;
            } else {
              float sn, cs;
              sincosf(0.5f * dq, &sn, &cs);
              float ql[4] = {cs, jnt_axis[3 * j] * sn, jnt_axis[3 * j + 1] * sn, jnt_axis[3 * j + 2] * sn};
              mulquat(q2, quat, ql);
              quat[0] = q2[0]; quat[1] = q2[1]; quat[2] = q2[2]; quat[3] = q2[3];
              rotq(t, quat, jnt_pos + 3 * j);
              pos[0] = anchor[0] - t[0]; pos[1] = anchor[1] - t[1]; pos[2] = anchor[2] - t[2];
            }
          }
        }
        normalize4(quat);
      }
      xpos[3 * b] = pos[0]; xpos[3 * b + 1] = pos[1]; xpos[3 * b + 2] = pos[2];
      xquat[4 * b] = quat[0]; xquat[4 * b + 1] = quat[1]; xquat[4 * b + 2] = quat[2]; xquat[4 * b + 3] = quat[3];
      float t[3], mat[9];
      rotq(t, quat, body_ipos + 3 * b);
      xipos[3 * b] = pos[0] + t[0]; xipos[3 * b + 1] = pos[1] + t[1]; xipos[3 * b + 2] = pos[2] + t[2];
      if (emit) {
        quat2mat(mat, quat);
        float* gx = dd.xmat.p + (size_t)w * dd.xmat.stride + 9 * b;
#pragma unroll
        for (int k = 0; k < 9; k++) gx[k] = mat[k];
      }
    }
  }
  __syncwarp();

  PHASE_MARK(1);
  PSYNC();
  // geom / site world poses -> global (and shared for collidable geoms)
  float* gpose = s + L.gpose;
  {
    const float* geom_pos = MP(geom_pos); const float* geom_quat = MP(geom_quat);
    const float* geom_rb = MP(geom_rbound); const float* geom_mar = MP(geom_margin);
    float* gxp = dd.geom_xpos.p + (size_t)w * dd.geom_xpos.stride;
    float* gxm = dd.geom_xmat.p + (size_t)w * dd.geom_xmat.stride;
    #pragma unroll 1
    for (int gi = lane; gi < m.nposegeom; gi += 32) {
      int g = m.posegeom[gi];
      int cs = m.geom_cslot[g];
      if (!emit && cs < 0) continue;  // a geom that cannot collide is posed for its consumers only
      int b = m.geom_bodyid[g];
      float p[3], q[4], mat[9];
      rotq(p, xquat + 4 * b, geom_pos + 3 * g);
      p[0] += xpos[3 * b]; p[1] += xpos[3 * b + 1]; p[2] += xpos[3 * b + 2];
      mulquat(q, xquat + 4 * b, geom_quat + 4 * g);
      quat2mat(mat, q);
      if (emit) {
        gxp[3 * g] = p[0]; gxp[3 * g + 1] = p[1]; gxp[3 * g + 2] = p[2];
#pragma unroll
        for (int k = 0; k < 9; k++) gxm[9 * g + k] = mat[k];
      }
      if (cs >= 0) {
        float* gp = gpose + GP * cs;
        gp[0] = p[0]; gp[1] = p[1]; gp[2] = p[2];
#pragma unroll
        for (int k = 0; k < 9; k++) gp[3 + k] = mat[k];
        gp[12] = geom_rb[g]; gp[13] = geom_mar[g];  // per-world values: the broadphase reads nothing else
      }
    }
    const float* site_pos = MP(site_pos); const float* site_quat = MP(site_quat);
    float* sxp = dd.site_xpos.p + (size_t)w * dd.site_xpos.stride;
    float* sxm = dd.site_xmat.p + (size_t)w * dd.site_xmat.stride;
    #pragma unroll 1
    for (int g = emit ? lane : m.nsite; g < m.nsite; g += 32) {
      int b = m.site_bodyid[g];
      float p[3], q[4], mat[9];
      rotq(p, xquat + 4 * b, site_pos + 3 * g);
      mulquat(q, xquat + 4 * b, site_quat + 4 * g);
      quat2mat(mat, q);
      sxp[3 * g] = p[0] + xpos[3 * b]; sxp[3 * g + 1] = p[1] + xpos[3 * b + 1]; sxp[3 * g + 2] = p[2] + xpos[3 * b + 2];
#pragma unroll
      for (int k = 0; k < 9; k++) sxm[9 * g + k] = mat[k];
    }
  }

  PHASE_MARK(2);
  PSYNC();
  // ---------------- phase 2: subtree com, spatial inertias, motion vectors -----------------------
  {
    const float* mass = MP(body_mass); const float* sub = MP(body_subtreemass);
    #pragma unroll 1
    for (int b = lane; b < nb; b += 32) {
      float acc[3] = {0.f, 0.f, 0.f};
      const unsigned long long desc = m.body_submask[b];
      FOR_BITS64(desc, d) {
        float md = mass[d];
        acc[0] += md * xipos[3 * d]; acc[1] += md * xipos[3 * d + 1]; acc[2] += md * xipos[3 * d + 2];
      }
      if (sub[b] < MINVAL) { acc[0] = xipos[3 * b]; acc[1] = xipos[3 * b + 1]; acc[2] = xipos[3 * b + 2]; }
      else { float inv = 1.f / sub[b]; acc[0] *= inv; acc[1] *= inv; acc[2] *= inv; }
      scom[3 * b] = acc[0]; scom[3 * b + 1] = acc[1]; scom[3 * b + 2] = acc[2];
    }
  }
  __syncwarp();
  // Internal reference point c0 = com of the moving bodies (those with a dof in their chain; static terrain
  // mass would drag the point far from the robot and cost fp32 digits); all cdof / cinert / cvel are expressed
  // about c0 (MuJoCo uses subtree_com[root]; results are identical, cvel is converted on output).
  float c0[3];
  {
    const float* mass = MP(body_mass);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, am = 0.f;
    #pragma unroll 1
    for (int b = lane; b < nb; b += 32) {
      if (m.body_dofmask[b] != 0ull) {
        float mb = mass[b];
        a0 += mb * xipos[3 * b]; a1 += mb * xipos[3 * b + 1]; a2 += mb * xipos[3 * b + 2]; am += mb;
      }
    }
    a0 = wsum(a0); a1 = wsum(a1); a2 = wsum(a2); am = wsum(am);
    if (am < MINVAL) { c0[0] = scom[0]; c0[1] = scom[1]; c0[2] = scom[2]; }
    else { float inv = 1.f / am; c0[0] = a0 * inv; c0[1] = a1 * inv; c0[2] = a2 * inv; }
  }
  if (emit) {  // body poses / coms leave now (coalesced); their shared-memory home is recycled after phase 4
    float* g0 = dd.xpos.p + (size_t)w * dd.xpos.stride;
    float* g1 = dd.xquat.p + (size_t)w * dd.xquat.stride;
    float* g2 = dd.xipos.p + (size_t)w * dd.xipos.stride;
    float* g3 = dd.subtree_com.p + (size_t)w * dd.subtree_com.stride;
    #pragma unroll 1
    for (int i = lane; i < 3 * nb; i += 32) { g0[i] = xpos[i]; g2[i] = xipos[i]; g3[i] = scom[i]; }
    #pragma unroll 1
    for (int i = lane; i < 4 * nb; i += 32) g1[i] = xquat[i];
  }
  {
    const float* mass = MP(body_mass); const float* inertia = MP(body_inertia);
    const float* body_iquat = MP(body_iquat);
    #pragma unroll 1
    for (int b = lane; b < nb; b += 32) {
      float q[4], mat[9], dif[3];
      mulquat(q, xquat + 4 * b, body_iquat + 4 * b);
      quat2mat(mat, q);
      dif[0] = xipos[3 * b] - c0[0]; dif[1] = xipos[3 * b + 1] - c0[1]; dif[2] = xipos[3 * b + 2] - c0[2];
      float ms = mass[b];
      const float* in = inertia + 3 * b;
      float t[9];
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++)
          t[3 * i + j] = mat[3 * i] * in[0] * mat[3 * j] + mat[3 * i + 1] * in[1] * mat[3 * j + 1] +
                         mat[3 * i + 2] * in[2] * mat[3 * j + 2];
      float* ci = cinert + SI * b;
      if (b == 0) {
#pragma unroll
        for (int k = 0; k < 10; k++) ci[k] = 0.f;
      } else {
        ci[0] = t[0] + ms * (dif[1] * dif[1] + dif[2] * dif[2]);
        ci[1] = t[4] + ms * (dif[0] * dif[0] + dif[2] * dif[2]);
        ci[2] = t[8] + ms * (dif[0] * dif[0] + dif[1] * dif[1]);
        ci[3] = t[1] - ms * dif[0] * dif[1];
        ci[4] = t[2] - ms * dif[0] * dif[2];
        ci[5] = t[5] - ms * dif[1] * dif[2];
        ci[6] = ms * dif[0]; ci[7] = ms * dif[1]; ci[8] = ms * dif[2]; ci[9] = ms;
      }
    }
    #pragma unroll 1
    for (int j = lane; j < njnt; j += 32) {
      int b = m.jnt_bodyid[j], da = m.jnt_dofadr[j], ty = m.jnt_type[j];
      float off[3] = {c0[0] - xanchor[3 * j], c0[1] - xanchor[3 * j + 1], c0[2] - xanchor[3 * j + 2]};
      if (ty == JNT_FREE) {
        float mat[9];
        quat2mat(mat, xquat + 4 * b);
        for (int k = 0; k < 3; k++) {
          float* c = cdof + SD * (da + k);
          c[0] = c[1] = c[2] = 0.f; c[3] = c[4] = c[5] = 0.f; c[3 + k] = 1.f;
          float ax[3] = {mat[k], mat[3 + k], mat[6 + k]};
          float* r = cdof + SD * (da + 3 + k);
          r[0] = ax[0]; r[1] = ax[1]; r[2] = ax[2];
          cross3(r + 3, ax, off);
        }
      } else if (ty == JNT_SLIDE) {
        float* c = cdof + SD * da;
        c[0] = c[1] = c[2] = 0.f;
        c[3] = xaxis[3 * j]; c[4] = xaxis[3 * j + 1]; c[5] = xaxis[3 * j + 2];
      } else {
        float* c = cdof + SD * da;
        c[0] = xaxis[3 * j]; c[1] = xaxis[3 * j + 1]; c[2] = xaxis[3 * j + 2];
        cross3(c + 3, xaxis + 3 * j, off);
      }
    }
  }
  __syncwarp();

  PHASE_MARK(3);
  PSYNC();
  // ---------------- phase 3: composite inertias -> joint-space inertia M (packed lower) ----------
  #pragma unroll 1
  for (int b = lane; b < nb; b += 32) {
    float acc[10];
#pragma unroll
    for (int k = 0; k < 10; k++) acc[k] = 0.f;
    const unsigned long long sub = m.body_submask[b] & ~1ull;
    FOR_BITS64(sub, d) {
#pragma unroll
      for (int k = 0; k < 10; k++) acc[k] += cinert[SI * d + k];
    }
#pragma unroll
    for (int k = 0; k < 10; k++) crb[SI * b + k] = acc[k];
  }
  #pragma unroll 1
  for (int i = lane; i < m.ntri; i += 32) Mq[i] = 0.f;
  __syncwarp();
  {
    const float* arm = MP(dof_armature);
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) {
      float buf[6];
      mul_inert_vec(buf, crb + SI * m.dof_bodyid[i], cdof + SD * i);
      Mq[tri(i, i)] = dot6(cdof + SD * i, buf) + arm[i];
      for (int j = m.dof_parentid[i]; j >= 0; j = m.dof_parentid[j]) Mq[tri(i, j)] = dot6(cdof + SD * j, buf);
    }
  }
  __syncwarp();

  PHASE_MARK(4);
  PSYNC();
  // ---------------- phase 4: velocities, bias forces, actuation, qfrc_smooth ----------------------
  #pragma unroll 1
  for (int b = lane; b < nb; b += 32) {
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, snap[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const unsigned long long mask = m.body_dofmask[b];
    int own0 = m.body_dofadr[b];
    FOR_BITS64(mask, d) {
      const float* c = cdof + SD * d;
      if (own0 >= 0 && d >= own0) {
        int j = m.dof_jntid[d];
        int off = d - m.jnt_dofadr[j];
        float* cd = cdofdot + SD * d;
        if (m.jnt_type[j] == JNT_FREE) {
          if (off < 3) { cd[0] = cd[1] = cd[2] = cd[3] = cd[4] = cd[5] = 0.f; }
          else {
            if (off == 3) { for (int k = 0; k < 6; k++) snap[k] = v[k]; }
            cross_motion(cd, snap, c);
          }
        } else cross_motion(cd, v, c);
      }
      float qd = qvel[d];
#pragma unroll
      for (int k = 0; k < 6; k++) v[k] += c[k] * qd;
    }
#pragma unroll
    for (int k = 0; k < 6; k++) cvel[SD * b + k] = v[k];
    if (emit) {
      // output cvel in MuJoCo's convention: linear part at subtree_com[root]
      int r = m.body_rootid[b];
      float dr[3] = {scom[3 * r] - c0[0], scom[3 * r + 1] - c0[1], scom[3 * r + 2] - c0[2]}, t[3];
      cross3(t, v, dr);
      float* gc = dd.cvel.p + (size_t)w * dd.cvel.stride + 6 * b;
      gc[0] = v[0]; gc[1] = v[1]; gc[2] = v[2];
      gc[3] = v[3] + t[0]; gc[4] = v[4] + t[1]; gc[5] = v[5] + t[2];
      // The quantities mjlab's EntityData derives from (xpos, subtree_com, cvel, xquat) with gathers and quaternion
      // kernels (entity/data.py:190-516), written here once per body: world velocity of the link origin and of
      // the body com, and in the link frame the linear / angular velocity, projected gravity and the heading.
      float dl[3] = {xpos[3 * b] - c0[0], xpos[3 * b + 1] - c0[1], xpos[3 * b + 2] - c0[2]}, tl[3];
      float dc[3] = {xipos[3 * b] - c0[0], xipos[3 * b + 1] - c0[1], xipos[3 * b + 2] - c0[2]}, tc[3];
      cross3(tl, v, dl);
      cross3(tc, v, dc);
      float lin[3] = {v[3] + tl[0], v[4] + tl[1], v[5] + tl[2]};
      float* lw = dd.link_vel_w.p + (size_t)w * dd.link_vel_w.stride + 6 * b;
      float* cw = dd.com_vel_w.p + (size_t)w * dd.com_vel_w.stride + 6 * b;
      float* lb = dd.link_state_b.p + (size_t)w * dd.link_state_b.stride + 10 * b;
      const float* q = xquat + 4 * b;
      float qi[4] = {q[0], -q[1], -q[2], -q[3]}, lbv[3], abv[3], gbv[3];
      const float down[3] = {0.f, 0.f, -1.f};
      rotq(lbv, qi, lin);
      rotq(abv, qi, v);
      rotq(gbv, qi, down);
#pragma unroll
      for (int k = 0; k < 3; k++) {
        lw[k] = lin[k]; lw[3 + k] = v[k];
        cw[k] = v[3 + k] + tc[k]; cw[3 + k] = v[k];
        lb[k] = lbv[k]; lb[3 + k] = abv[k]; lb[6 + k] = gbv[k];
      }
      lb[9] = atan2f(2.f * (q[1] * q[2] + q[0] * q[3]), 1.f - 2.f * (q[2] * q[2] + q[3] * q[3]));
    }
  }
  __syncwarp();
  #pragma unroll 1
  for (int b = lane; b < nb; b += 32) {
    float a[6] = {0.f, 0.f, 0.f, -m.gravity[0], -m.gravity[1], -m.gravity[2]};
    const unsigned long long mask = m.body_dofmask[b];
    FOR_BITS64(mask, d) {
      float qd = qvel[d];
#pragma unroll
      for (int k = 0; k < 6; k++) a[k] += cdofdot[SD * d + k] * qd;
    }
    float t[6], t1[6], t2[6];
    mul_inert_vec(t, cinert + SI * b, cvel + SD * b);
    cross_force(t1, cvel + SD * b, t);
    mul_inert_vec(t2, cinert + SI * b, a);
    // net external wrench on the body about c0: xfrc_applied (force at xipos) minus bias wrench
    const float* xf = xfrc + 6 * b;
    float arm[3] = {xipos[3 * b] - c0[0], xipos[3 * b + 1] - c0[1], xipos[3 * b + 2] - c0[2]}, tq[3];
    cross3(tq, arm, xf);
    float* cf = cacc + SD * b;  // region reused: [bias wrench]
    float* cx = crb + SD * b;   // region reused: [applied wrench]
    if (b == 0) {
#pragma unroll
      for (int k = 0; k < 6; k++) { cf[k] = 0.f; cx[k] = 0.f; }
    } else {
#pragma unroll
      for (int k = 0; k < 6; k++) cf[k] = t2[k] + t1[k];
      cx[0] = tq[0] + xf[3]; cx[1] = tq[1] + xf[4]; cx[2] = tq[2] + xf[5];
      cx[3] = xf[0]; cx[4] = xf[1]; cx[5] = xf[2];
    }
  }
  #pragma unroll 1
  for (int i = lane; i < nv; i += 32) tmpv[i] = 0.f;  // qfrc_actuator
  __syncwarp();
  {
    const float* gp = MP(actuator_gainprm); const float* bp = MP(actuator_biasprm);
    const float* cr = MP(actuator_ctrlrange); const float* fr = MP(actuator_forcerange);
    const float* gear = MP(actuator_gear);
    float* gaf = dd.actuator_force.p + (size_t)w * dd.actuator_force.stride;
    float* cprev = dd.ctrl_prev.p + (size_t)w * dd.ctrl_prev.stride;
    bool cdiff = false;
    #pragma unroll 1
    for (int a = lane; a < nu; a += 32) {
      int j = m.actuator_trnid[a];
      float g = gear[a];
      float len = qpos[m.jnt_qposadr[j]] * g, vel = qvel[m.jnt_dofadr[j]] * g;
      float c = ctrl[a];
      if (STEP) { cdiff |= c != cprev[a]; cprev[a] = c; }
      if (m.actuator_ctrllimited[a]) c = fminf(fmaxf(c, cr[2 * a]), cr[2 * a + 1]);
      float f = gp[10 * a] * c + bp[10 * a] + bp[10 * a + 1] * len + bp[10 * a + 2] * vel;
      if (m.actuator_forcelimited[a]) f = fminf(fmaxf(f, fr[2 * a]), fr[2 * a + 1]);
      actf[a] = f;
      gaf[a] = f;
      atomicAdd(&tmpv[m.jnt_dofadr[j]], g * f);  // one actuator per dof in practice; exact either way
    }
    ctrl_changed = __any_sync(FULL, cdiff);
  }
  __syncwarp();
  {
    const float* damp = MP(dof_damping); const float* stiff = MP(jnt_stiffness);
    const float* qpos0 = MP(qpos0);
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) {
      float sb[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, sx[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const unsigned long long sub = m.dof_bodymask[i];
      FOR_BITS64(sub, b) {
#pragma unroll
        for (int k = 0; k < 6; k++) { sb[k] += cacc[SD * b + k]; sx[k] += crb[SD * b + k]; }
      }
      float bias = dot6(cdof + SD * i, sb);
      float passive = -damp[i] * qvel[i];
      int j = m.dof_jntid[i];
      if (m.jnt_type[j] != JNT_FREE && stiff[j] != 0.f)
        passive -= stiff[j] * (qpos[m.jnt_qposadr[j]] - qpos0[m.jnt_qposadr[j]]);
      float fs = passive - bias + qfrc_applied[i] + tmpv[i] + dot6(cdof + SD * i, sx);
      qfrc_smooth[i] = fs;
      qacc_smooth[i] = fs;
      if (m.debug & 1) {
        dd.qfrc_bias.p[(size_t)w * dd.qfrc_bias.stride + i] = bias;
        dd.qfrc_smooth.p[(size_t)w * dd.qfrc_smooth.stride + i] = fs;
      }
    }
  }
  __syncwarp();
  if (m.debug & 1) {
    float* gM = dd.qM.p + (size_t)w * dd.qM.stride;
    #pragma unroll 1
    for (int p = lane; p < nv * nv; p += 32) {
      int i = p / nv, j = p % nv;
      gM[p] = i >= j ? Mq[tri(i, j)] : Mq[tri(j, i)];
    }
  }

  PHASE_MARK(5);
  PSYNC();
  // ---------------- phase 5: collision (static pair table, bounding-sphere filter, primitives) ----
  float* con = s + L.contacts;   // overlays the smooth-only regions (cinert, crb, cdofdot, cacc, ...)
  float* lim = s + L.limits;
  int* gstart = (int*)(s + L.gstart);
  int ncon = 0, overflow = 0;
  {
    int* pairlist = (int*)(s + L.pairlist);
    const float* gmar = MP(geom_margin);
    int ncand = 0;
    // pairs without a height field: the flat table (all pairs when the model has no field)
    const int* nhp = CVX ? m.nh_pairs : nullptr;
    const int np = CVX ? m.n_nhpair : m.npair;
    unsigned pw_next = lane < np ? m.pair_word[nhp ? nhp[lane] : lane] : 0u;
    #pragma unroll 1
    for (int p0 = 0; p0 < np; p0 += 32) {
      const int k = p0 + lane;
      const int p = (nhp && k < np) ? nhp[k] : k;
      bool hit = false;
      const unsigned pw = pw_next;  // slot1 | slot2 << 12 | (geom1 is a height field) << 30 | (geom1 is a plane) << 31
      if (k + 32 < np) pw_next = m.pair_word[nhp ? nhp[k + 32] : k + 32];  // in flight during this batch
      if (k < np) {
        const float* a = gpose + GP * (pw & 0xfffu);
        const float* b = gpose + GP * ((pw >> 12) & 0xfffu);
        float margin = fmaxf(a[13], b[13]);
        float dif[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
        if (pw >> 31) {
          float n[3] = {a[3 + 2], a[3 + 5], a[3 + 8]};
          hit = dot3(dif, n) <= margin + b[12];
        } else {
          float bound = margin + a[12] + b[12];
          hit = dot3(dif, dif) <= bound * bound;
        }
      }
      unsigned bal = __ballot_sync(FULL, hit);
      if (hit) {
        int slot = ncand + __popc(bal & ((1u << lane) - 1u));
        if (slot < L.maxpair) pairlist[slot] = p;
      }
      ncand += __popc(bal);
    }
    if (CVX && m.nhf > 0) {
      // height-field pairs, field by field.  A terrain is a grid of fields and the robot stands on one or two
      // of them: first the fields whose box meets the sphere around all the geoms that can touch a field, then
      // only their pairs, each with the exact test (the geom's bounding sphere against the field's box - the
      // fields' own bounding spheres all contain the robot).  The candidates are put back in pair-table order.
      float lo[3] = {1e30f, 1e30f, 1e30f}, hi[3] = {-1e30f, -1e30f, -1e30f};
      #pragma unroll 1
      for (int q = lane; q < m.nhfd; q += 32) {
        const float* c = gpose + GP * m.hfd_slot[q];
        const float r = c[12] + c[13];
        for (int k = 0; k < 3; k++) { lo[k] = fminf(lo[k], c[k] - r); hi[k] = fmaxf(hi[k], c[k] + r); }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
        for (int k = 0; k < 3; k++) {
          lo[k] = fminf(lo[k], __shfl_xor_sync(FULL, lo[k], o));
          hi[k] = fmaxf(hi[k], __shfl_xor_sync(FULL, hi[k], o));
        }
      const float cw[3] = {0.5f * (lo[0] + hi[0]), 0.5f * (lo[1] + hi[1]), 0.5f * (lo[2] + hi[2])};
      const float ext[3] = {hi[0] - cw[0], hi[1] - cw[1], hi[2] - cw[2]};
      const float Rw = sqrtf(dot3(ext, ext)) * 1.0001f + 1e-6f;
      const int nbefore = ncand;
      int nnear = 0;
      #pragma unroll 1
      for (int h0 = 0; h0 < m.nhf; h0 += 32) {
        const int h = h0 + lane;
        bool near = false;
        if (h < m.nhf) {
          const float* a = cpose(gpose, m, m.hfl_slot[h]);
          const float4 hb = m.hfl_box[h];
          const float reach = Rw + gmar[m.hfl_geom[h]];
          const float dif[3] = {cw[0] - a[0], cw[1] - a[1], cw[2] - a[2]};
          const float lx = a[3] * dif[0] + a[6] * dif[1] + a[9] * dif[2], ly = a[4] * dif[0] + a[7] * dif[1] + a[10] * dif[2];
          const float lz = a[5] * dif[0] + a[8] * dif[1] + a[11] * dif[2];
          near = fabsf(lx) <= hb.x + reach && fabsf(ly) <= hb.y + reach && lz - reach <= hb.z && lz + reach >= -hb.w;
        }
        unsigned nm = __ballot_sync(FULL, near);
        nnear += __popc(nm);
        #pragma unroll 1
        while (nm) {
          const int hh = h0 + __ffs((int)nm) - 1;
          nm &= nm - 1u;
          const float* a = cpose(gpose, m, m.hfl_slot[hh]);
          const float4 hb = m.hfl_box[hh];
          const float amar = gmar[m.hfl_geom[hh]];
          const int en = m.hfl_start[hh + 1];
          #pragma unroll 1
          for (int k0 = m.hfl_start[hh]; k0 < en; k0 += 32) {
            const int k = k0 + lane;
            bool hit = false;
            int p = 0;
            if (k < en) {
              p = m.hfl_pairs[k];
              const float* b = gpose + GP * ((m.pair_word[p] >> 12) & 0xfffu);
              const float reach = fmaxf(amar, b[13]) + b[12];
              const float dif[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
              const float lx = a[3] * dif[0] + a[6] * dif[1] + a[9] * dif[2], ly = a[4] * dif[0] + a[7] * dif[1] + a[10] * dif[2];
              const float lz = a[5] * dif[0] + a[8] * dif[1] + a[11] * dif[2];
              hit = fabsf(lx) <= hb.x + reach && fabsf(ly) <= hb.y + reach && lz - reach <= hb.z && lz + reach >= -hb.w;
            }
            unsigned bal = __ballot_sync(FULL, hit);
            if (hit) {
              int slot = ncand + __popc(bal & ((1u << lane) - 1u));
              if (slot < L.maxpair) pairlist[slot] = p;
            }
            ncand += __popc(bal);
          }
        }
      }
      const int nn = min(ncand, L.maxpair);
      if (nn > nbefore && (nnear > 1 || nbefore > 0)) {
        // rank sort (pair indices are distinct) through the scratch of hfield_lanes
        int* tmp = (int*)(s + L.gV);
        __syncwarp();
        #pragma unroll 1
        for (int i = lane; i < nn; i += 32) {
          const int v = pairlist[i];
          int rank = 0;
          for (int k = 0; k < nn; k++) rank += pairlist[k] < v ? 1 : 0;
          tmp[rank] = v;
        }
        __syncwarp();
        for (int i = lane; i < nn; i += 32) pairlist[i] = tmp[i];
        __syncwarp();
      }
    }
    PHASE_MARK(17);  // pair-table broadphase
    const float* gsize = MP(geom_size);
    if (m.nstatic > 0) {
      // grid-static candidates: lane = dynamic geom, visiting the cells under its bounding sphere.  Two passes
      // (count, then write at the scanned offset) keep the list in (geom, ix, iy, item) order, as the oracle's.
      #pragma unroll 1
      for (int q0 = 0; q0 < m.ndyn; q0 += 32) {
        int q = q0 + lane;
        int cnt = 0, wr = 0, tot = 0;
        #pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
          if (q < m.ndyn) {
            int g = m.dyn_cgeom[q];
            const float* c = gpose + GP * m.geom_cslot[g];
            float r = c[12], mg = c[13];
            int ct = m.geom_contype[g], ca = m.geom_conaffinity[g];
            // (cell range widened by 1e-4 cell: never narrower than the exact range, whatever the rounding of the
            // fast division; a cell visited in excess only adds candidates that the reach test below rejects)
            const float icell = 1.f / m.grid_cell;
            int ix0 = max((int)floorf((c[0] - r - m.grid_x0) * icell - 1e-4f), 0);
            int ix1 = min((int)floorf((c[0] + r - m.grid_x0) * icell + 1e-4f), m.grid_nx - 1);
            int iy0 = max((int)floorf((c[1] - r - m.grid_y0) * icell - 1e-4f), 0);
            int iy1 = min((int)floorf((c[1] + r - m.grid_y0) * icell + 1e-4f), m.grid_ny - 1);
            #pragma unroll 1
            for (int ix = ix0; ix <= ix1; ix++) {
              #pragma unroll 1
              for (int iy = iy0; iy <= iy1; iy++) {
                int cell = ix * m.grid_ny + iy;
                int it1 = m.grid_start[cell + 1];
                #pragma unroll 1
                for (int it = m.grid_start[cell]; it < it1; it++) {
                  int k = m.grid_items[it];
                  if (ix != max(m.static_cell0[2 * k], ix0) || iy != max(m.static_cell0[2 * k + 1], iy0)) continue;
                  int sg = m.static_geom[k];
                  if (!((ct & m.geom_conaffinity[sg]) || (m.geom_contype[sg] & ca))) continue;
                  // conservative reach test (never rejects a pair the narrowphase would accept)
                  const float* sp = m.static_pose + 16 * (size_t)k;
                  float reach = r + fmaxf(mg, gmar[sg]);
                  float d2;
                  if (m.geom_type[sg] == G_BOX) d2 = point_box_dist2(c, sp, gsize + 3 * sg);
                  else {
                    float dif[3] = {c[0] - sp[0], c[1] - sp[1], c[2] - sp[2]};
                    d2 = dot3(dif, dif); reach += sp[12];
                  }
                  if (d2 > reach * reach * 1.0001f + 1e-12f) continue;
                  if (pass == 0) cnt++;
                  else { if (wr < L.maxpair) pairlist[wr] = (int)(0x80000000u | ((unsigned)q << 20) | (unsigned)k); wr++; }
                }
              }
            }
          }
          if (pass == 1 && cnt > 1) {
            // the lane's candidates in ascending static index: the order no longer depends on the cell a
            // candidate was found in (same rule in the oracle)
            const int lo = wr - cnt, hi = min(wr, L.maxpair);
            #pragma unroll 1
            for (int a = lo + 1; a < hi; a++) {
              int v = pairlist[a], b = a - 1;
              while (b >= lo && (unsigned)pairlist[b] > (unsigned)v) { pairlist[b + 1] = pairlist[b]; b--; }
              pairlist[b + 1] = v;
            }
          }
          if (pass == 0) {
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              int t = __shfl_up_sync(FULL, incl, o);
              if (lane >= o) incl += t;
            }
            wr = ncand + incl - cnt;
            tot = __shfl_sync(FULL, incl, 31);
          }
        }
        ncand += tot;
      }
    }
    PHASE_MARK(18);  // grid broadphase
    if (ncand > L.maxpair) { ncand = L.maxpair; overflow = 1; }
    __syncwarp();
    const float* ggap = MP(geom_gap);
    const float* gfri = MP(geom_friction); const float* gsolref = MP(geom_solref);
    const float* gsolimp = MP(geom_solimp); const float* gsolmix = MP(geom_solmix);
    const float* inv = MP(body_invweight0);
    float* g_dist = dd.contact_dist.p + (size_t)w * dd.contact_dist.stride;
    float* g_pos = dd.contact_pos.p + (size_t)w * dd.contact_pos.stride;
    float* g_frame = dd.contact_frame.p + (size_t)w * dd.contact_frame.stride;
    int* g_geom = dd.contact_geom.p + (size_t)w * dd.contact_geom.stride;
    #pragma unroll 1
    for (int q0 = 0; q0 < ncand; q0 += 32) {
      int qi = q0 + lane;
      RawCon rc[8];
      int n = 0, g1 = 0, g2 = 0;
      float margin = 0.f;
      bool hf = false;
      const float *hfa = nullptr, *hfb = nullptr;
      if (qi < ncand) {
        int p = pairlist[qi];
        const float *a, *b;
        if (p >= 0) {
          g1 = m.pair_geom1[p]; g2 = m.pair_geom2[p];
          a = cpose(gpose, m, m.geom_cslot[g1]);
          b = gpose + GP * m.geom_cslot[g2];
        } else {  // grid-static candidate: (dynamic geom, static geom), ordered by (type, id)
          int k = p & 0xfffff;
          g1 = m.dyn_cgeom[(p >> 20) & 0x7ff]; g2 = m.static_geom[k];
          a = gpose + GP * m.geom_cslot[g1];
          b = m.static_pose + 16 * (size_t)k;
          int ta = m.geom_type[g1], tb = m.geom_type[g2];
          if (ta > tb || (ta == tb && g1 > g2)) {
            int tg = g1; g1 = g2; g2 = tg;
            const float* tp = a; a = b; b = tp;
          }
        }
        int t1 = m.geom_type[g1], t2 = m.geom_type[g2];
        margin = fmaxf(gmar[g1], gmar[g2]);
        const float* s1 = gsize + 3 * g1; const float* s2 = gsize + 3 * g2;
        if (CVX && t1 == G_HFIELD) {
          hf = t2 != G_HFIELD; hfa = a; hfb = b;
        } else if (CVX && (t2 == G_MESH || ((1u << t1 | 1u << t2) & (1u << G_ELLIPSOID | 1u << G_CYLINDER)))) {
          n = convex_narrowphase(rc, margin, m, g1, g2, a, b, s1, s2);
        } else if (t1 == G_PLANE) {
          float pn[3] = {a[3 + 2], a[3 + 5], a[3 + 8]};
          if (t2 == G_SPHERE) n = plane_sphere(rc[0], margin, a, pn, b, s2[0]);
          else if (t2 == G_CAPSULE) {
            float ax[3] = {b[3 + 2], b[3 + 5], b[3 + 8]}, e[3];
            e[0] = b[0] + ax[0] * s2[1]; e[1] = b[1] + ax[1] * s2[1]; e[2] = b[2] + ax[2] * s2[1];
            if (plane_sphere(rc[n], margin, a, pn, e, s2[0])) { rc[n].yh[0] = ax[0]; rc[n].yh[1] = ax[1]; rc[n].yh[2] = ax[2]; n++; }
            e[0] = b[0] - ax[0] * s2[1]; e[1] = b[1] - ax[1] * s2[1]; e[2] = b[2] - ax[2] * s2[1];
            if (plane_sphere(rc[n], margin, a, pn, e, s2[0])) { rc[n].yh[0] = ax[0]; rc[n].yh[1] = ax[1]; rc[n].yh[2] = ax[2]; n++; }
          } else if (t2 == G_BOX) {
            float dif[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
            float dist = dot3(dif, pn);
            for (int i = 0; i < 8 && n < 4; i++) {
              float v[3] = {(i & 1) ? s2[0] : -s2[0], (i & 2) ? s2[1] : -s2[1], (i & 4) ? s2[2] : -s2[2]};
              float cr[3] = {b[3] * v[0] + b[4] * v[1] + b[5] * v[2], b[6] * v[0] + b[7] * v[1] + b[8] * v[2],
                             b[9] * v[0] + b[10] * v[1] + b[11] * v[2]};
              float ld = dot3(pn, cr);
              if (dist + ld > margin || ld > 0.f) continue;
              rc[n].dist = dist + ld;
              for (int k = 0; k < 3; k++) {
                rc[n].pos[k] = b[k] + cr[k] - pn[k] * (0.5f * rc[n].dist);
                rc[n].n[k] = pn[k]; rc[n].yh[k] = 0.f;
              }
              n++;
            }
          }
        } else if (t1 == G_SPHERE && t2 == G_SPHERE) {
          n = sphere_sphere(rc[0], margin, a, s1[0], b, s2[0]);
        } else if (t1 == G_SPHERE && t2 == G_CAPSULE) {
          float ax[3] = {b[3 + 2], b[3 + 5], b[3 + 8]};
          float vec[3] = {a[0] - b[0], a[1] - b[1], a[2] - b[2]};
          float x = fminf(fmaxf(dot3(ax, vec), -s2[1]), s2[1]);
          float pt[3] = {b[0] + ax[0] * x, b[1] + ax[1] * x, b[2] + ax[2] * x};
          n = sphere_sphere(rc[0], margin, a, s1[0], pt, s2[0]);
        } else if (t2 == G_BOX) {
          if (t1 == G_SPHERE) n = sphere_box(rc[0], margin, a, s1[0], b, s2);
          else if (t1 == G_CAPSULE) n = capsule_box(rc, margin, a, s1, b, s2);
          else if (t1 == G_BOX) n = box_box(rc, margin, a, s1, b, s2);
        } else if (t1 == G_CAPSULE && t2 == G_CAPSULE) {
          float a1[3] = {a[3 + 2], a[3 + 5], a[3 + 8]}, a2[3] = {b[3 + 2], b[3 + 5], b[3 + 8]};
          float dif[3] = {a[0] - b[0], a[1] - b[1], a[2] - b[2]};
          float ma = dot3(a1, a1), mb = -dot3(a1, a2), mc = dot3(a2, a2);
          float u = -dot3(a1, dif), v = dot3(a2, dif);
          float det = ma * mc - mb * mb;
          float len1 = s1[1], len2 = s2[1];
          // parallel axes: MuJoCo tests |det| < 1e-15 in double; in fp32 det = sin^2(angle) of exactly parallel
          // unit axes evaluates to ~1e-7, so the test is made at 1e-6 (angles below 0.06 degrees)
          if (fabsf(det) >= 1e-6f) {
            float x1 = (mc * u - mb * v) / det, x2 = (ma * v - mb * u) / det;
            if (x1 > len1) { x1 = len1; x2 = (v - mb * len1) / mc; }
            else if (x1 < -len1) { x1 = -len1; x2 = (v + mb * len1) / mc; }
            if (x2 > len2) { x2 = len2; x1 = (u - mb * len2) / ma; }
            else if (x2 < -len2) { x2 = -len2; x1 = (u + mb * len2) / ma; }
            x1 = fminf(fmaxf(x1, -len1), len1);
            float v1[3] = {a[0] + a1[0] * x1, a[1] + a1[1] * x1, a[2] + a1[2] * x1};
            float v2[3] = {b[0] + a2[0] * x2, b[1] + a2[1] * x2, b[2] + a2[2] * x2};
            n = sphere_sphere(rc[0], margin, v1, s1[0], v2, s2[0]);
          } else {
            for (int e = 0; e < 2; e++) {
              float x1 = e ? -len1 : len1;
              float v1[3] = {a[0] + a1[0] * x1, a[1] + a1[1] * x1, a[2] + a1[2] * x1};
              float t[3] = {v1[0] - b[0], v1[1] - b[1], v1[2] - b[2]};
              float x2 = fminf(fmaxf(dot3(a2, t), -len2), len2);
              float v2[3] = {b[0] + a2[0] * x2, b[1] + a2[1] * x2, b[2] + a2[2] * x2};
              n += sphere_sphere(rc[n], margin, v1, s1[0], v2, s2[0]);
            }
          }
        }
      }
      PHASE_MARK(19);  // primitive narrowphase
      if (CVX) {
        if (__any_sync(FULL, hf)) {
          int nh = hfield_lanes(rc, hf, margin, m, gsize, g1, g2, hfa, hfb, (int*)(s + L.gV), lane);
          if (hf) n = nh;
        }
      }
      PHASE_MARK(20);  // height-field pairs (total of 21-23 + merge)
      // deterministic compaction in (pair order, contact index) order
      int incl = n;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
      }
      int base = ncon + incl - n;
      int tot = __shfl_sync(FULL, incl, 31);
      if (n > 0) {
        // contact parameters (mj_contactParam)
        int condim; float fri0, solref[2], solimp[5];
        int pr1 = m.geom_priority[g1], pr2 = m.geom_priority[g2];
        if (pr1 != pr2) {
          int g = pr1 > pr2 ? g1 : g2;
          condim = m.geom_condim[g]; fri0 = gfri[3 * g];
          solref[0] = gsolref[2 * g]; solref[1] = gsolref[2 * g + 1];
          for (int k = 0; k < 5; k++) solimp[k] = gsolimp[5 * g + k];
        } else {
          condim = max(m.geom_condim[g1], m.geom_condim[g2]);
          fri0 = fmaxf(gfri[3 * g1], gfri[3 * g2]);
          float m1 = gsolmix[g1], m2 = gsolmix[g2], mix;
          if (m1 >= MINVAL && m2 >= MINVAL) mix = m1 / (m1 + m2);
          else if (m1 < MINVAL && m2 < MINVAL) mix = 0.5f;
          else mix = m1 < MINVAL ? 0.f : 1.f;
          if (gsolref[2 * g1] > 0.f && gsolref[2 * g2] > 0.f) {
            solref[0] = mix * gsolref[2 * g1] + (1.f - mix) * gsolref[2 * g2];
            solref[1] = mix * gsolref[2 * g1 + 1] + (1.f - mix) * gsolref[2 * g2 + 1];
          } else {
            solref[0] = fminf(gsolref[2 * g1], gsolref[2 * g2]);
            solref[1] = fminf(gsolref[2 * g1 + 1], gsolref[2 * g2 + 1]);
          }
          for (int k = 0; k < 5; k++) solimp[k] = mix * gsolimp[5 * g1 + k] + (1.f - mix) * gsolimp[5 * g2 + k];
        }
        float mu = fmaxf(fri0, MINMU);
        float incm = margin - fmaxf(ggap[g1], ggap[g2]);
        int b1 = m.geom_bodyid[g1], b2 = m.geom_bodyid[g2];
        // impedance / reference parameters (mj_makeImpedance; pos = dist, margin = includemargin)
        float dmin = fminf(fmaxf(solimp[0], MINIMP), MAXIMP), dmax = fminf(fmaxf(solimp[1], MINIMP), MAXIMP);
        float width = fmaxf(solimp[2], MINVAL), mid = fminf(fmaxf(solimp[3], MINIMP), MAXIMP);
        float power = fmaxf(solimp[4], 1.f);
        float K, B;
        if (solref[0] > 0.f) {
          float tc = fmaxf(solref[0], 2.f * m.timestep), dr = solref[1];
          K = 1.f / fmaxf(MINVAL, dmax * dmax * tc * tc * dr * dr);
          B = 2.f / fmaxf(MINVAL, dmax * tc);
        } else { K = -solref[0] / (dmax * dmax); B = -solref[1] / dmax; }
        float tran = inv[2 * b1] + inv[2 * b2];
        #pragma unroll 1
        for (int i = 0; i < n; i++) {
          int c = base + i;
          if (c >= MC) break;
          float fr[9] = {rc[i].n[0], rc[i].n[1], rc[i].n[2], rc[i].yh[0], rc[i].yh[1], rc[i].yh[2], 0.f, 0.f, 0.f};
          make_frame(fr);
          g_dist[c] = rc[i].dist;
          for (int k = 0; k < 3; k++) g_pos[3 * c + k] = rc[i].pos[k];
          for (int k = 0; k < 9; k++) g_frame[9 * c + k] = fr[k];
          g_geom[2 * c] = g1; g_geom[2 * c + 1] = g2;
          float r[3] = {rc[i].pos[0] - c0[0], rc[i].pos[1] - c0[1], rc[i].pos[2] - c0[2]};
          for (int mm = 0; mm < 3; mm++) {
            float t[3];
            cross3(t, r, fr + 3 * mm);
            con[(CS0 + 6 * mm + 0) * MC + c] = t[0]; con[(CS0 + 6 * mm + 1) * MC + c] = t[1];
            con[(CS0 + 6 * mm + 2) * MC + c] = t[2];
            con[(CS0 + 6 * mm + 3) * MC + c] = fr[3 * mm]; con[(CS0 + 6 * mm + 4) * MC + c] = fr[3 * mm + 1];
            con[(CS0 + 6 * mm + 5) * MC + c] = fr[3 * mm + 2];
          }
          float x = fabsf(rc[i].dist - incm) / width, imp;
          if (x >= 1.f) imp = dmax;
          else if (x <= 0.f) imp = dmin;
          else {
            float y;
            if (power == 1.f) y = x;
            else if (x <= mid) y = __powf(x, power) / __powf(mid, power - 1.f);
            else y = 1.f - __powf(1.f - x, power) / __powf(1.f - mid, power - 1.f);
            imp = dmin + y * (dmax - dmin);
          }
          // R: frictionless -> (1-imp)/imp*tran ; pyramidal -> 2 mu'^2 * (1-imp)/imp*tran*(1+mu^2)
          float diag = condim == 1 ? tran : tran * (1.f + mu * mu);
          float R = fmaxf(MINVAL, (1.f - imp) * diag / imp);
          if (condim > 1) { float mup = mu * rsqrtf(m.impratio); R = fmaxf(MINVAL, 2.f * mup * mup * R); }
          bool excluded = !(rc[i].dist < incm);
          con[CDIST * MC + c] = rc[i].dist;
          con[CMU * MC + c] = mu;
          con[CD * MC + c] = excluded ? 0.f : 1.f / R;
          con[CKI * MC + c] = K * imp * (rc[i].dist - incm);
          con[CB * MC + c] = B;
          ((int*)con)[CINFO * MC + c] = b1 | (b2 << 8) | ((excluded ? 0 : condim) << 16);
        }
      }
      ncon += tot;
    }
    if (ncon > MC) { ncon = MC; overflow = 1; }
  }
  __syncwarp();

  PHASE_MARK(6);
  PSYNC();
  // ---------------- phase 6: joint-limit rows, body-pair groups ----------------------------------
  int nlim = 0;
  {
    const float* range = MP(jnt_range); const float* jmar = MP(jnt_margin);
    const float* jsolref = MP(jnt_solref); const float* jsolimp = MP(jnt_solimp);
    const float* dinv = MP(dof_invweight0);
    #pragma unroll 1
    for (int j0 = 0; j0 < njnt; j0 += 32) {
      int j = j0 + lane;
      int side = 0; float dist = 0.f;
      if (j < njnt && m.jnt_limited[j] && m.jnt_type[j] != JNT_FREE) {
        float value = qpos[m.jnt_qposadr[j]];
        float dlo = value - range[2 * j], dhi = range[2 * j + 1] - value;
        if (dlo < jmar[j]) { side = -1; dist = dlo; }
        else if (dhi < jmar[j]) { side = 1; dist = dhi; }
        // (both sides active at once needs range width < 2*margin; not representable here)
      }
      unsigned bal = __ballot_sync(FULL, side != 0);
      if (side != 0) {
        int r = nlim + __popc(bal & ((1u << lane) - 1u));
        if (r < NLC) {
          int dof = m.jnt_dofadr[j];
          const float* si = jsolimp + 5 * j;
          float dmin = fminf(fmaxf(si[0], MINIMP), MAXIMP), dmax = fminf(fmaxf(si[1], MINIMP), MAXIMP);
          float width = fmaxf(si[2], MINVAL), mid = fminf(fmaxf(si[3], MINIMP), MAXIMP), power = fmaxf(si[4], 1.f);
          float x = fabsf(dist - jmar[j]) / width, imp;
          if (x >= 1.f) imp = dmax;
          else if (x <= 0.f) imp = dmin;
          else {
            float y;
            if (power == 1.f) y = x;
            else if (x <= mid) y = __powf(x, power) / __powf(mid, power - 1.f);
            else y = 1.f - __powf(1.f - x, power) / __powf(1.f - mid, power - 1.f);
            imp = dmin + y * (dmax - dmin);
          }
          float K, B;
          if (jsolref[2 * j] > 0.f) {
            float tc = fmaxf(jsolref[2 * j], 2.f * m.timestep), dr = jsolref[2 * j + 1];
            K = 1.f / fmaxf(MINVAL, dmax * dmax * tc * tc * dr * dr);
            B = 2.f / fmaxf(MINVAL, dmax * tc);
          } else { K = -jsolref[2 * j] / (dmax * dmax); B = -jsolref[2 * j + 1] / dmax; }
          float R = fmaxf(MINVAL, (1.f - imp) * dinv[dof] / imp);
          float Jd = -(float)side;
          float vel = Jd * qvel[dof];
          ((int*)lim)[LINFO * NLC + r] = dof | ((side > 0 ? 1 : 0) << 16);
          lim[LD * NLC + r] = 1.f / R;
          lim[LJAR * NLC + r] = B * vel + K * imp * (dist - jmar[j]);  // -aref (J a is added by the solver)
        }
      }
      nlim += __popc(bal);
    }
    if (nlim > NLC) { nlim = NLC; overflow = 1; }
  }
  // groups = maximal runs of contacts with the same (b1,b2); group dof set = chain(b1) xor chain(b2)
  int ngroup = 0;
  #pragma unroll 1
  for (int c00 = 0; c00 < ncon; c00 += 32) {
    int c = c00 + lane;
    bool start = false;
    int key = 0;
    if (c < ncon) {
      key = ((int*)con)[CINFO * MC + c] & 0xffff;
      start = (c == 0) || ((((int*)con)[CINFO * MC + c - 1] & 0xffff) != key);
    }
    unsigned bal = __ballot_sync(FULL, start);
    __syncwarp();  // (the neighbour's word is read above and rewritten below: only its top byte changes, but keep
                   // the accesses ordered - compute-sanitizer racecheck is clean with the two barriers)
    int before = ngroup + __popc(bal & ((1u << lane) - 1u));
    if (c < ncon) {
      int g = start ? before : before - 1;
      ((int*)con)[CINFO * MC + c] = (((int*)con)[CINFO * MC + c] & 0xffffff) | (g << 24);
      if (start) gstart[g] = c;
    }
    ngroup += __popc(bal);
    __syncwarp();
  }
  if (lane == 0) gstart[ngroup] = ncon;
  __syncwarp();
  // The Hessian keeps the dof tree's zero pattern unless a contact couples two branches (both bodies move and
  // neither chain contains the other): only then the factorisation takes the dense schedule.
  bool treeok = !(m.debug & 2);
  // kd: highest dof that any constraint row touches.  Dofs above it are unconstrained: eliminating them from
  // M once (phase 7) leaves the Schur complement on the leading block, and the Newton iterations run on that
  // block only (n x n instead of nv x nv; the other accelerations follow by back-substitution, phase 8).
  int kd = -1;
  #pragma unroll 1
  for (int g0 = 0; g0 < ngroup; g0 += 32) {
    bool bad = false;
    if (g0 + lane < ngroup) {
      int key = ((int*)con)[CINFO * MC + gstart[g0 + lane]] & 0xffff;
      unsigned long long m1 = m.body_dofmask[key & 0xff], m2 = m.body_dofmask[key >> 8];
      unsigned long long c = m1 & m2, x = m1 ^ m2;
      bad = c != m1 && c != m2;
      if (x) kd = max(kd, 63 - __clzll((long long)x));
    }
    if (__any_sync(FULL, bad)) treeok = false;
  }
  #pragma unroll 1
  for (int r = lane; r < nlim; r += 32) kd = max(kd, ((int*)lim)[LINFO * NLC + r] & 0xffff);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kd = max(kd, __shfl_xor_sync(FULL, kd, o));
  // n: the leading block the solver works on; a multiple of four pivots is eliminated (block factorisation)
  int n = nv - (((nv - (kd + 1)) >> 2) << 2);
  if (n > L.ndcap || (m.debug & 4)) n = nv;
  const bool reduced = n < nv;
  int nefc = nlim;
  {
    int cnt = 0;
    #pragma unroll 1
    for (int c = lane; c < ncon; c += 32) {
      int dim = ((int*)con)[CINFO * MC + c] >> 16 & 0xf;
      cnt += dim == 0 ? 0 : (dim == 1 ? 1 : 2 * (dim - 1));
    }
    cnt = (int)wsum((float)cnt);
    nefc += cnt;
  }

  float* gV = s + L.gV;
#define MULJ(x, dc, dl, acc) mulJ(x, dc, dl, acc, con, lim, gstart, gV, cdof, m.body_dofmask, ncon, nlim, ngroup, MC, NLC, lane)
  // CJAR <- -aref = B*vel_row + K*imp*(pos-margin) for contact rows (0 for unused rows)
  if (nefc > 0) {
    MULJ(qvel, CJV0, LJV, false);
    #pragma unroll 1
    for (int c = lane; c < ncon; c += 32) {
      float B = con[CB * MC + c], ki = con[CKI * MC + c];
      int dim = ((int*)con)[CINFO * MC + c] >> 16 & 0xf;
      int nr = dim == 0 ? 0 : (dim == 1 ? 1 : 4);
#pragma unroll
      for (int r = 0; r < 4; r++) con[(CJAR0 + r) * MC + c] = r < nr ? B * con[(CJV0 + r) * MC + c] + ki : 0.f;
    }
    __syncwarp();
  }

  PHASE_MARK(7);
  PSYNC();
  // ---------------- phase 7: unconstrained acceleration -------------------------------------------
  #pragma unroll 1
  for (int i = lane; i < (m.ntri + 3) >> 2; i += 32) ((float4*)H)[i] = ((const float4*)Mq)[i];  // both rows are 16 B aligned and padded
  __syncwarp();
  float* Mred = s + L.Mred;
  ldl_factor(H, invdiag, nv, SCHED, true, lane, 0, (reduced && nefc > 0) ? n : 0, Mred);
  SOLVE(qacc_smooth, true);
  if (m.debug & 1)
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) dd.qacc_smooth.p[(size_t)w * dd.qacc_smooth.stride + i] = qacc_smooth[i];

  PHASE_MARK(8);
  PSYNC();
  // ---------------- phase 8: Newton solver (primal, exact line search) ----------------------------
  int niter = 0, nls = 0;
  float cost = 0.f;
  const float* Mr = reduced ? Mred : Mq;  // reduced problem: Schur complement of M on the leading block
  const float* qs = qfrc_smooth;
  const float scale = 1.f / (m.meaninertia * (float)max(1, nv));
  float* gA = s + L.gA; float* gu = s + L.gu; int* glist = (int*)(s + L.glist); float* gW = s + L.gW;
  float oldcost = 0.f;
  bool first = true;
  // Conjugate gradient variant (opt.solver = CG; mujoco_warp's second solver): same cost, same update pass and
  // line search, search direction -M^-1 grad + beta * previous (Polak-Ribiere, preconditioned by M whose factor
  // phase 7 left in H - on a reduced problem its leading block is the factor of the Schur complement).  The
  // Hessian scratch is unused, so its weight region holds the direction and the previous (grad, M^-1 grad).
  const bool cg = m.solver == SOL_CG_;
  float* search = cg ? gW : s + L.search;  // Newton: search = -grad in place
  float* cgM = gW + pad4i(nv); float* cgG0 = gW + 2 * pad4i(nv); float* cgM0 = gW + 3 * pad4i(nv);
  bool refine = false;  // active set unchanged: the Hessian factor of the previous iteration is still valid
  int stall = 0;
  bool run = nefc > 0;  // this warp still iterates (under phase_sync finished warps keep voting at the loop top)
  if (nefc == 0) {
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) { qacc[i] = qacc_smooth[i]; qfrc_c[i] = 0.f; }
    __syncwarp();
  } else {
    // Reduced problem (n < nv): minimising the Gauss term over the unconstrained dofs in closed form leaves
    // 1/2 (a-a_s)^T Mr (a-a_s) on the leading block, Mr = Schur complement of M (snapshot of phase 7); the
    // code below is the full-size solver with (Mr, Mr a_s) in place of (M, qfrc_smooth).
    if (reduced) {
      symv(Mr, qacc_smooth, tmpv, n, lane);
      qs = tmpv;
    }
    // Shifted warm start: when this environment's control changed since its previous step (the first sub-step after
    // an action), the previous solution is moved by the change of the unconstrained acceleration, a_ws + (a_s -
    // a_s,prev): the constraint part a - a_s of the previous solution is then the better guess (-0.95 Newton
    // iterations on those sub-steps; with an unchanged control the plain warm start is better by 0.4).  The
    // minimiser reached is the same; MuJoCo's rule (fall back to a_s when it is cheaper) still applies.
    if (ctrl_changed) {
      const float* asp = dd.qacc_smooth_prev.p + (size_t)w * dd.qacc_smooth_prev.stride;
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) qacc_ws[i] += qacc_smooth[i] - asp[i];
      __syncwarp();
    }
    // warm start: qacc_warmstart unless qacc_smooth is cheaper (mj_fwdConstraint)
    symv(Mr, qacc_ws, Ma, n, lane);
    MULJ(qacc_smooth, CJV0, LJV, false);
    #pragma unroll 1
    for (int c = lane; c < ncon; c += 32)
#pragma unroll
      for (int r = 0; r < 4; r++) con[(CJV0 + r) * MC + c] += con[(CJAR0 + r) * MC + c];
    #pragma unroll 1
    for (int r = lane; r < nlim; r += 32) lim[LJV * NLC + r] += lim[LJAR * NLC + r];
    __syncwarp();
    float csm = rows_cost(CJV0, LJV, con, lim, ncon, nlim, MC, NLC, lane);
    MULJ(qacc_ws, CJAR0, LJAR, true);
    float cw = rows_cost(CJAR0, LJAR, con, lim, ncon, nlim, MC, NLC, lane);
    float gs = 0.f;
    #pragma unroll 1
    for (int i = lane; i < n; i += 32) gs += (Ma[i] - qs[i]) * (qacc_ws[i] - qacc_smooth[i]);
    cw += 0.5f * wsum(gs);
    bool use_smooth = cw > csm;
    #pragma unroll 1
    for (int i = lane; i < n; i += 32) qacc[i] = use_smooth ? qacc_smooth[i] : qacc_ws[i];
    __syncwarp();
    if (use_smooth) {
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) Ma[i] = qs[i];  // M * qacc_smooth
      #pragma unroll 1
      for (int c = lane; c < ncon; c += 32)
#pragma unroll
        for (int r = 0; r < 4; r++) con[(CJAR0 + r) * MC + c] = con[(CJV0 + r) * MC + c];
      #pragma unroll 1
      for (int r = lane; r < nlim; r += 32) lim[LJAR * NLC + r] = lim[LJV * NLC + r];
      __syncwarp();
    }
  }
  #pragma unroll 1
  while (true) {
    if (psync) { if (!__syncthreads_or(run ? 1 : 0)) break; } else if (!run) break;
    if (run) do {
      // ---- constraint update: forces, cost, active set, qfrc_constraint = J^T f ---------------
      float cst = 0.f;
      bool changed = false;
      #pragma unroll 1
      for (int c = lane; c < ncon; c += 32) {
        float D = con[CD * MC + c], mu = con[CMU * MC + c];
        int info = ((int*)con)[CINFO * MC + c];
        int dim = info >> 16 & 0xf;
        float f[4];
        int act = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
          float v = con[(CJAR0 + r) * MC + c];
          bool on = v < 0.f;
          f[r] = on ? -D * v : 0.f;
          if (on) { cst += 0.5f * D * v * v; act |= 1 << r; }
        }
        changed |= act != (info >> 20 & 0xf);
        ((int*)con)[CINFO * MC + c] = (info & (int)0xff0fffff) | (act << 20);
        float F0, F1, F2;
        if (dim == 1) { F0 = f[0]; F1 = 0.f; F2 = 0.f; }
        else { F0 = f[0] + f[1] + f[2] + f[3]; F1 = mu * (f[0] - f[1]); F2 = mu * (f[2] - f[3]); }
        con[(CJV0 + 0) * MC + c] = F0; con[(CJV0 + 1) * MC + c] = F1; con[(CJV0 + 2) * MC + c] = F2;
        // weights of this contact's 3x3 block W = B^T D_active B for the Hessian assembly
        float w0 = (act & 1) ? D : 0.f, w1 = (act & 2) ? D : 0.f, w2 = (act & 4) ? D : 0.f, w3 = (act & 8) ? D : 0.f;
        bool pyr = dim > 1;  // frictionless (condim 1) contacts contribute the normal row only
        if (!cg) {
          gW[0 * MC + c] = pyr ? w0 + w1 + w2 + w3 : w0;
          gW[1 * MC + c] = pyr ? mu * (w0 - w1) : 0.f;
          gW[2 * MC + c] = pyr ? mu * (w2 - w3) : 0.f;
          gW[3 * MC + c] = pyr ? mu * mu * (w0 + w1) : 0.f;
          gW[4 * MC + c] = pyr ? mu * mu * (w2 + w3) : 0.f;
        }
      }
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) qfrc_c[i] = 0.f;
      __syncwarp();
      #pragma unroll 1
      for (int r = lane; r < nlim; r += 32) {
        float v = lim[LJAR * NLC + r];
        int info = ((int*)lim)[LINFO * NLC + r];
        int act = v < 0.f ? 1 : 0;
        changed |= act != (info >> 20 & 1);
        ((int*)lim)[LINFO * NLC + r] = (info & 0xfffff) | (act << 20);
        if (act) {
          float D = lim[LD * NLC + r];
          cst += 0.5f * D * v * v;
          atomicAdd(&qfrc_c[info & 0xffff], ((info >> 16 & 1) ? -1.f : 1.f) * (-D * v));
        }
      }
      changed = __any_sync(FULL, changed);
      // group wrench: W_g = sum_c sum_m F_m S_m  (lanes (gi, comp))
      #pragma unroll 1
      for (int g0 = 0; g0 < ngroup; g0 += 5) {
        int gi = lane / 6, comp = lane - 6 * gi, g = g0 + gi;
        if (gi < 5 && g < ngroup) {
          float acc = 0.f;
          for (int c = gstart[g]; c < gstart[g + 1]; c++)
            acc += con[(CJV0 + 0) * MC + c] * con[(CS0 + comp) * MC + c] +
                   con[(CJV0 + 1) * MC + c] * con[(CS0 + 6 + comp) * MC + c] +
                   con[(CJV0 + 2) * MC + c] * con[(CS0 + 12 + comp) * MC + c];
          gV[6 * g + comp] = acc;
        }
      }
      __syncwarp();
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        float acc = qfrc_c[i];
        #pragma unroll 1
        for (int g = 0; g < ngroup; g++) {
          int key = ((int*)con)[CINFO * MC + gstart[g]] & 0xffff;
          unsigned long long m2 = m.body_dofmask[key >> 8];
          unsigned long long mk = m.body_dofmask[key & 0xff] ^ m2;
          if (mk >> i & 1ull) {
            float v = dot6(cdof + SD * i, gV + 6 * g);
            acc += (m2 >> i & 1ull) ? v : -v;
          }
        }
        qfrc_c[i] = acc;
      }
      __syncwarp();
      float gg = 0.f, gn = 0.f, fn = 0.f;
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        float fi = Ma[i] - qs[i];
        float g = fi - qfrc_c[i];
        grad[i] = g;
        gn += g * g;
        fn += fi * fi;
        gg += fi * (qacc[i] - qacc_smooth[i]);
      }
      cost = wsum(cst) + 0.5f * wsum(gg);
      gn = wsum(gn);
      fn = wsum(fn);
      if (!first) {
        float improvement = scale * (oldcost - cost), gradient = scale * sqrtf(gn);
        // MuJoCo stops when the scaled improvement or gradient drops below `tolerance` (1e-8).  In fp32 the cost
        // (1e3..1e5 here) resolves improvements only down to ~1e-4, so "no measurable improvement" can still
        // leave a residual of several newtons in the constraint forces: the improvement test is honoured only
        // once the gradient is small against the forces it balances (|M a - f_smooth| vs |J^T f|).
        constexpr float newton_small = 1e-10f;
        const bool small = gn <= newton_small * fmaxf(fn, 1.f);
        if (gradient < m.tolerance) { run = false; break; }
        // Exact termination: the cost is one quadratic per active set, and a Newton step with exact line
        // search lands on that quadratic's minimiser; if the active set did not change across the move, the
        // new point is the minimiser of the true (convex) cost - up to the error of the fp32 solve, hence the
        // same gradient condition.  When the set is unchanged but the residual is not yet small, the next
        // iteration is one step of iterative refinement: same Hessian, its factor is reused.
        if (small && (improvement < m.tolerance || (!changed && !cg))) { run = false; break; }
        stall = improvement <= 0.f ? stall + 1 : 0;
        if (stall >= 2) { run = false; break; }  // two moves without any measurable decrease: fp32 floor reached
        refine = !changed && !cg;
      }
      if (niter >= m.iterations) { run = false; break; }
      first = false;
    } while (0);
    PHASE_MARK(12);
    PSYNC();
    if (run && !refine && !cg) {
      // ---- Hessian H = M + J^T D_active J via per-body-pair 6x6 blocks -------------------------
      {  // leading block only: the rows of the eliminated dofs keep the factor of M (needed after the loop)
        const int nt = n * (n + 1) >> 1;
        #pragma unroll 1
        for (int i = lane; i < nt >> 2; i += 32) ((float4*)H)[i] = ((const float4*)Mr)[i];  // 16 B aligned regions
        if (lane < (nt & 3)) H[(nt & ~3) + lane] = Mr[(nt & ~3) + lane];
      }
      __syncwarp();
      #pragma unroll 1
      for (int r = lane; r < nlim; r += 32) {
        if (lim[LJAR * NLC + r] < 0.f) {
          int d = ((int*)lim)[LINFO * NLC + r] & 0xffff;
          atomicAdd(&H[tri(d, d)], lim[LD * NLC + r]);
        }
      }
      #pragma unroll 1
      for (int g = 0; g < ngroup; g++) {
        // A (6x6 symmetric, 21 entries), lane e owns entry (a,b)
        if (lane < 21) {
          // (a, b), a <= b, of the lane's entry: 3-bit fields of two packed constants
          const int a = (int)(0x591b692449240000ull >> (3 * lane)) & 7, b = (int)(0x5b2c76356346c688ull >> (3 * lane)) & 7;
          float acc = 0.f;
          for (int c = gstart[g]; c < gstart[g + 1]; c++) {
            float W00 = gW[c], W01 = gW[MC + c], W02 = gW[2 * MC + c], W11 = gW[3 * MC + c], W22 = gW[4 * MC + c];
            float sa0 = con[(CS0 + a) * MC + c], sb0 = con[(CS0 + b) * MC + c];
            float sa1 = con[(CS0 + 6 + a) * MC + c], sb1 = con[(CS0 + 6 + b) * MC + c];
            float sa2 = con[(CS0 + 12 + a) * MC + c], sb2 = con[(CS0 + 12 + b) * MC + c];
            acc += W00 * sa0 * sb0 + W01 * (sa0 * sb1 + sa1 * sb0) + W02 * (sa0 * sb2 + sa2 * sb0) +
                   W11 * sa1 * sb1 + W22 * sa2 * sb2;
          }
          gA[a * 6 + b] = acc;
          gA[b * 6 + a] = acc;
        }
        // dof list of the group (ascending) with signs folded into u
        int key = ((int*)con)[CINFO * MC + gstart[g]] & 0xffff;
        unsigned long long m2 = m.body_dofmask[key >> 8];
        unsigned long long mk = m.body_dofmask[key & 0xff] ^ m2;
        unsigned lo = (unsigned)mk, hi = (unsigned)(mk >> 32);
        int nlo = __popc(lo), ns = nlo + __popc(hi);
        if (lo >> lane & 1u) glist[__popc(lo & ((1u << lane) - 1u))] = lane;
        if (hi >> lane & 1u) glist[nlo + __popc(hi & ((1u << lane) - 1u))] = 32 + lane;
        __syncwarp();
        // u_a = sign_a * A * cdof_a: one (dof, component) per lane
        #pragma unroll 1
        for (int t = lane; t < 6 * ns; t += 32) {
          int a = t / 6, k = t - 6 * a;
          int d = glist[a];
          const float* c = cdof + SD * d;
          const float* ga = gA + 6 * k;
          float v = ga[0] * c[0] + ga[1] * c[1] + ga[2] * c[2] + ga[3] * c[3] + ga[4] * c[4] + ga[5] * c[5];
          gu[t] = (m2 >> d & 1ull) ? v : -v;
        }
        __syncwarp();
        // H[da, db] += u_a . (sign_b cdof_b) for the pairs a >= b of the group's dof list, one pair per lane
        const int npr = ns * (ns + 1) >> 1;
        #pragma unroll 1
        for (int p = lane; p < npr; p += 32) {
          int a = (int)((sqrtf(8.f * (float)p + 1.f) - 1.f) * 0.5f);
          if ((a * (a + 1) >> 1) > p) a--;
          if (((a + 1) * (a + 2) >> 1) <= p) a++;
          int b = p - (a * (a + 1) >> 1);
          int da = glist[a], db = glist[b];
          const float* u = gu + 6 * a;
          const float* c = cdof + SD * db;
          float v = u[0] * c[0] + u[1] * c[1] + u[2] * c[2] + u[3] * c[3] + u[4] * c[4] + u[5] * c[5];
          H[(da * (da + 1) >> 1) + db] += (m2 >> db & 1ull) ? v : -v;
        }
        __syncwarp();
      }
    }
    PHASE_MARK(13);
    PSYNC();
    if (run && !cg) {
      if (!refine) ldl_factor(H, invdiag, n, SCHED, treeok, lane, (nv - n) >> 2);
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) search[i] = -grad[i];  // (grad and search share one vector)
      __syncwarp();
      ldl_solve(H, invdiag, search, n, lane);
    }
    if (run && cg) {
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) cgM[i] = grad[i];
      __syncwarp();
      ldl_solve(H, invdiag, cgM, n, lane);  // M^-1 grad (factor of M, phase 7)
      float num = 0.f, den = 0.f;
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) { num += grad[i] * (cgM[i] - cgM0[i]); den += cgG0[i] * cgM0[i]; }
      num = wsum(num); den = wsum(den);
      const float beta = niter == 0 ? 0.f : fmaxf(0.f, num / fmaxf(den, MINVAL));
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        search[i] = -cgM[i] + (niter == 0 ? 0.f : beta * search[i]);
        cgG0[i] = grad[i]; cgM0[i] = cgM[i];
      }
      __syncwarp();
    }
    PHASE_MARK(14);
    PSYNC();
    if (run) do {
      // ---- exact line search along `search` --------------------------------------------------
      symv(Mr, search, Mv, n, lane);
      MULJ(search, CJV0, LJV, false);
      float g1 = 0.f, g2 = 0.f, sn = 0.f;
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) {
        g1 += search[i] * (Ma[i] - qs[i]);
        g2 += 0.5f * search[i] * Mv[i];
        sn += search[i] * search[i];
      }
      g1 = wsum(g1); g2 = wsum(g2); sn = sqrtf(wsum(sn));
      if (sn < MINVAL) { run = false; break; }
      float gtol = m.tolerance * m.ls_tolerance * sn / scale;
      // each lane keeps its rows in registers for the whole search (<= 2 contacts + 1 limit per lane)
      float lsJ[9], lsV[9], lsDV[9];  // residual, its slope, and D * slope per row
      const bool wide = ncon > 32, anylim = nlim > 0;  // second contact per lane / limit rows present (warp-uniform)
#pragma unroll
      for (int q = 0; q < 2; q++) {
        int c = lane + 32 * q;
        bool ok = c < ncon && (q == 0 || wide);
        const float D = ok ? con[CD * MC + c] : 0.f;
#pragma unroll
        for (int r = 0; r < 4; r++) {
          lsJ[4 * q + r] = ok ? con[(CJAR0 + r) * MC + c] : 0.f;
          lsV[4 * q + r] = ok ? con[(CJV0 + r) * MC + c] : 0.f;
          lsDV[4 * q + r] = D * lsV[4 * q + r];
        }
      }
      {
        bool ok = lane < nlim;
        lsJ[8] = ok ? lim[LJAR * NLC + lane] : 0.f;
        lsV[8] = ok ? lim[LJV * NLC + lane] : 0.f;
        lsDV[8] = ok ? lim[LD * NLC + lane] * lsV[8] : 0.f;
      }
      auto ls_eval = [&](float al, float& d0, float& d1) {
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int q = 0; q < 4; q++) {
          float x = fmaf(al, lsV[q], lsJ[q]);
          if (x < 0.f) { a0 = fmaf(lsDV[q], x, a0); a1 = fmaf(lsDV[q], lsV[q], a1); }
        }
        if (wide) {  // (environments with at most 32 contacts - nearly all - skip the second contact's rows)
#pragma unroll
          for (int q = 4; q < 8; q++) {
            float x = fmaf(al, lsV[q], lsJ[q]);
            if (x < 0.f) { a0 = fmaf(lsDV[q], x, a0); a1 = fmaf(lsDV[q], lsV[q], a1); }
          }
        }
        if (anylim) {
          float x = fmaf(al, lsV[8], lsJ[8]);
          if (x < 0.f) { a0 = fmaf(lsDV[8], x, a0); a1 = fmaf(lsDV[8], lsV[8], a1); }
        }
        // rows beyond the register window (ncon > 64 or nlim > 32)
        #pragma unroll 1
        for (int c = lane + 64; c < ncon; c += 32) {
          float D = con[CD * MC + c];
#pragma unroll
          for (int r = 0; r < 4; r++) {
            float jv = con[(CJV0 + r) * MC + c];
            float x = con[(CJAR0 + r) * MC + c] + al * jv;
            if (x < 0.f) { a0 += D * x * jv; a1 += D * jv * jv; }
          }
        }
        #pragma unroll 1
        for (int r = lane + 32; r < nlim; r += 32) {
          float jv = lim[LJV * NLC + r];
          float x = lim[LJAR * NLC + r] + al * jv;
          if (x < 0.f) { float D = lim[LD * NLC + r]; a0 += D * x * jv; a1 += D * jv * jv; }
        }
        d0 = wsum(a0) + g1 + 2.f * al * g2;
        d1 = fmaxf(wsum(a1) + 2.f * g2, MINVAL);
        nls++;
      };
      PHASE_MARK(15);
      float alpha = 0.f, d0, d1;
      // Slope and curvature at 0 are evaluated, for Newton and CG alike.  For a Newton direction (H search = -grad)
      // they could be taken from grad . search with a first trial step of 1, one evaluation fewer per iteration;
      // that saved no measurable time on the GPU, and the worst of 1024 stiff envs of the config-C parity states
      // moved from 1.8e-4 to 3.3e-4.
      ls_eval(0.f, d0, d1);
      if (d0 < 0.f) {
        float lo_a = 0.f, hi_a = -1.f;  // hi_a < 0: no upper bracket yet
        // stop once the slope is 1e-3 of its value at 0 (emulated bench workload: 7.0 -> 3.4 evaluations per
        // Newton iteration, iteration count unchanged: 4.665 -> 4.67)
        constexpr float ls_rtol = 1e-3f;
        const float dstop = fmaxf(gtol, ls_rtol * fabsf(d0));
        alpha = -d0 / d1;
        #pragma unroll 1
        for (int it = 0; it < m.ls_iterations; it++) {
          ls_eval(alpha, d0, d1);
          if (fabsf(d0) < dstop) break;
          if (d0 < 0.f) lo_a = alpha; else hi_a = alpha;
          float nxt = alpha - d0 / d1;
          if (hi_a >= 0.f && !(nxt > lo_a && nxt < hi_a)) nxt = 0.5f * (lo_a + hi_a);
          if (nxt == alpha) break;
          // The derivative is piecewise linear: a Newton step taken inside the root's piece lands on the root, and
          // the next evaluation returns fp32 noise, never |d0| < gtol (gtol ~ 1e-8 |search|).  A step below a few
          // ulp of alpha is that situation: take it and stop instead of dithering until the bracket collapses.
          if (fabsf(nxt - alpha) <= 4e-7f * fabsf(alpha)) { alpha = nxt; break; }
          alpha = nxt;
        }
      }
      PHASE_MARK(16);
      if (alpha == 0.f) { run = false; break; }
      #pragma unroll 1
      for (int i = lane; i < n; i += 32) { qacc[i] += alpha * search[i]; Ma[i] += alpha * Mv[i]; }
      #pragma unroll 1
      for (int c = lane; c < ncon; c += 32)
#pragma unroll
        for (int r = 0; r < 4; r++) con[(CJAR0 + r) * MC + c] += alpha * con[(CJV0 + r) * MC + c];
      #pragma unroll 1
      for (int r = lane; r < nlim; r += 32) lim[LJAR * NLC + r] += alpha * lim[LJV * NLC + r];
      __syncwarp();
      oldcost = cost;
      niter++;
    } while (0);
  }
  if (nefc > 0) {
    if (reduced) {
      // eliminated dofs: a_c = a_s,c - L_cc^-1 L_cd (a_d - a_s,d), i.e. rows k >= n of L x = 0 with x_d given
      // (the factor of M from phase 7 is intact in those rows: x_k = -(1/d_k) sum_{j<k} A[k,j] x_j)
      #pragma unroll 1
      for (int i = lane; i < nv; i += 32) Mv[i] = i < n ? qacc[i] - qacc_smooth[i] : 0.f;
      __syncwarp();
      #pragma unroll 1
      for (int k = n; k < nv; k++) {
        const int rk = k * (k + 1) >> 1;
        float part = lane < k ? H[rk + lane] * Mv[lane] : 0.f;
        if (lane + 32 < k) part += H[rk + 32 + lane] * Mv[lane + 32];
        part = wsum(part);
        if (lane == 0) Mv[k] = -invdiag[k] * part;
        __syncwarp();
      }
      #pragma unroll 1
      for (int i = n + lane; i < nv; i += 32) { qacc[i] = qacc_smooth[i] + Mv[i]; qfrc_c[i] = 0.f; }
      __syncwarp();
    }
  }

  if (STEP) {
    float* asp = dd.qacc_smooth_prev.p + (size_t)w * dd.qacc_smooth_prev.stride;
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) asp[i] = qacc_smooth[i];
  }
  PHASE_MARK(9);
  PSYNC();
  // ---------------- phase 9: contact forces, sensors -----------------------------------------------
  {
    float* g_force = dd.contact_force.p + (size_t)w * dd.contact_force.stride;
    #pragma unroll 1
    for (int c = lane; c < ncon; c += 32) {
      float D = con[CD * MC + c], mu = con[CMU * MC + c];
      int dim = ((int*)con)[CINFO * MC + c] >> 16 & 0xf;
      float f[4];
#pragma unroll
      for (int r = 0; r < 4; r++) { float v = con[(CJAR0 + r) * MC + c]; f[r] = (nefc > 0 && v < 0.f) ? -D * v : 0.f; }
      float F0, F1, F2;
      if (dim == 0) { F0 = F1 = F2 = 0.f; }
      else if (dim == 1) { F0 = f[0]; F1 = F2 = 0.f; }
      else { F0 = f[0] + f[1] + f[2] + f[3]; F1 = mu * (f[0] - f[1]); F2 = mu * (f[2] - f[3]); }
      con[(CJV0 + 0) * MC + c] = F0; con[(CJV0 + 1) * MC + c] = F1; con[(CJV0 + 2) * MC + c] = F2;
      g_force[3 * c] = F0; g_force[3 * c + 1] = F1; g_force[3 * c + 2] = F2;
    }
    __syncwarp();
    float* sd = dd.sensordata.p + (size_t)w * dd.sensordata.stride;
    const float* g_pos = dd.contact_pos.p + (size_t)w * dd.contact_pos.stride;
    const int* g_geom = dd.contact_geom.p + (size_t)w * dd.contact_geom.stride;
    #pragma unroll 1
    for (int sidx = 0; sidx < m.nsensor; sidx++) {
      int dataspec = m.sensor_intprm[3 * sidx], reduce = m.sensor_intprm[3 * sidx + 1], num = m.sensor_intprm[3 * sidx + 2];
      int adr = m.sensor_adr[sidx], sdim = m.sensor_dim[sidx];
      int slot = sdim / max(num, 1);
      int ot = m.sensor_objtype[sidx], oi = m.sensor_objid[sidx];
      int rt = m.sensor_reftype[sidx], ri = m.sensor_refid[sidx];
      #pragma unroll 1
      for (int k = lane; k < sdim; k += 32) sd[adr + k] = 0.f;
      int nmatch = 0;
      float net[3] = {0.f, 0.f, 0.f}, wp[3] = {0.f, 0.f, 0.f}, wsm = 0.f;
      #pragma unroll 1
      for (int c00 = 0; c00 < ncon; c00 += 32) {
        int c = c00 + lane;
        int dir = 0;
        if (c < ncon && (((int*)con)[CINFO * MC + c] >> 16 & 0xf) != 0) {
          int g1 = g_geom[2 * c], g2 = g_geom[2 * c + 1];
          auto match = [&](int type, int id, int geom) -> bool {
            if (type < 0) return true;
            int b = m.geom_bodyid[geom];
            if (type == OBJ_GEOM) return geom == id;
            if (type == OBJ_BODY) return b == id;
            if (type == OBJ_XBODY) return (m.body_ancmask[b] >> id & 1ull) != 0ull;
            return false;
          };
          if (match(ot, oi, g1) && match(rt, ri, g2)) dir = 1;
          else if (match(ot, oi, g2) && match(rt, ri, g1)) dir = -1;
        }
        unsigned bal = __ballot_sync(FULL, dir != 0);
        if (dir != 0) {
          float F0 = con[(CJV0 + 0) * MC + c], F1 = con[(CJV0 + 1) * MC + c], F2 = con[(CJV0 + 2) * MC + c];
          float fw[3];
          for (int k = 0; k < 3; k++)
            fw[k] = dir * (con[(CS0 + 3 + k) * MC + c] * F0 + con[(CS0 + 9 + k) * MC + c] * F1 + con[(CS0 + 15 + k) * MC + c] * F2);
          if (reduce == 3) {
            float mag = sqrtf(dot3(fw, fw));
            for (int k = 0; k < 3; k++) { net[k] += fw[k]; wp[k] += mag * g_pos[3 * c + k]; }
            wsm += mag;
          } else if (reduce == 0) {
            int idx = nmatch + __popc(bal & ((1u << lane) - 1u));
            if (idx < num) {
              float* q = sd + adr + idx * slot;
              int a = 0;
              if (dataspec & 1) a++;
              if (dataspec & 2) { q[a] = F0; q[a + 1] = dir * F1; q[a + 2] = dir * F2; a += 3; }
              if (dataspec & 4) a += 3;
              if (dataspec & 8) q[a++] = con[CDIST * MC + c];
              if (dataspec & 16) { for (int k = 0; k < 3; k++) q[a + k] = g_pos[3 * c + k]; a += 3; }
              if (dataspec & 32) { for (int k = 0; k < 3; k++) q[a + k] = dir * con[(CS0 + 3 + k) * MC + c]; a += 3; }
            }
          }
        }
        nmatch += __popc(bal);
      }
      __syncwarp();
      if (reduce == 3) {
        for (int k = 0; k < 3; k++) { net[k] = wsum(net[k]); wp[k] = wsum(wp[k]); }
        wsm = wsum(wsm);
        if (nmatch > 0 && lane == 0) {
          int a = 0;
          if (dataspec & 1) sd[adr + a++] = (float)nmatch;
          if (dataspec & 2) { for (int k = 0; k < 3; k++) sd[adr + a + k] = net[k]; a += 3; }
          if (dataspec & 4) a += 3;
          if (dataspec & 8) sd[adr + a++] = 0.f;
          if (dataspec & 16) { for (int k = 0; k < 3; k++) sd[adr + a + k] = wsm > 0.f ? wp[k] / wsm : 0.f; a += 3; }
          if (dataspec & 32) { float nn[3] = {net[0], net[1], net[2]}; normalize3(nn); for (int k = 0; k < 3; k++) sd[adr + a + k] = nn[k]; }
        }
      } else if (reduce == 0 && (dataspec & 1)) {
        int filled = min(nmatch, num);
        #pragma unroll 1
        for (int i = lane; i < filled; i += 32) sd[adr + i * slot] = (float)nmatch;
      }
    }
  }

  PHASE_MARK(10);
  PSYNC();
  // ---------------- phase 10: integrate (implicitfast / Euler), write state ------------------------
  float* gq = dd.qpos.p + (size_t)w * dd.qpos.stride;
  float* gv = dd.qvel.p + (size_t)w * dd.qvel.stride;
  if (STEP) {
    const float h = m.timestep;
    const float* damp = MP(dof_damping); const float* bp = MP(actuator_biasprm);
    const float* fr = MP(actuator_forcerange); const float* gear = MP(actuator_gear);
    #pragma unroll 1
    for (int i = lane; i < (m.ntri + 3) >> 2; i += 32) ((float4*)H)[i] = ((const float4*)Mq)[i];  // both rows are 16 B aligned and padded
    __syncwarp();
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) H[tri(i, i)] += h * damp[i];
    __syncwarp();
    if (m.integrator == INT_IMPLICITFAST) {
      #pragma unroll 1
      for (int a = lane; a < nu; a += 32) {
        float bv = bp[10 * a + 2];
        if (bv == 0.f) continue;
        if (m.actuator_forcelimited[a]) {
          float f = actf[a];
          if (f <= fr[2 * a] || f >= fr[2 * a + 1]) continue;
        }
        int dof = m.jnt_dofadr[m.actuator_trnid[a]];
        atomicAdd(&H[tri(dof, dof)], -h * gear[a] * gear[a] * bv);
      }
    }
    bool anydamp = false;
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) anydamp |= damp[i] > 0.f;
    anydamp = __any_sync(FULL, anydamp);
    if (m.integrator == INT_IMPLICITFAST || anydamp) {
      #pragma unroll 1
      for (int i = lane; i < nv; i += 32) tmpv[i] = qfrc_smooth[i] + qfrc_c[i];
      __syncwarp();
      FACTOR(true);
      SOLVE(tmpv, true);
    } else {
      #pragma unroll 1
      for (int i = lane; i < nv; i += 32) tmpv[i] = qacc[i];
      __syncwarp();
    }
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) qvel[i] += h * tmpv[i];
    __syncwarp();
    #pragma unroll 1
    for (int j = lane; j < njnt; j += 32) {
      int qa = m.jnt_qposadr[j], da = m.jnt_dofadr[j];
      if (m.jnt_type[j] == JNT_FREE) {
        qpos[qa] += h * qvel[da]; qpos[qa + 1] += h * qvel[da + 1]; qpos[qa + 2] += h * qvel[da + 2];
        float v[3] = {qvel[da + 3], qvel[da + 4], qvel[da + 5]};
        float n = sqrtf(dot3(v, v));
        float q[4] = {qpos[qa + 3], qpos[qa + 4], qpos[qa + 5], qpos[qa + 6]};
        if (n > MINVAL) {
          float sn, cs;
          sincosf(0.5f * h * n, &sn, &cs);
          float inv = sn / n;
          float qr[4] = {cs, v[0] * inv, v[1] * inv, v[2] * inv}, qn[4];
          mulquat(qn, q, qr);
          q[0] = qn[0]; q[1] = qn[1]; q[2] = qn[2]; q[3] = qn[3];
        }
        normalize4(q);
        qpos[qa + 3] = q[0]; qpos[qa + 4] = q[1]; qpos[qa + 5] = q[2]; qpos[qa + 6] = q[3];
      } else qpos[qa] += h * qvel[da];
    }
    __syncwarp();
    if (lane == 0) dd.time.p[(size_t)w * dd.time.stride] += h;
    float* gws = dd.qacc_warmstart.p + (size_t)w * dd.qacc_warmstart.stride;
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) gws[i] = qacc[i];
  }
  // outputs that live contiguously in shared memory leave through bulk (TMA) stores
  {
    float* gqa = dd.qacc.p + (size_t)w * dd.qacc.stride;
    #pragma unroll 1
    for (int i = lane; i < nv; i += 32) gqa[i] = qacc[i];
    if (m.debug & 1) {
      float* gfc = dd.qfrc_constraint.p + (size_t)w * dd.qfrc_constraint.stride;
      #pragma unroll 1
      for (int i = lane; i < nv; i += 32) gfc[i] = qfrc_c[i];
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0 && STEP) {
      bulk_s2g(gq, qpos, 4u * dd.qpos.stride);
      bulk_s2g(gv, qvel, 4u * dd.qvel.stride);
      bulk_commit_wait();
    }
    PHASE_MARK(11);
    if (lane == 0) {
      dd.ncon.p[(size_t)w * dd.ncon.stride] = ncon;
      dd.nefc.p[(size_t)w * dd.nefc.stride] = nefc;
      dd.solver_niter.p[(size_t)w * dd.solver_niter.stride] = niter;
      dd.solver_nd.p[(size_t)w * dd.solver_nd.stride] = nefc > 0 ? n : 0;  // size of the block the solver worked on
      dd.solver_nls.p[(size_t)w * dd.solver_nls.stride] = nls;
      dd.overflow.p[(size_t)w * dd.overflow.stride] = overflow;
      dd.solver_cost.p[(size_t)w * dd.solver_cost.stride] = cost;
    }
  }
}
