// b2sim.cu — libb2sim.so: C ABI (include/b2sim.h) around the fused sm_100a step kernel.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/b2sim.h"
#include "b2_kernel.cuh"
#include "b2_tables.h"
#include "b2_env.cuh"
#include "b2_trackenv.cuh"

static thread_local std::string g_err;
static int fail(const std::string& msg) {
  g_err = msg;
  return 1;
}
#define CUDA_OK(expr)                                                                     \
  do {                                                                                    \
    cudaError_t e_ = (expr);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(std::string(#expr) + ": " + cudaGetErrorString(e_));                    \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

struct Field {
  std::string name;
  void* ptr = nullptr;
  int dtype = B2_F32;
  int ndim = 1;
  int64_t shape[4] = {1, 1, 1, 1};
  int64_t stride[4] = {0, 0, 0, 1};
  FArr* farr = nullptr;  // model float arrays: where the kernel reads the pointer from
  int64_t n = 0;         // elements per world
};

// b2_step_n runs this many environment partitions on internal streams once each holds at least 1024 environments
static constexpr int B2_PARTITIONS = 2;

struct b2_sim {
  int device = 0;
  int nworld = 0;
  DevModel hm;
  DevData hd;
  std::vector<Field> data_fields, model_fields;
  std::vector<void*> allocs;
  int64_t launches = 0;
  int* order = nullptr;       // heavy-first dispatch order (device)
  int sorted_dispatch = 1;     // heavy-first order, recomputed before every sub-step (measured 447 vs 462 us against once per
                               // b2_step_n: fresh Newton counts keep phase-synchronous CTAs balanced)
  int has_convex = 0;          // the model has mesh / height-field collision pairs: kernels with the convex routines
  cudaStream_t side[B2_PARTITIONS] = {};  // b2_step_n: one internal stream per environment partition
  cudaEvent_t ev_fork = nullptr, ev_join[B2_PARTITIONS] = {};
  size_t smem_bytes = 0;
  std::map<std::string, std::vector<double>> mf;  // host copy of float model arrays
  std::map<std::string, std::vector<int>> mi;
};

static int pad4(int n) { return (n + 3) & ~3; }

template <typename T>
static int dev_upload(b2_sim* s, const std::vector<T>& h, const T** out) {
  void* p = nullptr;
  size_t bytes = sizeof(T) * std::max<size_t>(h.size(), 1);
  CUDA_OK(cudaMalloc(&p, bytes));
  s->allocs.push_back(p);
  if (!h.empty()) CUDA_OK(cudaMemcpy(p, h.data(), sizeof(T) * h.size(), cudaMemcpyHostToDevice));
  *out = (const T*)p;
  return 0;
}

__global__ void b2_tile_kernel(const float* __restrict__ src, float* __restrict__ dst, int n,
                               long long total) {
  long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid < total) dst[tid] = src[tid % n];
}
__global__ void b2_init_rows_kernel(float* dst, int stride, const float* __restrict__ src, int n,
                                    int nworld) {
  long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid < (long long)nworld * n) dst[(tid / n) * stride + (tid % n)] = src[tid % n];
}

// World poses of the grid-static geoms are constant: written into every world's geom_xpos / geom_xmat once.
__global__ void b2_static_rows_kernel(float* xpos, int xpos_stride, float* xmat, int xmat_stride,
                                      const float* __restrict__ pose, const int* __restrict__ static_geom,
                                      int nstatic, int nworld) {
  long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (long long)nworld * nstatic) return;
  int k = (int)(tid % nstatic), g = static_geom[k];
  size_t w = (size_t)(tid / nstatic);
  const float* p = pose + 16 * (size_t)k;
  for (int i = 0; i < 3; i++) xpos[w * xpos_stride + 3 * g + i] = p[i];
  for (int i = 0; i < 9; i++) xmat[w * xmat_stride + 9 * g + i] = p[3 + i];
}

// Heavy-first dispatch: order worlds by the previous step's (Newton iterations, contacts),
// descending, with a one-CTA counting sort (128 buckets).  Only scheduling changes, not results.
// Key = (Newton iterations, solver block class, contacts / 8): under phase-synchronous execution the warps of a
// CTA wait for each other at every phase boundary, so a CTA should hold environments of equal cost.
__device__ __forceinline__ int b2_order_key(int niter, int nd, int ncon, int nd_small) {
  return min(niter, 15) * 8 + (nd > nd_small ? 4 : 0) + min(ncon >> 3, 3);
}
__global__ void b2_order_kernel(const int* __restrict__ niter, int niter_stride, const int* __restrict__ ncon,
                                int ncon_stride, const int* __restrict__ nd, int nd_stride, int nd_small,
                                int base_world, int count, int* __restrict__ order) {
  __shared__ int hist[128];
  __shared__ int base[128];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  // (keys stay in registers between the two passes: up to 4 worlds per thread, the common case; more are re-read)
  int keys[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int k = threadIdx.x + j * blockDim.x;
    keys[j] = -1;
    if (k < count) {
      int w = base_world + k;
      keys[j] = 127 - b2_order_key(niter[(size_t)w * niter_stride], nd[(size_t)w * nd_stride], ncon[(size_t)w * ncon_stride], nd_small);
      atomicAdd(&hist[keys[j]], 1);
    }
  }
  for (int k = threadIdx.x + 4 * blockDim.x; k < count; k += blockDim.x) {
    int w = base_world + k;
    atomicAdd(&hist[127 - b2_order_key(niter[(size_t)w * niter_stride], nd[(size_t)w * nd_stride], ncon[(size_t)w * ncon_stride], nd_small)], 1);
  }
  __syncthreads();
  if (threadIdx.x < 32) {  // exclusive prefix over the 128 buckets: 4 per lane + a warp scan
    int h0 = hist[4 * threadIdx.x], h1 = hist[4 * threadIdx.x + 1], h2 = hist[4 * threadIdx.x + 2], h3 = hist[4 * threadIdx.x + 3];
    int sum = h0 + h1 + h2 + h3, incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((int)threadIdx.x >= o) incl += t;
    }
    int ex = incl - sum;
    base[4 * threadIdx.x] = ex; base[4 * threadIdx.x + 1] = ex + h0;
    base[4 * threadIdx.x + 2] = ex + h0 + h1; base[4 * threadIdx.x + 3] = ex + h0 + h1 + h2;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int k = threadIdx.x + j * blockDim.x;
    if (k < count) order[base_world + atomicAdd(&base[keys[j]], 1)] = base_world + k;
  }
  for (int k = threadIdx.x + 4 * blockDim.x; k < count; k += blockDim.x) {
    int w = base_world + k;
    int key = 127 - b2_order_key(niter[(size_t)w * niter_stride], nd[(size_t)w * nd_stride], ncon[(size_t)w * ncon_stride], nd_small);
    order[base_world + atomicAdd(&base[key], 1)] = w;
  }
}

// inner shapes of model float fields: dims after the (broadcast) world dimension
struct ShapeSpec { const char* name; int second; };  // second = trailing dim (0 -> 1-D)
static const ShapeSpec kModelShapes[] = {
    {"body_pos", 3}, {"body_quat", 4}, {"body_ipos", 3}, {"body_iquat", 4}, {"body_mass", 0},
    {"body_subtreemass", 0}, {"body_inertia", 3}, {"body_invweight0", 2}, {"jnt_pos", 3},
    {"jnt_axis", 3}, {"jnt_range", 2}, {"jnt_solref", 2}, {"jnt_solimp", 5}, {"jnt_margin", 0},
    {"jnt_stiffness", 0}, {"dof_armature", 0}, {"dof_damping", 0}, {"dof_frictionloss", 0},
    {"dof_invweight0", 0}, {"geom_size", 3}, {"geom_pos", 3}, {"geom_quat", 4},
    {"geom_friction", 3}, {"geom_solref", 2}, {"geom_solimp", 5}, {"geom_solmix", 0},
    {"geom_margin", 0}, {"geom_gap", 0}, {"geom_rbound", 0}, {"geom_rgba", 4}, {"site_pos", 3},
    {"site_quat", 4}, {"actuator_gainprm", 10}, {"actuator_biasprm", 10},
    {"actuator_ctrlrange", 2}, {"actuator_forcerange", 2}, {"actuator_gear", 0}, {"qpos0", 0}};

static FArr* model_farr(DevModel& m, const std::string& name) {
#define F_(x) if (name == #x) return &m.x;
  F_(body_pos) F_(body_quat) F_(body_ipos) F_(body_iquat) F_(body_mass) F_(body_subtreemass)
  F_(body_inertia) F_(body_invweight0) F_(jnt_pos) F_(jnt_axis) F_(jnt_range) F_(jnt_solref)
  F_(jnt_solimp) F_(jnt_margin) F_(jnt_stiffness) F_(dof_armature) F_(dof_damping)
  F_(dof_frictionloss) F_(dof_invweight0) F_(geom_size) F_(geom_pos) F_(geom_quat)
  F_(geom_friction) F_(geom_solref) F_(geom_solimp) F_(geom_solmix) F_(geom_margin) F_(geom_gap)
  F_(geom_rbound) F_(geom_rgba) F_(site_pos) F_(site_quat) F_(actuator_gainprm)
  F_(actuator_biasprm) F_(actuator_ctrlrange) F_(actuator_forcerange) F_(actuator_gear) F_(qpos0)
#undef F_
  return nullptr;
}

static int add_data(b2_sim* s, const char* name, DArr* arr, int n, int second = 0) {
  int stride = pad4(std::max(n, 0));
  if (stride == 0) stride = 4;
  void* p = nullptr;
  size_t bytes = sizeof(float) * (size_t)s->nworld * stride;
  CUDA_OK(cudaMalloc(&p, bytes));
  CUDA_OK(cudaMemset(p, 0, bytes));
  s->allocs.push_back(p);
  arr->p = (float*)p; arr->stride = stride; arr->n = n;
  Field f;
  f.name = name; f.ptr = p; f.dtype = B2_F32; f.n = n;
  if (second == 9) {  // rotation matrices are exposed as (nworld, n, 3, 3) like mjwarp's mat33 arrays
    f.ndim = 4; f.shape[0] = s->nworld; f.shape[1] = n / 9; f.shape[2] = 3; f.shape[3] = 3;
    f.stride[0] = stride; f.stride[1] = 9; f.stride[2] = 3; f.stride[3] = 1;
  } else if (second > 0) {
    f.ndim = 3; f.shape[0] = s->nworld; f.shape[1] = n / second; f.shape[2] = second;
    f.stride[0] = stride; f.stride[1] = second; f.stride[2] = 1;
  } else {
    f.ndim = 2; f.shape[0] = s->nworld; f.shape[1] = n;
    f.stride[0] = stride; f.stride[1] = 1;
  }
  s->data_fields.push_back(f);
  return 0;
}
static int add_idata(b2_sim* s, const char* name, IArr* arr, int n, int second = 0) {
  int stride = pad4(std::max(n, 1));
  void* p = nullptr;
  size_t bytes = sizeof(int) * (size_t)s->nworld * stride;
  CUDA_OK(cudaMalloc(&p, bytes));
  CUDA_OK(cudaMemset(p, 0, bytes));
  s->allocs.push_back(p);
  arr->p = (int*)p; arr->stride = stride; arr->n = n;
  Field f;
  f.name = name; f.ptr = p; f.dtype = B2_I32; f.n = n;
  if (second > 0) {
    f.ndim = 3; f.shape[0] = s->nworld; f.shape[1] = n / second; f.shape[2] = second;
    f.stride[0] = stride; f.stride[1] = second; f.stride[2] = 1;
  } else if (n == 1) {
    f.ndim = 1; f.shape[0] = s->nworld; f.stride[0] = stride;
  } else {
    f.ndim = 2; f.shape[0] = s->nworld; f.shape[1] = n; f.stride[0] = stride; f.stride[1] = 1;
  }
  s->data_fields.push_back(f);
  return 0;
}

static int launch(b2_sim* s, bool step, cudaStream_t st, int base = 0, int count = -1, int emit = 1) {
  if (count < 0) count = s->nworld;
  s->hd.emit = emit;
  s->hd.world_base = base;
  s->hd.world_count = count;
  const int grid = (count + B2_WARPS_PER_CTA - 1) / B2_WARPS_PER_CTA;
  if (step && s->sorted_dispatch && s->order && count >= 512 && s->hd.world_mask == nullptr) {
    b2_order_kernel<<<1, 1024, 0, st>>>(s->hd.solver_niter.p, s->hd.solver_niter.stride, s->hd.ncon.p,
                                        s->hd.ncon.stride, s->hd.solver_nd.p, s->hd.solver_nd.stride,
                                        s->hm.lay.ndcap, base, count, s->order);
    s->launches++;
    s->hd.world_order = s->order;
  } else {
    s->hd.world_order = nullptr;
  }
  // Phase-synchronous execution (CTA barriers at phase boundaries: instruction-cache locality, -14 % measured)
  // needs every warp of every CTA to own an environment (no early exits, no mask).
  s->hd.phase_sync = s->hd.world_mask == nullptr && count % B2_WARPS_PER_CTA == 0;
  if (step)
    if (s->has_convex) b2_step_kernel<3><<<grid, 32 * B2_WARPS_PER_CTA, s->smem_bytes, st>>>(s->hm, s->hd);
    else b2_step_kernel<1><<<grid, 32 * B2_WARPS_PER_CTA, s->smem_bytes, st>>>(s->hm, s->hd);
  else
    if (s->has_convex) b2_step_kernel<2><<<grid, 32 * B2_WARPS_PER_CTA, s->smem_bytes, st>>>(s->hm, s->hd);
    else b2_step_kernel<0><<<grid, 32 * B2_WARPS_PER_CTA, s->smem_bytes, st>>>(s->hm, s->hd);
  s->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

extern "C" {

const char* b2_last_error(void) { return g_err.c_str(); }
const char* b2_version(void) { return "b2sim 0.1.0 (sm_100a)"; }

// Debug builds (-DB2_PHASE_TIMING): cumulative per-phase cycles (sum over warps); reset on read.
int b2_phase_cycles(unsigned long long* out32) {
#ifdef B2_PHASE_TIMING
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out32, b2::g_phase_cycles, sizeof(unsigned long long) * 32);
  unsigned long long z[32] = {0};
  cudaMemcpyToSymbol(b2::g_phase_cycles, z, sizeof(z));
  return 0;
#else
  (void)out32;
  return 1;
#endif
}

// Sizes and index ranges of the model table (mjModel field names).  Returns "" when consistent.
static std::string validate_desc(const B2ModelDesc* desc) {
  std::map<std::string, const B2Array*> by;
  for (int i = 0; i < desc->narray; i++) {
    const B2Array& a = desc->arrays[i];
    if (!a.name || a.n < 0 || (a.n > 0 && !a.data)) return "array without name or data";
    if (a.dtype != B2_I32 && a.dtype != B2_F64) return std::string("array '") + a.name + "': dtype must be int32 or float64";
    by[a.name] = &a;
  }
  auto scalar = [&](const char* k, long long* out) -> bool {
    auto it = by.find(k);
    if (it == by.end() || it->second->n < 1) return false;
    *out = it->second->dtype == B2_I32 ? ((const int32_t*)it->second->data)[0] : (long long)((const double*)it->second->data)[0];
    return true;
  };
  long long nq, nv, nu, nbody, njnt, ngeom, nsite, nsensor, npair, nstatic = 0;
  if (!scalar("nq", &nq) || !scalar("nv", &nv) || !scalar("nu", &nu) || !scalar("nbody", &nbody) || !scalar("njnt", &njnt) ||
      !scalar("ngeom", &ngeom) || !scalar("nsite", &nsite) || !scalar("nsensor", &nsensor) || !scalar("npair", &npair))
    return "missing size scalar (nq nv nu nbody njnt ngeom nsite nsensor npair)";
  scalar("nstatic", &nstatic);
  if (nq < 1 || nv < 1 || nbody < 1 || nu < 0 || njnt < 0 || ngeom < 0 || nsite < 0 || nsensor < 0 || npair < 0 || nstatic < 0)
    return "negative or zero model size";
  struct Req { const char* name; int dtype; long long n; long long lo, hi; };  // index range checked for lo <= v < hi
  const long long NO = -(1ll << 40);
  std::vector<Req> req = {
    {"body_parentid", B2_I32, nbody, 0, nbody}, {"body_rootid", B2_I32, nbody, 0, nbody}, {"body_jntadr", B2_I32, nbody, -1, njnt},
    {"body_jntnum", B2_I32, nbody, 0, njnt + 1}, {"body_dofadr", B2_I32, nbody, -1, nv}, {"body_dofnum", B2_I32, nbody, 0, nv + 1},
    {"jnt_type", B2_I32, njnt, 0, 4}, {"jnt_qposadr", B2_I32, njnt, 0, nq}, {"jnt_dofadr", B2_I32, njnt, 0, nv},
    {"jnt_bodyid", B2_I32, njnt, 0, nbody}, {"jnt_limited", B2_I32, njnt, 0, 2}, {"dof_bodyid", B2_I32, nv, 0, nbody},
    {"dof_jntid", B2_I32, nv, 0, njnt}, {"dof_parentid", B2_I32, nv, -1, nv}, {"geom_type", B2_I32, ngeom, 0, 9},
    {"geom_bodyid", B2_I32, ngeom, 0, nbody}, {"geom_condim", B2_I32, ngeom, 1, 7}, {"geom_priority", B2_I32, ngeom, NO, -NO},
    {"site_bodyid", B2_I32, nsite, 0, nbody}, {"actuator_trnid", B2_I32, nu, 0, njnt},
    {"actuator_ctrllimited", B2_I32, nu, 0, 2}, {"actuator_forcelimited", B2_I32, nu, 0, 2},
    {"pair_geom1", B2_I32, npair, 0, ngeom}, {"pair_geom2", B2_I32, npair, 0, ngeom},
    {"sensor_objtype", B2_I32, nsensor, NO, -NO}, {"sensor_objid", B2_I32, nsensor, NO, -NO}, {"sensor_reftype", B2_I32, nsensor, NO, -NO},
    {"sensor_refid", B2_I32, nsensor, NO, -NO}, {"sensor_intprm", B2_I32, 3 * nsensor, NO, -NO}, {"sensor_adr", B2_I32, nsensor, 0, 1 << 20},
    {"sensor_dim", B2_I32, nsensor, 0, 1 << 20},
    {"body_pos", B2_F64, 3 * nbody}, {"body_quat", B2_F64, 4 * nbody}, {"body_ipos", B2_F64, 3 * nbody}, {"body_iquat", B2_F64, 4 * nbody},
    {"body_mass", B2_F64, nbody}, {"body_subtreemass", B2_F64, nbody}, {"body_inertia", B2_F64, 3 * nbody}, {"body_invweight0", B2_F64, 2 * nbody},
    {"jnt_pos", B2_F64, 3 * njnt}, {"jnt_axis", B2_F64, 3 * njnt}, {"jnt_range", B2_F64, 2 * njnt}, {"jnt_solref", B2_F64, 2 * njnt},
    {"jnt_solimp", B2_F64, 5 * njnt}, {"jnt_margin", B2_F64, njnt}, {"jnt_stiffness", B2_F64, njnt}, {"dof_armature", B2_F64, nv},
    {"dof_damping", B2_F64, nv}, {"dof_frictionloss", B2_F64, nv}, {"dof_invweight0", B2_F64, nv}, {"geom_size", B2_F64, 3 * ngeom},
    {"geom_pos", B2_F64, 3 * ngeom}, {"geom_quat", B2_F64, 4 * ngeom}, {"geom_friction", B2_F64, 3 * ngeom}, {"geom_solref", B2_F64, 2 * ngeom},
    {"geom_solimp", B2_F64, 5 * ngeom}, {"geom_solmix", B2_F64, ngeom}, {"geom_margin", B2_F64, ngeom}, {"geom_gap", B2_F64, ngeom},
    {"geom_rbound", B2_F64, ngeom}, {"geom_rgba", B2_F64, 4 * ngeom}, {"site_pos", B2_F64, 3 * nsite}, {"site_quat", B2_F64, 4 * nsite},
    {"actuator_gainprm", B2_F64, 10 * nu}, {"actuator_biasprm", B2_F64, 10 * nu}, {"actuator_ctrlrange", B2_F64, 2 * nu},
    {"actuator_forcerange", B2_F64, 2 * nu}, {"actuator_gear", B2_F64, nu}, {"qpos0", B2_F64, nq},
  };
  if (nstatic > 0) {
    req.push_back({"geom_contype", B2_I32, ngeom, NO, -NO});
    req.push_back({"geom_conaffinity", B2_I32, ngeom, NO, -NO});
    req.push_back({"static_geom", B2_I32, nstatic, 0, ngeom});
    req.push_back({"static_cell0", B2_I32, 2 * nstatic, 0, 1 << 20});
    req.push_back({"grid_params", B2_F64, 5});
  }
  for (const Req& r : req) {
    auto it = by.find(r.name);
    long long have = it == by.end() ? 0 : it->second->n;
    if (have != r.n) return std::string("array '") + r.name + "' has " + std::to_string(have) + " elements, expected " + std::to_string(r.n);
    if (r.n == 0) continue;
    if (it->second->dtype != r.dtype) return std::string("array '") + r.name + "' has the wrong dtype";
    if (r.dtype == B2_I32 && r.lo != NO) {
      const int32_t* v = (const int32_t*)it->second->data;
      for (long long i = 0; i < r.n; i++)
        if (v[i] < r.lo || v[i] >= r.hi) return std::string("array '") + r.name + "' holds an index out of range";
    }
  }
  for (const char* k : {"dyn_cgeom", "grid_items"}) {
    auto it = by.find(k);
    if (it == by.end()) continue;
    if (it->second->dtype != B2_I32) return std::string("array '") + k + "' has the wrong dtype";
    long long hi = std::string(k) == "dyn_cgeom" ? ngeom : nstatic;
    const int32_t* v = (const int32_t*)it->second->data;
    for (long long i = 0; i < it->second->n; i++)
      if (v[i] < 0 || v[i] >= hi) return std::string("array '") + k + "' holds an index out of range";
  }
  {  // parents precede children (the kinematic walks and the factorisation schedule rely on it)
    const int32_t* bp = (const int32_t*)by["body_parentid"]->data;
    for (long long b = 1; b < nbody; b++) if (bp[b] >= b) return "body_parentid: parents must precede children";
    const int32_t* dp = (const int32_t*)by["dof_parentid"]->data;
    for (long long d = 0; d < nv; d++) if (dp[d] >= d) return "dof_parentid: parents must precede children";
  }
  return "";
}

int b2_create(const B2ModelDesc* desc, int nworld, int ncon_per_world, int njmax, int cuda_device,
              b2_sim** out) {
  if (!desc || !out || nworld <= 0) return fail("b2_create: bad arguments");
  {
    std::string why = validate_desc(desc);  // host-only: a malformed table must not reach the index loops
    if (!why.empty()) return fail("b2_create: " + why);
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("b2_create: no CUDA device available (this library has no CPU path)");
  if (cuda_device < 0 || cuda_device >= ndev) return fail("b2_create: bad cuda_device");
  DeviceGuard guard(cuda_device);
  b2_sim* s = new b2_sim();
  s->device = cuda_device;
  s->nworld = nworld;
  for (int i = 0; i < desc->narray; i++) {
    const B2Array& a = desc->arrays[i];
    if (a.dtype == B2_I32) {
      s->mi[a.name] = std::vector<int>((const int32_t*)a.data, (const int32_t*)a.data + a.n);
    } else if (a.dtype == B2_F64) {
      s->mf[a.name] = std::vector<double>((const double*)a.data, (const double*)a.data + a.n);
    } else {
      delete s;
      return fail("b2_create: unsupported array dtype");
    }
  }
  auto geti = [&](const char* k) -> int {
    if (s->mi.count(k)) return s->mi[k].empty() ? 0 : s->mi[k][0];
    if (s->mf.count(k)) return (int)s->mf[k][0];
    return 0;
  };
  auto getf = [&](const char* k) -> double {
    if (s->mf.count(k)) return s->mf[k][0];
    if (s->mi.count(k)) return s->mi[k][0];
    return 0.0;
  };
  DevModel& m = s->hm;
  memset(&m, 0, sizeof(m));
  m.nq = geti("nq"); m.nv = geti("nv"); m.nu = geti("nu"); m.nbody = geti("nbody");
  m.njnt = geti("njnt"); m.ngeom = geti("ngeom"); m.nsite = geti("nsite");
  m.nsensor = geti("nsensor"); m.nsensordata = geti("nsensordata"); m.npair = geti("npair");
  m.ntri = m.nv * (m.nv + 1) / 2;
  if (m.nv > 64 || m.nbody > 64) { delete s; return fail("b2_create: nv and nbody must be <= 64"); }
  if (m.nv < 1) { delete s; return fail("b2_create: model has no degrees of freedom"); }
  m.integrator = geti("opt_integrator"); m.iterations = geti("opt_iterations");
  m.ls_iterations = geti("opt_ls_iterations");
  m.timestep = (float)getf("opt_timestep"); m.tolerance = (float)getf("opt_tolerance");
  m.ls_tolerance = (float)getf("opt_ls_tolerance"); m.impratio = (float)getf("opt_impratio");
  m.meaninertia = (float)getf("stat_meaninertia");
  for (int k = 0; k < 3; k++) m.gravity[k] = (float)desc->gravity[k];
  if (geti("opt_cone") != 0) { delete s; return fail("b2_create: only pyramidal cones are supported"); }
  m.solver = geti("opt_solver");
  if (m.solver != SOL_NEWTON_ && m.solver != SOL_CG_) {
    delete s;
    return fail("b2_create: solver must be Newton or CG (PGS works on the dual problem and is not implemented)");
  }
  m.maxcon = ncon_per_world > 0 ? std::min(ncon_per_world, 255) : 48;
  m.njmax = njmax > 0 ? njmax : 300;

  // ---- derived integer tables ---------------------------------------------------------------
  const std::vector<int>& parent = s->mi["body_parentid"];
  const std::vector<int>& dofadr = s->mi["body_dofadr"];
  const std::vector<int>& dofnum = s->mi["body_dofnum"];
  int nb = m.nbody;
  std::vector<int> depth(nb, 0);
  std::vector<unsigned long long> dofmask(nb, 0ull), ancmask(nb, 0ull);
  int maxdepth = 1;
  ancmask[0] = 1ull;
  for (int b = 1; b < nb; b++) {
    depth[b] = depth[parent[b]] + 1;
    maxdepth = std::max(maxdepth, depth[b]);
    dofmask[b] = dofmask[parent[b]];
    for (int k = 0; k < dofnum[b]; k++) dofmask[b] |= 1ull << (dofadr[b] + k);
    ancmask[b] = ancmask[parent[b]] | (1ull << b);
  }
  std::vector<int> chain((size_t)nb * maxdepth, 0);
  for (int b = 1; b < nb; b++) {
    int c = b;
    for (int k = depth[b] - 1; k >= 0; k--) { chain[(size_t)b * maxdepth + k] = c; c = parent[c]; }
  }
  m.maxdepth = maxdepth;
  std::vector<unsigned long long> submask(nb, 0ull), dofbody(std::max(m.nv, 1), 0ull);
  for (int d = 0; d < nb; d++)
    for (int a = 0; a < nb; a++)
      if (ancmask[d] >> a & 1ull) submask[a] |= 1ull << d;
  for (int b = 1; b < nb; b++)
    for (int i = 0; i < m.nv; i++)
      if (dofmask[b] >> i & 1ull) dofbody[i] |= 1ull << b;
  // compact kinematic records (fast path: every body has at most one joint)
  std::vector<float> kinrec((size_t)nb * 16, 0.f);
  int fastkin = 1;
  {
    const std::vector<int>& jn = s->mi["body_jntnum"]; const std::vector<int>& ja = s->mi["body_jntadr"];
    const std::vector<double>& bp = s->mf["body_pos"]; const std::vector<double>& bq = s->mf["body_quat"];
    const std::vector<double>& jp = s->mf["jnt_pos"]; const std::vector<double>& jax = s->mf["jnt_axis"];
    const std::vector<double>& q0 = s->mf["qpos0"];
    for (int b = 0; b < nb; b++) {
      if (jn[b] > 1) { fastkin = 0; break; }
      float* r = kinrec.data() + 16 * b;
      for (int k = 0; k < 3; k++) r[k] = (float)bp[3 * b + k];
      for (int k = 0; k < 4; k++) r[4 + k] = (float)bq[4 * b + k];
      int type = 0xff, j = 0, qa = 0;
      if (jn[b] == 1) {
        j = ja[b]; type = s->mi["jnt_type"][j]; qa = s->mi["jnt_qposadr"][j];
        for (int k = 0; k < 3; k++) { r[8 + k] = (float)jp[3 * j + k]; r[12 + k] = (float)jax[3 * j + k]; }
        r[3] = (float)q0[qa];
      }
      int tj = type | (j << 8);
      memcpy(&r[11], &tj, 4);
      memcpy(&r[15], &qa, 4);
    }
  }
  m.fastkin = fastkin;
  // World pose (pos[3], mat[9], rbound) of a geom on a jointless child of the world body, in double from world 0's
  // model values: such geoms never move, so they are posed here once and shared by all worlds.
  auto welded = [&](int g) { int b = s->mi["geom_bodyid"][g]; return b == 0 || (parent[b] == 0 && dofnum[b] == 0); };
  auto world_pose = [&](int g, float* o) {
    const std::vector<double>& bp = s->mf["body_pos"]; const std::vector<double>& bq = s->mf["body_quat"];
    const std::vector<double>& gp = s->mf["geom_pos"]; const std::vector<double>& gq = s->mf["geom_quat"];
    auto qmul = [](const double* a, const double* b, double* r) {
      r[0] = a[0]*b[0] - a[1]*b[1] - a[2]*b[2] - a[3]*b[3];
      r[1] = a[0]*b[1] + a[1]*b[0] + a[2]*b[3] - a[3]*b[2];
      r[2] = a[0]*b[2] - a[1]*b[3] + a[2]*b[0] + a[3]*b[1];
      r[3] = a[0]*b[3] + a[1]*b[2] - a[2]*b[1] + a[3]*b[0];
    };
    auto q2m = [](const double* q, double* R) {
      R[0] = q[0]*q[0] + q[1]*q[1] - q[2]*q[2] - q[3]*q[3]; R[1] = 2*(q[1]*q[2] - q[0]*q[3]); R[2] = 2*(q[1]*q[3] + q[0]*q[2]);
      R[3] = 2*(q[1]*q[2] + q[0]*q[3]); R[4] = q[0]*q[0] - q[1]*q[1] + q[2]*q[2] - q[3]*q[3]; R[5] = 2*(q[2]*q[3] - q[0]*q[1]);
      R[6] = 2*(q[1]*q[3] - q[0]*q[2]); R[7] = 2*(q[2]*q[3] + q[0]*q[1]); R[8] = q[0]*q[0] - q[1]*q[1] - q[2]*q[2] + q[3]*q[3];
    };
    const int b = s->mi["geom_bodyid"][g];
    double Rb[9], q[4], R[9];
    q2m(&bq[4 * b], Rb);
    qmul(&bq[4 * b], &gq[4 * g], q);
    double nq = std::sqrt(q[0]*q[0] + q[1]*q[1] + q[2]*q[2] + q[3]*q[3]);
    for (double& x : q) x /= nq;
    q2m(q, R);
    for (int i = 0; i < 3; i++)
      o[i] = (float)(bp[3 * b + i] + Rb[3 * i] * gp[3 * g] + Rb[3 * i + 1] * gp[3 * g + 1] + Rb[3 * i + 2] * gp[3 * g + 2]);
    for (int i = 0; i < 9; i++) o[3 + i] = (float)R[i];
    o[12] = (float)s->mf["geom_rbound"][g];
  };
  // Pose slots of the collision geoms in shared memory.  Height fields welded to the world (a terrain has tens of
  // them) get no slot: their pose records live in global memory (fixed_pose, slot code -2 - index) - 56 bytes of
  // shared memory per field and per environment otherwise, and a pose computation per step.
  std::vector<int> cslot(m.ngeom, -1), cgeom, fixed_geom;
  {
    std::vector<char> second(m.ngeom, 0);
    for (int p = 0; p < m.npair; p++) second[s->mi["pair_geom2"][p]] = 1;
    for (int p = 0; p < m.npair; p++) {
      for (int g : {s->mi["pair_geom1"][p], s->mi["pair_geom2"][p]}) {
        if (cslot[g] != -1) continue;
        if (s->mi["geom_type"][g] == G_HFIELD && !second[g] && welded(g)) { cslot[g] = -2 - (int)fixed_geom.size(); fixed_geom.push_back(g); }
        else { cslot[g] = (int)cgeom.size(); cgeom.push_back(g); }
      }
    }
  }
  m.nfixed = (int)fixed_geom.size();
  std::vector<float> fixed_pose((size_t)std::max(m.nfixed, 1) * 16, 0.f);
  for (int f = 0; f < m.nfixed; f++) world_pose(fixed_geom[f], fixed_pose.data() + 16 * (size_t)f);
  // grid-static collision set: static geoms never move, so their world poses are computed here once (in
  // double, from world 0's model values) and shared by all worlds; only the other geoms are posed per step
  m.nstatic = geti("nstatic");
  m.ndyn = (int)s->mi["dyn_cgeom"].size();
  std::vector<int> posegeom;
  std::vector<float> static_pose((size_t)std::max(m.nstatic, 1) * 16, 0.f);
  {
    std::vector<char> is_static(m.ngeom, 0);
    const std::vector<int>& sg = s->mi["static_geom"];
    if ((int)sg.size() != m.nstatic) { delete s; return fail("b2_create: static_geom / nstatic mismatch"); }
    if (m.nstatic >= (1 << 20) || m.ndyn >= (1 << 11)) { delete s; return fail("b2_create: static grid too large"); }
    for (int k = 0; k < m.nstatic; k++) {
      int g = sg[k], b = s->mi["geom_bodyid"][g];
      if (g < 0 || g >= m.ngeom || parent[b] != 0 || dofnum[b] != 0) {
        delete s;
        return fail("b2_create: grid-static geoms must sit on a jointless child of the world body");
      }
      is_static[g] = 1;
      world_pose(g, static_pose.data() + 16 * (size_t)k);
    }
    for (int g : fixed_geom) is_static[g] = 1;
    for (int g = 0; g < m.ngeom; g++) if (!is_static[g]) posegeom.push_back(g);
    m.nposegeom = (int)posegeom.size();
    for (int g : s->mi["dyn_cgeom"]) {
      if (g < 0 || g >= m.ngeom || is_static[g]) { delete s; return fail("b2_create: bad dyn_cgeom entry"); }
      if (cslot[g] < 0) { cslot[g] = (int)cgeom.size(); cgeom.push_back(g); }
    }
    if (m.nstatic > 0) {
      const std::vector<double>& gpar = s->mf["grid_params"];
      if (gpar.size() != 5) { delete s; return fail("b2_create: grid_params must hold [x0, y0, cell, nx, ny]"); }
      m.grid_x0 = (float)gpar[0]; m.grid_y0 = (float)gpar[1]; m.grid_cell = (float)gpar[2];
      m.grid_nx = (int)gpar[3]; m.grid_ny = (int)gpar[4];
      if ((int)s->mi["grid_start"].size() != m.grid_nx * m.grid_ny + 1 || (int)s->mi["static_cell0"].size() != 2 * m.nstatic) {
        delete s;
        return fail("b2_create: static grid tables have inconsistent sizes");
      }
    }
  }
  m.ncg = (int)cgeom.size();
  {  // every collision pair must have a narrowphase routine (primitives, or the convex routines of b2_convex.h)
    const std::vector<int>& gt = s->mi["geom_type"];
    auto prim = [](int t) { return t == G_SPHERE || t == G_CAPSULE || t == G_BOX; };
    auto smooth = [](int t) { return t == G_ELLIPSOID || t == G_CYLINDER; };
    auto conv = [&](int t) { return prim(t) || t == G_MESH || smooth(t); };  // shapes the GJK/EPA routine takes (b2_convex.h)
    const std::vector<int>& did = s->mi["geom_dataid"];
    const int nmesh = (int)s->mi["mesh_vertnum"].size(), nhf = (int)s->mi["hfield_nrow"].size();
    for (int p = 0; p < m.npair; p++) {
      int g1 = s->mi["pair_geom1"][p], g2 = s->mi["pair_geom2"][p];
      int t1 = gt[g1], t2 = gt[g2];
      bool ok = (t1 == G_PLANE && conv(t2)) || (t1 == G_HFIELD && conv(t2)) || (conv(t1) && conv(t2) && t1 <= t2);
      if (t2 == G_MESH || t1 == G_HFIELD || smooth(t1) || smooth(t2)) s->has_convex = 1;
      if (!ok) { delete s; return fail("b2_create: collision pair with an unsupported geom type combination"); }
      for (int g : {g1, g2}) {
        int t = gt[g];
        if (t != G_MESH && t != G_HFIELD) continue;
        int id = g < (int)did.size() ? did[g] : -1;
        if (id < 0 || id >= (t == G_MESH ? nmesh : nhf)) { delete s; return fail("b2_create: colliding mesh / hfield geom without asset data (geom_dataid)"); }
        if (t == G_MESH && (s->mi["mesh_vertnum"][id] < 1 || (size_t)3 * (s->mi["mesh_vertadr"][id] + s->mi["mesh_vertnum"][id]) > s->mf["mesh_vert"].size())) {
          delete s; return fail("b2_create: mesh vertex range outside mesh_vert");
        }
        if (t == G_HFIELD && (s->mi["hfield_nrow"][id] < 2 || s->mi["hfield_ncol"][id] < 2 || (size_t)4 * (id + 1) > s->mf["hfield_size"].size() ||
                              (size_t)s->mi["hfield_adr"][id] + (size_t)s->mi["hfield_nrow"][id] * s->mi["hfield_ncol"][id] > s->mf["hfield_data"].size())) {
          delete s; return fail("b2_create: hfield sample range outside hfield_data");
        }
      }
    }
    for (int g : s->mi["dyn_cgeom"]) {
      if (!conv(gt[g])) { delete s; return fail("b2_create: unsupported dynamic geom type for the static grid"); }
      if (gt[g] == G_MESH || smooth(gt[g])) s->has_convex = 1;
    }
    for (int g : s->mi["static_geom"]) if (!prim(gt[g])) { delete s; return fail("b2_create: unsupported grid-static geom type"); }
  }
  int rc = 0;
#define UPI(field, key) rc |= dev_upload<int>(s, s->mi[key], &m.field)
  UPI(body_parentid, "body_parentid"); UPI(body_rootid, "body_rootid"); UPI(body_jntadr, "body_jntadr");
  UPI(body_jntnum, "body_jntnum"); UPI(body_dofadr, "body_dofadr"); UPI(body_dofnum, "body_dofnum");
  UPI(jnt_type, "jnt_type"); UPI(jnt_qposadr, "jnt_qposadr"); UPI(jnt_dofadr, "jnt_dofadr");
  UPI(jnt_bodyid, "jnt_bodyid"); UPI(jnt_limited, "jnt_limited"); UPI(dof_bodyid, "dof_bodyid");
  UPI(dof_jntid, "dof_jntid"); UPI(dof_parentid, "dof_parentid"); UPI(geom_type, "geom_type");
  UPI(geom_bodyid, "geom_bodyid"); UPI(geom_condim, "geom_condim"); UPI(geom_priority, "geom_priority");
  UPI(site_bodyid, "site_bodyid"); UPI(actuator_trnid, "actuator_trnid");
  UPI(actuator_ctrllimited, "actuator_ctrllimited"); UPI(actuator_forcelimited, "actuator_forcelimited");
  UPI(pair_geom1, "pair_geom1"); UPI(pair_geom2, "pair_geom2"); UPI(sensor_objtype, "sensor_objtype");
  UPI(geom_contype, "geom_contype"); UPI(geom_conaffinity, "geom_conaffinity"); UPI(dyn_cgeom, "dyn_cgeom");
  UPI(static_geom, "static_geom"); UPI(static_cell0, "static_cell0"); UPI(grid_start, "grid_start");
  UPI(grid_items, "grid_items");
  UPI(geom_dataid, "geom_dataid"); UPI(mesh_vertadr, "mesh_vertadr"); UPI(mesh_vertnum, "mesh_vertnum");
  UPI(hfield_adr, "hfield_adr"); UPI(hfield_nrow, "hfield_nrow"); UPI(hfield_ncol, "hfield_ncol");
  UPI(sensor_objid, "sensor_objid"); UPI(sensor_reftype, "sensor_reftype");
  UPI(sensor_refid, "sensor_refid"); UPI(sensor_intprm, "sensor_intprm"); UPI(sensor_adr, "sensor_adr");
  UPI(sensor_dim, "sensor_dim");
#undef UPI
  rc |= dev_upload<int>(s, depth, &m.body_depth);
  rc |= dev_upload<int>(s, chain, &m.body_chain);
  rc |= dev_upload<unsigned long long>(s, dofmask, &m.body_dofmask);
  rc |= dev_upload<unsigned long long>(s, ancmask, &m.body_ancmask);
  rc |= dev_upload<unsigned long long>(s, submask, &m.body_submask);
  rc |= dev_upload<unsigned long long>(s, dofbody, &m.dof_bodymask);
  {
    const float* kr = nullptr;
    rc |= dev_upload<float>(s, kinrec, &kr);
    m.kinrec = (const float4*)kr;
  }
  for (auto kv : {std::make_pair("mesh_vert", &m.mesh_vert), std::make_pair("hfield_size", &m.hfield_size),
                  std::make_pair("hfield_data", &m.hfield_data)}) {
    const std::vector<double>& h = s->mf[kv.first];
    std::vector<float> hf(h.begin(), h.end());
    rc |= dev_upload<float>(s, hf, kv.second);
  }
  rc |= dev_upload<int>(s, posegeom, &m.posegeom);
  rc |= dev_upload<float>(s, static_pose, &m.static_pose);
  {
    if (m.ncg >= 4096) { b2_destroy(s); return fail("b2_create: too many collision geoms"); }
    std::vector<unsigned> pw(std::max(m.npair, 1), 0u);
    for (int p = 0; p < m.npair; p++) {
      int g1 = s->mi["pair_geom1"][p], g2 = s->mi["pair_geom2"][p];
      pw[p] = (unsigned)std::max(cslot[g1], 0) | ((unsigned)std::max(cslot[g2], 0) << 12) | (s->mi["geom_type"][g1] == G_PLANE ? 0x80000000u : 0u) |
              (s->mi["geom_type"][g1] == G_HFIELD ? 0x40000000u : 0u);
    }
    rc |= dev_upload<unsigned>(s, pw, &m.pair_word);
    // height-field pairs grouped by field: the kernel first finds the fields under the robot, then tests only
    // their pairs (a terrain is a grid of fields; the flat pair table would test every one of them)
    std::vector<int> hf_geom, hf_slot, hf_start, hf_pairs, hfd, nh;  // (hf_slot: pose slot, or -2 - index into fixed_pose)
    std::vector<std::vector<int>> per;
    std::vector<float> box;
    for (int p = 0; p < m.npair; p++) {
      int g1 = s->mi["pair_geom1"][p], g2 = s->mi["pair_geom2"][p];
      if (s->mi["geom_type"][g1] != G_HFIELD) { nh.push_back(p); continue; }
      size_t h = std::find(hf_geom.begin(), hf_geom.end(), g1) - hf_geom.begin();
      if (h == hf_geom.size()) {
        hf_geom.push_back(g1); hf_slot.push_back(cslot[g1]); per.emplace_back();
        const int id = s->mi["geom_dataid"][g1];
        for (int k = 0; k < 4; k++) box.push_back((float)s->mf["hfield_size"][4 * (size_t)id + k]);
      }
      per[h].push_back(p);
      if (std::find(hfd.begin(), hfd.end(), cslot[g2]) == hfd.end()) hfd.push_back(cslot[g2]);
    }
    m.nhf = (int)hf_geom.size(); m.nhfd = (int)hfd.size(); m.n_nhpair = m.npair;
    m.hfl_slot = m.hfl_geom = m.hfl_start = m.hfl_pairs = m.hfd_slot = m.nh_pairs = nullptr; m.hfl_box = nullptr;
    if (m.nhf > 0) {
      for (auto& v : per) { hf_start.push_back((int)hf_pairs.size()); hf_pairs.insert(hf_pairs.end(), v.begin(), v.end()); }
      hf_start.push_back((int)hf_pairs.size());
      m.n_nhpair = (int)nh.size();
      if (nh.empty()) nh.push_back(0);
      const float* bp = nullptr;
      rc |= dev_upload<int>(s, hf_slot, &m.hfl_slot); rc |= dev_upload<int>(s, hf_start, &m.hfl_start);
      rc |= dev_upload<int>(s, hf_geom, &m.hfl_geom);
      rc |= dev_upload<int>(s, hf_pairs, &m.hfl_pairs); rc |= dev_upload<int>(s, hfd, &m.hfd_slot);
      rc |= dev_upload<int>(s, nh, &m.nh_pairs); rc |= dev_upload<float>(s, box, &bp);
      m.hfl_box = (const float4*)bp;
    }
  }
  rc |= dev_upload<int>(s, cslot, &m.geom_cslot);
  rc |= dev_upload<float>(s, fixed_pose, &m.fixed_pose);
  if (fixed_geom.empty()) fixed_geom.push_back(0);
  rc |= dev_upload<int>(s, fixed_geom, &m.fixed_geom);
  rc |= dev_upload<int>(s, cgeom, &m.cgeom);
  {
    // schedules of the bottom-up blocked factorisation (b2_kernel.cuh: ldl_factor)
    std::vector<unsigned> dense, sparse;
    b2_build_ldl_schedules(m.nv, s->mi["dof_parentid"].data(), dense, sparse, m.ldl_start);
    m.ldl_nsparse = (int)sparse.size();
    rc |= dev_upload<unsigned>(s, dense, &m.ldl_dense);
    rc |= dev_upload<unsigned>(s, sparse, &m.ldl_sparse);
  }
  if (rc) { b2_destroy(s); return 1; }
  // supported sensor set: contact sensors with data in {found,force,dist,pos,normal}, reduce none/netforce
  for (int i = 0; i < m.nsensor; i++) {
    int ds = s->mi["sensor_intprm"][3 * i], rd = s->mi["sensor_intprm"][3 * i + 1];
    if ((ds & ~(1 | 2 | 8 | 16 | 32)) || (rd != 0 && rd != 3)) {
      b2_destroy(s);
      return fail("b2_create: contact sensor data/reduce combination not implemented");
    }
  }
  // int model fields visible to callers
  auto add_imodel = [&](const char* name, const int* p, int n) {
    Field f; f.name = name; f.ptr = (void*)p; f.dtype = B2_I32; f.ndim = 1; f.shape[0] = n; f.stride[0] = 1; f.n = n;
    s->model_fields.push_back(f);
  };
  add_imodel("geom_bodyid", m.geom_bodyid, m.ngeom); add_imodel("site_bodyid", m.site_bodyid, m.nsite);
  add_imodel("body_parentid", m.body_parentid, nb); add_imodel("body_rootid", m.body_rootid, nb);
  add_imodel("jnt_type", m.jnt_type, m.njnt); add_imodel("jnt_qposadr", m.jnt_qposadr, m.njnt);
  add_imodel("jnt_dofadr", m.jnt_dofadr, m.njnt); add_imodel("dof_bodyid", m.dof_bodyid, m.nv);
  add_imodel("geom_type", m.geom_type, m.ngeom); add_imodel("geom_condim", m.geom_condim, m.ngeom);
  add_imodel("geom_priority", m.geom_priority, m.ngeom);
  add_imodel("actuator_trnid", m.actuator_trnid, m.nu);

  // ---- float model arrays (fp32 on device; shared by all worlds until expanded) -----------------
  for (const ShapeSpec& sp : kModelShapes) {
    const std::vector<double>& h = s->mf[sp.name];
    std::vector<float> hf(h.begin(), h.end());
    const float* p = nullptr;
    if (dev_upload<float>(s, hf, &p)) { b2_destroy(s); return 1; }
    FArr* fa = model_farr(m, sp.name);
    fa->p = p; fa->stride = 0; fa->n = (int)hf.size();
    Field f; f.name = sp.name; f.ptr = (void*)p; f.dtype = B2_F32; f.farr = fa; f.n = (int64_t)hf.size();
    if (sp.second > 0) {
      f.ndim = 3; f.shape[0] = nworld; f.shape[1] = (int64_t)hf.size() / sp.second; f.shape[2] = sp.second;
      f.stride[0] = 0; f.stride[1] = sp.second; f.stride[2] = 1;
    } else {
      f.ndim = 2; f.shape[0] = nworld; f.shape[1] = (int64_t)hf.size(); f.stride[0] = 0; f.stride[1] = 1;
    }
    s->model_fields.push_back(f);
  }

  // ---- data -------------------------------------------------------------------------------------
  DevData& d = s->hd;
  memset(&d, 0, sizeof(d));
  d.nworld = nworld;
  int nq = m.nq, nv = m.nv, nu = m.nu, ng = m.ngeom, ns = m.nsite, mc = m.maxcon;
  rc = 0;
  rc |= add_data(s, "qpos", &d.qpos, nq); rc |= add_data(s, "qvel", &d.qvel, nv);
  rc |= add_data(s, "ctrl", &d.ctrl, nu); rc |= add_data(s, "qacc_warmstart", &d.qacc_warmstart, nv);
  rc |= add_data(s, "qfrc_applied", &d.qfrc_applied, nv);
  rc |= add_data(s, "xfrc_applied", &d.xfrc_applied, 6 * nb, 6);
  rc |= add_data(s, "act", &d.act, 0);
  rc |= add_data(s, "qacc", &d.qacc, nv); rc |= add_data(s, "xpos", &d.xpos, 3 * nb, 3);
  rc |= add_data(s, "xquat", &d.xquat, 4 * nb, 4); rc |= add_data(s, "xmat", &d.xmat, 9 * nb, 9);
  rc |= add_data(s, "xipos", &d.xipos, 3 * nb, 3); rc |= add_data(s, "subtree_com", &d.subtree_com, 3 * nb, 3);
  rc |= add_data(s, "cvel", &d.cvel, 6 * nb, 6); rc |= add_data(s, "geom_xpos", &d.geom_xpos, 3 * ng, 3);
  rc |= add_data(s, "geom_xmat", &d.geom_xmat, 9 * ng, 9); rc |= add_data(s, "site_xpos", &d.site_xpos, 3 * ns, 3);
  rc |= add_data(s, "site_xmat", &d.site_xmat, 9 * ns, 9);
  rc |= add_data(s, "link_vel_w", &d.link_vel_w, 6 * nb, 6); rc |= add_data(s, "com_vel_w", &d.com_vel_w, 6 * nb, 6);
  rc |= add_data(s, "link_state_b", &d.link_state_b, 10 * nb, 10);
  rc |= add_data(s, "sensordata", &d.sensordata, m.nsensordata);
  rc |= add_data(s, "actuator_force", &d.actuator_force, nu); rc |= add_data(s, "time", &d.time, 1);
  rc |= add_data(s, "qfrc_bias", &d.qfrc_bias, nv); rc |= add_data(s, "qfrc_smooth", &d.qfrc_smooth, nv);
  rc |= add_data(s, "qacc_smooth", &d.qacc_smooth, nv);
  rc |= add_data(s, "qfrc_constraint", &d.qfrc_constraint, nv);
  rc |= add_data(s, "qM", &d.qM, nv * nv, nv);
  rc |= add_data(s, "qM_packed", &d.qM_packed, m.ntri);
  rc |= add_data(s, "qacc_smooth_prev", &d.qacc_smooth_prev, nv);
  rc |= add_data(s, "ctrl_prev", &d.ctrl_prev, nu);
  rc |= add_data(s, "contact_dist", &d.contact_dist, mc); rc |= add_data(s, "contact_pos", &d.contact_pos, 3 * mc, 3);
  rc |= add_data(s, "contact_frame", &d.contact_frame, 9 * mc, 9);
  rc |= add_data(s, "contact_force", &d.contact_force, 3 * mc, 3);
  rc |= add_data(s, "solver_cost", &d.solver_cost, 1);
  rc |= add_idata(s, "ncon", &d.ncon, 1); rc |= add_idata(s, "nefc", &d.nefc, 1);
  rc |= add_idata(s, "solver_niter", &d.solver_niter, 1);
  rc |= add_idata(s, "contact_geom", &d.contact_geom, 2 * mc, 2);
  rc |= add_idata(s, "overflow", &d.overflow, 1);
  rc |= add_idata(s, "solver_nd", &d.solver_nd, 1);
  rc |= add_idata(s, "solver_nls", &d.solver_nls, 1);  // line-search derivative evaluations of the last step (diagnostic)
  if (rc) { b2_destroy(s); return 1; }
  // time is exposed as a 1-D (nworld,) tensor
  for (Field& f : s->data_fields)
    if (f.name == "time" || f.name == "solver_cost") { f.ndim = 1; }

  // ---- shared-memory layout (floats per environment) -------------------------------------------
  Layout& L = m.lay;
  int off = 0;
  auto alloc = [&](int n) { int o = off; off += pad4(std::max(n, 1)); return o; };
  L.maxcon = mc;
  L.nlimcap = pad4(std::max(m.njnt, 1));
  L.maxpair = m.nstatic > 0 ? 256 : 128;
  L.qpos = alloc(d.qpos.stride); L.qvel = alloc(d.qvel.stride); L.qacc_ws = alloc(d.qacc_warmstart.stride);
  L.cdof = alloc(7 * nv);
  int hsize = std::max(m.ntri, pad4(GP * m.ncg) + L.maxpair);
  L.H = alloc(hsize); L.gpose = L.H; L.pairlist = L.H + pad4(GP * m.ncg);
  L.invdiag = alloc(nv);
  L.qfrc_smooth = alloc(nv); L.qacc_smooth = alloc(nv); L.qacc = alloc(nv); L.Ma = alloc(nv);
  L.grad = alloc(nv); L.search = L.grad;  // search = -grad is formed in place
  L.Mv = alloc(nv); L.qfrc_c = alloc(nv); L.tmpv = alloc(nv);
  L.actf = alloc(nu);
  int ubase = off;
  // union A: regions that are dead once the smooth dynamics (phases 1-4) are done
  L.xpos = alloc(3 * nb); L.xquat = alloc(4 * nb); L.xipos = alloc(3 * nb); L.scom = alloc(3 * nb);
  L.cinert = alloc(11 * nb); L.crb = alloc(11 * nb);
  // joint anchors / axes are dead once the motion vectors exist (phase 2); cdofdot is first written in phase 4
  L.cdofdot = alloc(std::max(7 * nv, 2 * pad4(3 * m.njnt))); L.xanchor = L.cdofdot; L.xaxis = L.cdofdot + pad4(3 * m.njnt);
  L.cvel = alloc(7 * nb);
  L.cacc = alloc(7 * nb);
  int endA = off;
  off = ubase;
  // union B: constraint / solver regions
  L.contacts = alloc(C_NFIELD * mc); L.limits = alloc(L_NFIELD * L.nlimcap); L.gstart = alloc(mc + 1);
  // gV (group velocities / wrenches: J x, J^T f) and gu (Hessian projection) are never live together
  L.gV = alloc(std::max(6 * mc, 6 * nv)); L.gu = L.gV; L.glist = alloc(nv + 1); L.gA = alloc(36);
  L.gW = alloc(std::max(5 * mc, 4 * pad4(nv))); L.sens = off;  // (the CG variant keeps its four vectors here)
  // reduced Newton problem: room for the Schur complement on the largest leading block nv - 4k (k >= 1) whose
  // packed size fits 200 floats (G1: 19 x 19 = both legs + the first waist dof, 82 % of the bench workload's
  // environments; torso / arm contacts fall back to the full problem)
  L.ndcap = 0;
  for (int k = 1; nv - 4 * k >= 6; k++) {
    int cand = nv - 4 * k;
    if (cand * (cand + 1) / 2 <= 200) { L.ndcap = cand; break; }
  }
  L.Mred = alloc(L.ndcap * (L.ndcap + 1) / 2);
  int endB = off;
  // the lane-distributed height-field narrowphase keeps its owner records and its queue in the (then unused)
  // solver regions from gV on
  if (!s->mf["hfield_data"].empty()) endB = std::max(endB, L.gV + HF_SCRATCH);
  L.total = pad4(std::max(endA, endB));
  if (L.ndcap == 0) L.Mred = L.H;  // never used
  s->smem_bytes = sizeof(float) * ((size_t)L.total * B2_WARPS_PER_CTA + pad4(m.ldl_nsparse + 18));
  if (s->smem_bytes > 227 * 1024) {
    b2_destroy(s);
    return fail("b2_create: model too large for the per-environment shared-memory block");
  }
  {
    // The attribute is per function and per device, not per sim: only ever raise it, so that an earlier,
    // larger sim in the same process keeps launching after a smaller one is created.
    static size_t dev_max[64] = {0};
    if (s->smem_bytes > dev_max[cuda_device & 63]) {
      cudaError_t e1 = cudaFuncSetAttribute(b2_step_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes);
      cudaError_t e2 = cudaFuncSetAttribute(b2_step_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(b2_step_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes);
      if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(b2_step_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes);
      if (e1 != cudaSuccess || e2 != cudaSuccess) {
        b2_destroy(s);
        return fail(std::string("cudaFuncSetAttribute(max dynamic smem): ") + cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
      }
      dev_max[cuda_device & 63] = s->smem_bytes;
    }
  }
  {
    void* p = nullptr;
    if (cudaMalloc(&p, sizeof(int) * (size_t)nworld) != cudaSuccess) { b2_destroy(s); return fail("cudaMalloc(order)"); }
    s->allocs.push_back(p);
    s->order = (int*)p;
    for (int h = 0; h < B2_PARTITIONS; h++) {
      if (cudaStreamCreateWithFlags(&s->side[h], cudaStreamNonBlocking) != cudaSuccess ||
          cudaEventCreateWithFlags(&s->ev_join[h], cudaEventDisableTiming) != cudaSuccess) {
        b2_destroy(s);
        return fail("b2_create: stream/event creation failed");
      }
    }
    if (cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming) != cudaSuccess) { b2_destroy(s); return fail("event"); }
  }
  // qpos <- qpos0 in every world, then one forward pass so all derived fields are valid
  {
    long long total = (long long)nworld * nq;
    b2_init_rows_kernel<<<(unsigned)((total + 255) / 256), 256>>>(d.qpos.p, d.qpos.stride, m.qpos0.p, nq, nworld);
    s->launches++;
    if (m.nstatic > 0) {
      long long tot = (long long)nworld * m.nstatic;
      b2_static_rows_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(d.geom_xpos.p, d.geom_xpos.stride, d.geom_xmat.p,
                                                                     d.geom_xmat.stride, m.static_pose, m.static_geom,
                                                                     m.nstatic, nworld);
      s->launches++;
    }
    if (m.nfixed > 0) {
      long long tot = (long long)nworld * m.nfixed;
      b2_static_rows_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(d.geom_xpos.p, d.geom_xpos.stride, d.geom_xmat.p,
                                                                     d.geom_xmat.stride, m.fixed_pose, m.fixed_geom,
                                                                     m.nfixed, nworld);
      s->launches++;
    }
    if (launch(s, false, 0)) { b2_destroy(s); return 1; }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      std::string msg = std::string("b2_create: initial forward failed: ") + cudaGetErrorString(e);
      b2_destroy(s);
      return fail(msg);
    }
  }
  *out = s;
  return 0;
}

int b2_destroy(b2_sim* s) {
  if (!s) return 0;
  DeviceGuard guard(s->device);
  for (void* p : s->allocs) cudaFree(p);
  for (int h = 0; h < B2_PARTITIONS; h++) {
    if (s->side[h]) cudaStreamDestroy(s->side[h]);
    if (s->ev_join[h]) cudaEventDestroy(s->ev_join[h]);
  }
  if (s->ev_fork) cudaEventDestroy(s->ev_fork);
  delete s;
  return 0;
}

static Field* find_field(b2_sim* s, int which, const char* name) {
  std::vector<Field>& v = which == B2_DATA ? s->data_fields : s->model_fields;
  for (Field& f : v)
    if (f.name == name) return &f;
  return nullptr;
}
static void fill_tensor(b2_sim* s, const Field& f, B2Tensor* out) {
  out->ptr = f.ptr; out->dtype = f.dtype; out->ndim = f.ndim; out->device = s->device;
  for (int k = 0; k < 4; k++) { out->shape[k] = f.shape[k]; out->stride[k] = f.stride[k]; }
}

int b2_get_field(b2_sim* s, int which, const char* name, B2Tensor* out) {
  if (!s || !name || !out) return fail("b2_get_field: bad arguments");
  Field* f = find_field(s, which, name);
  if (!f) return fail(std::string("b2_get_field: unknown field '") + name + "'");
  fill_tensor(s, *f, out);
  return 0;
}
int b2_num_fields(b2_sim* s, int which) {
  return (int)(which == B2_DATA ? s->data_fields.size() : s->model_fields.size());
}
const char* b2_field_name(b2_sim* s, int which, int index) {
  std::vector<Field>& v = which == B2_DATA ? s->data_fields : s->model_fields;
  if (index < 0 || index >= (int)v.size()) return nullptr;
  return v[index].name.c_str();
}

int b2_expand_model_field(b2_sim* s, const char* name, void* stream, B2Tensor* out) {
  if (!s || !name) return fail("b2_expand_model_field: bad arguments");
  Field* f = find_field(s, B2_MODEL, name);
  if (!f || !f->farr) return fail(std::string("b2_expand_model_field: '") + name + "' is not an expandable model field");
  DeviceGuard guard(s->device);
  if (f->farr->stride == 0 && s->nworld > 1) {
    int n = f->farr->n;
    void* p = nullptr;
    long long total = (long long)s->nworld * n;
    CUDA_OK(cudaMalloc(&p, sizeof(float) * (size_t)total));
    s->allocs.push_back(p);
    b2_tile_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(f->farr->p, (float*)p, n, total);
    s->launches++;
    CUDA_OK(cudaGetLastError());
    f->farr->p = (const float*)p; f->farr->stride = n;
    {
      std::string nm = name;
      if (nm == "body_pos" || nm == "body_quat" || nm == "jnt_pos" || nm == "jnt_axis" || nm == "qpos0")
        s->hm.fastkin = 0;  // the compact kinematic records mirror the shared arrays only
    }
    f->ptr = p; f->stride[0] = n;
  }
  if (out) fill_tensor(s, *f, out);
  return 0;
}

int b2_set_option(b2_sim* s, const char* key, double v) {
  if (!s || !key) return fail("b2_set_option: bad arguments");
  std::string k = key;
  DevModel& m = s->hm;
  if (k == "iterations") m.iterations = (int)v;
  else if (k == "ls_iterations") m.ls_iterations = (int)v;
  else if (k == "tolerance") m.tolerance = (float)v;
  else if (k == "ls_tolerance") m.ls_tolerance = (float)v;
  else if (k == "timestep") m.timestep = (float)v;
  else if (k == "integrator") m.integrator = (int)v;
  else if (k == "solver") {
    if ((int)v != SOL_NEWTON_ && (int)v != SOL_CG_) return fail("b2_set_option: solver must be 1 (CG) or 2 (Newton)");
    m.solver = (int)v;
  }
  else if (k == "debug_outputs") m.debug = (m.debug & ~1) | ((int)v & 1);
  else if (k == "dense_factor") m.debug = (m.debug & ~2) | ((int)v ? 2 : 0);  // force the dense LDL schedule (tests)
  else if (k == "ls_parallel") { /* accepted for API parity; the line search here is exact */ }
  else if (k == "sorted_dispatch") s->sorted_dispatch = (int)v;
  else if (k == "full_solver") m.debug = (m.debug & ~4) | ((int)v ? 4 : 0);  // Newton on all dofs even when a leading block suffices (tests)
  else return fail("b2_set_option: unknown option '" + k + "'");
  return 0;
}
int b2_get_option(b2_sim* s, const char* key, double* v) {
  if (!s || !key || !v) return fail("b2_get_option: bad arguments");
  std::string k = key;
  const DevModel& m = s->hm;
  if (k == "iterations") *v = m.iterations;
  else if (k == "ls_iterations") *v = m.ls_iterations;
  else if (k == "tolerance") *v = m.tolerance;
  else if (k == "ls_tolerance") *v = m.ls_tolerance;
  else if (k == "timestep") *v = m.timestep;
  else if (k == "integrator") *v = m.integrator;
  else if (k == "solver") *v = m.solver;
  else if (k == "debug_outputs") *v = m.debug & 1;
  else if (k == "dense_factor") *v = (m.debug >> 1) & 1;
  else if (k == "smem_bytes_per_env") *v = 4.0 * m.lay.total;
  else if (k == "maxcon") *v = m.maxcon;
  else if (k == "full_solver") *v = (m.debug >> 2) & 1;
  else if (k == "reduced_block_cap") *v = m.lay.ndcap;
  else return fail("b2_get_option: unknown option '" + k + "'");
  return 0;
}

int b2_step(b2_sim* s, void* stream) {
  if (!s) return fail("b2_step: null sim");
  DeviceGuard guard(s->device);
  return launch(s, true, (cudaStream_t)stream);
}
int b2_forward(b2_sim* s, void* stream) {
  if (!s) return fail("b2_forward: null sim");
  DeviceGuard guard(s->device);
  return launch(s, false, (cudaStream_t)stream);
}
int b2_forward_masked(b2_sim* s, const unsigned char* world_mask_dev, void* stream) {
  if (!s) return fail("b2_forward_masked: null sim");
  DeviceGuard guard(s->device);
  s->hd.world_mask = world_mask_dev;
  int rc = launch(s, false, (cudaStream_t)stream);
  s->hd.world_mask = nullptr;
  return rc;
}
int b2_step_n(b2_sim* s, int n, void* stream) {
  if (!s) return fail("b2_step_n: null sim");
  DeviceGuard guard(s->device);
  if (n <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int np = B2_PARTITIONS;
  if (n > 1 && s->nworld >= 1024 * np) {
    // Environments are independent, so the sub-steps of one partition need not wait for the others:
    // fork the partitions onto internal streams (event fork/join, CUDA-graph capturable). Each
    // partition keeps per-sub-step launches (phase-aligned warps, fresh heavy-first order) while
    // its launch tails overlap the other partitions' work.
    int per = (((s->nworld + np - 1) / np + B2_WARPS_PER_CTA - 1) / B2_WARPS_PER_CTA) * B2_WARPS_PER_CTA;
    CUDA_OK(cudaEventRecord(s->ev_fork, st));
    for (int h = 0; h < np; h++) {
      int base = h * per, count = std::min(per, s->nworld - base);
      if (count <= 0) break;
      CUDA_OK(cudaStreamWaitEvent(s->side[h], s->ev_fork, 0));
      for (int i = 0; i < n; i++)
        if (launch(s, true, s->side[h], base, count, i == n - 1)) return 1;
      CUDA_OK(cudaEventRecord(s->ev_join[h], s->side[h]));
      CUDA_OK(cudaStreamWaitEvent(st, s->ev_join[h], 0));
    }
    return 0;
  }
  for (int i = 0; i < n; i++)
    if (launch(s, true, st, 0, -1, i == n - 1)) return 1;
  return 0;
}

int b2_velenv_pre(b2_sim* s, const float* action, const float* default_joint_pos,
                  const float* action_scale, void* stream) {
  if (!s || !action) return fail("b2_velenv_pre: bad arguments");
  DeviceGuard guard(s->device);
  long long total = (long long)s->nworld * s->hm.nu;
  if (total == 0) return 0;
  b2_velenv_pre_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      s->hd, s->hm.nu, action, default_joint_pos, action_scale);
  s->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int b2_velenv_post(b2_sim* s, const B2VelEnvArgs* args, void* stream) {
  if (!s || !args) return fail("b2_velenv_post: bad arguments");
  if (s->hm.nq != s->hm.nu + 7 || s->hm.nv != s->hm.nu + 6)
    return fail("b2_velenv_post: expects one floating base plus nu actuated hinge joints");
  DeviceGuard guard(s->device);
  b2_velenv_post_kernel<<<(s->nworld + 3) / 4, 128, 0, (cudaStream_t)stream>>>(  // one warp per environment
      s->hd, s->hm.nq, s->hm.nv, s->hm.nu, *args);
  s->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

static int trackenv_check(b2_sim* s, const B2TrackEnvArgs* a) {
  if (!s || !a) return fail("b2_trackenv: bad arguments");
  if (s->hm.nq != s->hm.nu + 7 || s->hm.nv != s->hm.nu + 6)
    return fail("b2_trackenv: expects one floating base plus nu actuated hinge joints");
  if (a->nb < 1 || a->nb > 32 || a->anchor < 0 || a->anchor >= a->nb || a->T < 2 || a->nee < 0 ||
      a->root_body < 0 || a->root_body >= s->hm.nbody || a->self_collision_adr < 0 ||
      a->self_collision_adr >= s->hm.nsensordata)
    return fail("b2_trackenv: bad sizes (1 <= nb <= 32 tracked bodies, anchor among them, T >= 2 clip frames)");
  return 0;
}
int b2_trackenv_post1(b2_sim* s, const B2TrackEnvArgs* args, void* stream) {
  if (trackenv_check(s, args)) return 1;
  DeviceGuard guard(s->device);
  b2_trackenv_post1_kernel<<<(s->nworld + 3) / 4, 128, 0, (cudaStream_t)stream>>>(s->hd, s->hm.nu, s->hm.nbody, *args);
  s->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}
int b2_trackenv_post2(b2_sim* s, const B2TrackEnvArgs* args, void* stream) {
  if (trackenv_check(s, args)) return 1;
  DeviceGuard guard(s->device);
  b2_trackenv_post2_kernel<<<(s->nworld + 3) / 4, 128, 0, (cudaStream_t)stream>>>(s->hd, s->hm.nu, s->hm.nbody, *args);
  s->launches++;
  CUDA_OK(cudaGetLastError());
  return 0;
}

int b2_step_host(b2_sim* s, const float* ctrl_host, int nsubstep, float* qpos_host, float* qvel_host,
                 void* stream) {
  if (!s) return fail("b2_step_host: null sim");
  DeviceGuard guard(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  const DevModel& m = s->hm; const DevData& d = s->hd;
  if (ctrl_host && m.nu > 0)
    CUDA_OK(cudaMemcpy2DAsync(d.ctrl.p, sizeof(float) * d.ctrl.stride, ctrl_host, sizeof(float) * m.nu,
                              sizeof(float) * m.nu, s->nworld, cudaMemcpyHostToDevice, st));
  if (nsubstep > 0 && b2_step_n(s, nsubstep, stream)) return 1;
  if (qpos_host)
    CUDA_OK(cudaMemcpy2DAsync(qpos_host, sizeof(float) * m.nq, d.qpos.p, sizeof(float) * d.qpos.stride,
                              sizeof(float) * m.nq, s->nworld, cudaMemcpyDeviceToHost, st));
  if (qvel_host)
    CUDA_OK(cudaMemcpy2DAsync(qvel_host, sizeof(float) * m.nv, d.qvel.p, sizeof(float) * d.qvel.stride,
                              sizeof(float) * m.nv, s->nworld, cudaMemcpyDeviceToHost, st));
  return 0;
}

int b2_stats(b2_sim* s, void* stream, B2Stats* out) {
  if (!s || !out) return fail("b2_stats: bad arguments");
  DeviceGuard guard(s->device);
  cudaStream_t st = (cudaStream_t)stream;
  const DevData& d = s->hd;
  size_t n = (size_t)s->nworld;
  std::vector<int> ncon(n * d.ncon.stride), nefc(n * d.nefc.stride), nit(n * d.solver_niter.stride), ovf(n * d.overflow.stride);
  CUDA_OK(cudaStreamSynchronize(st));
  CUDA_OK(cudaMemcpy(ncon.data(), d.ncon.p, sizeof(int) * ncon.size(), cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(nefc.data(), d.nefc.p, sizeof(int) * nefc.size(), cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(nit.data(), d.solver_niter.p, sizeof(int) * nit.size(), cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(ovf.data(), d.overflow.p, sizeof(int) * ovf.size(), cudaMemcpyDeviceToHost));
  memset(out, 0, sizeof(*out));
  out->ncon_cap = s->hm.maxcon; out->nefc_cap = s->hm.njmax;
  double sc = 0, se = 0, si = 0;
  for (size_t w = 0; w < n; w++) {
    int c = ncon[w * d.ncon.stride], e = nefc[w * d.nefc.stride], it = nit[w * d.solver_niter.stride];
    out->ncon_max = std::max(out->ncon_max, c); out->nefc_max = std::max(out->nefc_max, e);
    out->niter_max = std::max(out->niter_max, it);
    out->overflow_worlds += ovf[w * d.overflow.stride] ? 1 : 0;
    sc += c; se += e; si += it;
  }
  out->ncon_mean = sc / n; out->nefc_mean = se / n; out->niter_mean = si / n;
  return 0;
}

int64_t b2_launch_count(b2_sim* s) { return s ? s->launches : 0; }

int b2_algorithmic_bytes(b2_sim* s, void* stream, double* solver_bytes, double* step_bytes) {
  B2Stats st;
  if (b2_stats(s, stream, &st)) return 1;
  const DevModel& m = s->hm;
  double nv = m.nv, nefc = st.nefc_mean;
  // BASELINE.md §4 / SURVEY.md §8d: solver stage with J resident in HBM (the reference formulation)
  double solver = 4.0 * (nefc * nv + 3.0 * nefc + nv * nv + 5.0 * nv);
  // whole step: state in/out + consumer-visible kinematics (what this kernel actually moves)
  double in = m.nq + m.nv + m.nu + m.nv + m.nv + 6.0 * m.nbody;
  double outb = m.nq + 3.0 * m.nv + m.nu + m.nsensordata + (3 + 4 + 9 + 3 + 3 + 6) * (double)m.nbody +
                12.0 * m.nposegeom + 12.0 * m.nsite;  // geoms welded to the world are posed once at create, not per step
  if (solver_bytes) *solver_bytes = solver * s->nworld;
  if (step_bytes) *step_bytes = 4.0 * (in + outb) * s->nworld;
  return 0;
}

}  // extern "C"
