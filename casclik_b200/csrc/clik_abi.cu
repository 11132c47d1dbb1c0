// clik_abi.cu — host side of the C ABI declared in include/clik.h (libclik_b200.so).
//
// Loads the per-skill sm_100a cubin emitted by casclik_b200/codegen (CUDA runtime library API:
// cudaLibraryLoadData / cudaLibraryGetKernel), reads the image's manifest (sizes, optional kernels,
// input rows read), chooses the launch geometry (one CTA per block of instances; a balanced
// persistent grid for the opt-in TMA variant) and launches the fused controller-step kernels.
// No torch types, no Python; the static CUDA runtime loads libcuda lazily, so the library itself
// loads on a machine without a GPU and only the entry points that touch a device fail
// (CLIK_ERR_NOGPU / CLIK_ERR_CUDA).
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <cstdint>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/clik.h"
#include "clik_qp.cuh"

namespace clik { constexpr int PINV_TAIL_TILE = 1024; }   // = clik_pinv_group.cuh (not included here: it needs a Skill)

namespace {

thread_local std::string g_err;

clik_status fail(clik_status code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? CLIK_ERR_NOGPU \
                                                                               : CLIK_ERR_CUDA, \
                  "%s failed: %s", #call, cudaGetErrorString(e_));                            \
  } while (0)

// Every entry point runs on the skill's device and leaves the caller's current device as it found it
// (the caller may be torch, with its own idea of the current device).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
    if (prev != dev) err = cudaSetDevice(dev); else prev = -1;   // nothing to restore
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(dev)       \
  DeviceGuard guard_(dev);   \
  CK(guard_.err)

struct KernelInfo {
  cudaKernel_t kernel = nullptr;
  int grid = 0, block = 0, regs = 0, local_bytes = 0;
  int unroll = 1;    // instances per thread per grid-stride iteration (plain pinv kernel)
  int resident = 0;  // CTAs that fit on the device at once (SM count x occupancy)
};

// device scratch for the host-buffer pipeline (two slots, sized on demand)
constexpr int NSLOTS = 4;
struct Scratch {
  void* dev[NSLOTS] = {nullptr};
  size_t bytes[NSLOTS] = {0};
  cudaStream_t stream[NSLOTS] = {nullptr};
};

// input rows read by the compiled kernels (bit j = row j), exported by the cubin's size probe
struct ReadMask {
  unsigned t = 1u, q = 0xffffffffu, x = 0xffffffffu, y = 0xffffffffu;
};

}  // namespace

struct clik_skill {
  clik_skill_desc desc;
  cudaLibrary_t lib = nullptr;
  KernelInfo pinv, pinv_tma, pinv_rollout, pinv_fast, pinv_group, qp, qp_fast, qp_tail, qp_tail_capped, qp_rollout;
  KernelInfo nlp, nlp_rollout;   // NLP images (manifest flag 256)
  KernelInfo qp_duals, nlp_duals;   // constraint multipliers (manifest o[18]: bit 0 QP, bit 1 NLP; at most 32 rows)
  KernelInfo qp_vjp, nlp_vjp;       // reverse-mode derivative of the step (manifest o[19]: bit 0 QP, bit 1 NLP)
  bool qp_split = true;  // CLIK_QP_SPLIT=0: always the single full kernel
  int qp_tail_pick = -1; // CLIK_QP_TAIL_PICK: 0 always the uncapped tail kernel, 1 always the capped one, -1 by batch size
  bool pinv_split = true;     // CLIK_PINV_SPLIT=0: run-time mode tail inside the one kernel (thread mapping)
  bool pinv_group_all = false;  // CLIK_PINV_GROUP=1: whole batches through the sub-warp mapping (A/B measurements)
  int n_static = 1;           // statically compiled modes: where the group pass resumes the search
  ReadMask pinv_reads, qp_reads;   // (an NLP image reports its rows in the QP slots)
  bool use_tma = false;  // clik_skill_set_staging / CLIK_TMA=1: the TMA-staged persistent pinv kernel (device-resident batches)
  // programmatic dependent launch (clik_skill_set_overlap / CLIK_PDL): 0 = plain stream order,
  // 1 = the second launch of a two-launch step is scheduled while the first drains (it waits for the first
  // to complete before it reads), 2 = also the first launch of a step, i.e. successive steps on one stream
  // overlap tail and ramp — only for callers whose successive steps touch disjoint buffers
  int overlap = 1;
  int sm_count = 0;
  std::mutex mu;  // guards scratch and the single-instance slot
  Scratch scratch;
  // single-instance calls (the reference API's solve()): one page-locked, device-mapped slot holding the
  // inputs and outputs of one instance + a stream, so a call is: fill the slot, one launch, one wait
  double* one_host = nullptr;
  double* one_dev = nullptr;
  size_t one_doubles = 0;
  cudaStream_t one_stream = nullptr;
};

namespace {

// One launch; `dependent` adds the programmatic-stream-serialization attribute (the kernel side is in
// clik_math.cuh: griddepcontrol.launch_dependents at the start of every step kernel, griddepcontrol.wait
// before the first dependent read or as the last action).
cudaError_t launch(const KernelInfo& k, unsigned grid, void** args, cudaStream_t stream, bool dependent) {
  if (!dependent)
    return cudaLaunchKernel((const void*)k.kernel, dim3(grid), dim3(k.block), args, 0, stream);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(k.block);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelExC(&cfg, (const void*)k.kernel, args);
}

clik_status setup_kernel(clik_skill* s, const char* name, KernelInfo* k) {
  cudaError_t e = cudaLibraryGetKernel(&k->kernel, s->lib, name);
  if (e != cudaSuccess)
    return fail(CLIK_ERR_IMAGE, "cubin has no kernel %s: %s", name, cudaGetErrorString(e));
  cudaFuncAttributes attr;
  CK(cudaFuncGetAttributes(&attr, (const void*)k->kernel));
  k->regs = attr.numRegs;
  k->local_bytes = (int)attr.localSizeBytes;
  k->block = s->desc.block_threads > 0 ? s->desc.block_threads : 128;
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k->kernel, k->block, 0));
  if (per_sm < 1) per_sm = 1;
  k->resident = s->sm_count * per_sm;
  // grid cap = resident CTAs x waves.  waves = 1 is a persistent grid-stride launch; 0 lifts the
  // cap (one CTA per block_threads instances, hardware CTA scheduler balances the tail).
  int waves = 0;
  if (const char* w = getenv("CLIK_GRID_WAVES")) waves = atoi(w);
  k->grid = waves > 0 ? s->sm_count * per_sm * waves : 0x7fffffff;
  return CLIK_OK;
}

// Zero-copy host calls (kernel running on mapped host memory) may cap the grid: CTAs per SM of a grid-stride
// launch (0 = no cap).  Set around the launch by the host entry points.
thread_local int g_ctas_per_sm_cap = 0;
thread_local int g_sm_count = 0;

int grid_for(const KernelInfo& k, int64_t N) {
  const int64_t per_cta = (int64_t)k.block * k.unroll;
  int64_t need = (N + per_cta - 1) / per_cta;
  int64_t cap = k.grid;
  if (g_ctas_per_sm_cap > 0 && g_sm_count > 0) cap = std::min<int64_t>(cap, (int64_t)g_ctas_per_sm_cap * g_sm_count);
  return (int)std::max<int64_t>(1, std::min<int64_t>(need, cap));
}

// Persistent grid for the TMA-staged kernel: the fewest waves that cover all tiles, then the
// smallest grid that needs exactly that many waves, so every CTA walks the same number of tiles
// (+-1) and there is no ragged last wave.
int balanced_grid(const KernelInfo& k, int64_t N) {
  const int64_t tiles = (N + k.block - 1) / k.block;
  const int64_t waves = (tiles + k.resident - 1) / k.resident;
  return (int)std::max<int64_t>(1, (tiles + waves - 1) / waves);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

clik_status check_common(const clik_skill* s, int64_t N, const double* t, const double* q,
                         const double* x, const double* y) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  if (N < 0) return fail(CLIK_ERR_INVALID, "N < 0");
  if (N == 0) return CLIK_OK;
  if (!t || !q) return fail(CLIK_ERR_INVALID, "t and q are required");
  if (s->desc.n_virtual > 0 && !x) return fail(CLIK_ERR_INVALID, "skill has virtual_var: x is required");
  if (s->desc.n_input > 0 && !y) return fail(CLIK_ERR_INVALID, "skill reads input_var: y is required");
  return CLIK_OK;
}

// ---- dense QP kernel (the cs.conic call for numeric H/A/lb/ub) --------------------------------------
// Capacity tiers of the dense solver (working storage is per-thread local memory, so the larger tier is
// only instantiated for problems that need it).
template <int NXC, int MC>
__global__ void clik_qp_dense_kernel(long long N, int nx, int m, const double* __restrict__ h,
                                     const double* __restrict__ A, const double* __restrict__ lb,
                                     const double* __restrict__ ub, const double* __restrict__ x0,
                                     double* __restrict__ sol, int* __restrict__ status,
                                     unsigned* __restrict__ active, int max_iter) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    double Al[MC * NXC], lbl[MC], ubl[MC], hl[NXC], xs[NXC], x0l[NXC];
    for (int j = 0; j < nx; ++j) hl[j] = h[(long long)j * N + i];
    for (int r = 0; r < m; ++r) {
      lbl[r] = lb[(long long)r * N + i];
      ubl[r] = ub[(long long)r * N + i];
      for (int j = 0; j < nx; ++j) Al[r * nx + j] = A[(long long)(r * nx + j) * N + i];
    }
    if (x0) for (int j = 0; j < nx; ++j) x0l[j] = x0[(long long)j * N + i];
    unsigned mu, ml;
    int st = clik::qp_dual_active_set<NXC, MC>(nx, m, Al, lbl, ubl, hl, x0 ? x0l : nullptr, xs, &mu, &ml, max_iter);
    bool finite = true;
    for (int j = 0; j < nx; ++j) finite = finite && (fabs(xs[j]) < INFINITY);
    if (st == clik::QP_OK && !finite) st = clik::QP_INVALID;
    for (int j = 0; j < nx; ++j) sol[(long long)j * N + i] = xs[j];
    if (status) status[i] = st;
    if (active) { active[i] = mu; active[N + i] = ml; }
  }
}
constexpr int DENSE_NX = 16, DENSE_M = 32;          // tier 1
constexpr int DENSE_NX2 = 32, DENSE_M2 = 64;        // tier 2 (32 KB of local memory per thread)

// ---- measurement helpers -------------------------------------------------------------------------------
__global__ void dfma_peak_kernel(double* out, int iters, double a, double b) {
  // 8 independent dependent-chains per thread: enough ILP to saturate the fp64 pipe
  double x0 = threadIdx.x * 1e-9, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5,
         x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

__global__ void fill_kernel(double* p, size_t n, double v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    p[i] = v;
}

std::mutex g_flush_mu;
double* g_flush_buf[64] = {nullptr};
constexpr size_t FLUSH_BYTES = (size_t)256 << 20;  // 256 MiB > 126 MB L2

// ---- host-buffer calls ---------------------------------------------------------------------------------
// One array of a host call: the caller's pointer and how it reaches the device.
enum Dir { IN, OUT };
struct HostField {
  const void* host;                // caller's array (rows N apart); nullptr or rows == 0: absent
  Dir dir;                         // IN: read by the kernel; OUT: written by it
  int rows;                        // SoA rows
  int elem;                        // bytes per element
  bool broadcast = false;          // one value for every instance (t with t_stride 0)
  unsigned rowmask = 0xffffffffu;  // input rows the kernel reads (unread rows are not copied)
};

// A device pointer that converts to whatever pointer type the *_impl parameter it is passed to has.
struct DevPtr {
  void* p = nullptr;
  template <class T> operator T*() const { return static_cast<T*>(p); }
};

clik_status ensure_scratch(clik_skill* s, int slot, size_t bytes) {
  Scratch& sc = s->scratch;
  if (!sc.stream[slot]) CK(cudaStreamCreateWithFlags(&sc.stream[slot], cudaStreamNonBlocking));
  if (sc.bytes[slot] < bytes) {
    if (sc.dev[slot]) CK(cudaFree(sc.dev[slot]));
    sc.dev[slot] = nullptr;
    sc.bytes[slot] = 0;
    CK(cudaMalloc(&sc.dev[slot], bytes));
    sc.bytes[slot] = bytes;
  }
  return CLIK_OK;
}

// Chunk size of the host pipeline: small enough that H2D of chunk k+1, the kernel of chunk k and
// D2H of chunk k-1 overlap (both copy engines busy), large enough to amortise launch overheads.
int64_t host_chunk() {
  static int64_t v = [] {
    const char* e = getenv("CLIK_HOST_CHUNK");
    int64_t c = e ? atoll(e) : (1 << 17);
    return c < 1024 ? (int64_t)1024 : c;
  }();
  return v;
}

// Page-locked host memory (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory()) is mapped into
// the device address space under UVA.  If every buffer of a host call is such memory, the kernel
// runs directly on it: the SMs stream the inputs over PCIe and write the results back, both
// directions at once, with no staging copies (measured 6.4e8 vs 5.6e8 steps/s for the headline
// skill).  Returns false (-> staged pipeline) for ordinary pageable memory.
bool device_alias(const void* host, const void** dev) {
  if (host == nullptr) { *dev = nullptr; return true; }
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) { cudaGetLastError(); return false; }
  if (a.type != cudaMemoryTypeHost || a.devicePointer == nullptr) return false;
  *dev = a.devicePointer;
  return true;
}

// CLIK_ZC_STAGED=1: let the zero-copy path use the staged kernel too (bulk async copies straight from the
// mapped host arrays) when the skill has staging switched on
bool zero_copy_staged() {
  static bool v = [] { const char* e = getenv("CLIK_ZC_STAGED"); return e != nullptr && atoi(e) != 0; }();
  return v;
}

// Grid of a kernel that runs directly on mapped host memory: a grid-stride launch of 2 CTAs per SM instead of
// one CTA per 128 instances.  With ~1200 CTAs resident the 8 input rows are read at ~1200 scattered places at
// once; with 296 the requests the host sees are far more sequential: 6.2e8 -> 7.0e8 steps/s end to end for the
// tracking skill, 94 % of what two concurrent memcpys reach on this box (profiles/r2_ab18.txt).
// CLIK_ZC_CTAS_PER_SM overrides (0 = no cap).
int zero_copy_ctas_per_sm() {
  static int v = [] { const char* e = getenv("CLIK_ZC_CTAS_PER_SM"); return e ? atoi(e) : 2; }();
  return v;
}
struct GridCapScope {
  GridCapScope(int cap, int sms) { g_ctas_per_sm_cap = cap; g_sm_count = sms; }
  ~GridCapScope() { g_ctas_per_sm_cap = 0; }
};

bool zero_copy_enabled() {
  static bool v = [] { const char* e = getenv("CLIK_ZERO_COPY"); return e == nullptr || atoi(e) != 0; }();
  return v;
}

// copy the rows selected by `mask` as maximal runs of consecutive rows
template <class Copy>
clik_status for_row_runs(int rows, unsigned mask, Copy copy) {
  int r = 0;
  while (r < rows) {
    if (r < 32 && !((mask >> r) & 1u)) { ++r; continue; }
    int e = r + 1;
    while (e < rows && (e >= 32 || ((mask >> e) & 1u))) ++e;
    clik_status st = copy(r, e - r);
    if (st != CLIK_OK) return st;
    r = e;
  }
  return CLIK_OK;
}

// Instances [lo, lo + cnt) of a host batch whose rows are N apart (lo = 0, cnt = N: the whole batch), one
// HostField per array.  If every present array is page-locked memory mapped into the device, one launch runs on it
// directly (zero copy); otherwise the instances go through the chunked copy pipeline on the skill's scratch slots.
// `launch(p, n, ld, stream, zero_copy)` launches the step on n instances whose rows are ld apart, p[k] the device
// pointer of field k (nullptr exactly when the field is absent).  Returns once the results are in the host arrays.
template <size_t NF, class Launch>
clik_status run_host_batch(clik_skill* s, int64_t N, int64_t lo, int64_t cnt, const std::array<HostField, NF>& f,
                           Launch launch) {
  if (cnt <= 0) return CLIK_OK;
  std::lock_guard<std::mutex> lock(s->mu);
  ON_DEVICE(s->desc.device);
  std::array<DevPtr, NF> p;
  auto present = [&](size_t k) { return f[k].host != nullptr && f[k].rows > 0; };
  bool zero_copy = zero_copy_enabled();
  for (size_t k = 0; k < NF && zero_copy; ++k) {
    const void* dev = nullptr;
    zero_copy = device_alias(present(k) ? f[k].host : nullptr, &dev);
    if (dev && !f[k].broadcast) dev = (const char*)dev + lo * f[k].elem;
    p[k].p = const_cast<void*>(dev);
  }
  if (zero_copy) {
    clik_status st = ensure_scratch(s, 0, 256);
    if (st != CLIK_OK) return st;
    GridCapScope cap(zero_copy_ctas_per_sm(), s->sm_count);
    st = launch(p, cnt, N, s->scratch.stream[0], true);
    if (st != CLIK_OK) return st;
    CK(cudaStreamSynchronize(s->scratch.stream[0]));
    return CLIK_OK;
  }
  const int64_t chunk = std::min<int64_t>(cnt, host_chunk());
  size_t off[NF], bytes = 0;
  for (size_t k = 0; k < NF; ++k) {
    off[k] = bytes;
    bytes += (((size_t)f[k].rows * chunk * f[k].elem) + 255) & ~(size_t)255;
  }
  const int nslots = (int)std::min<int64_t>(NSLOTS, (cnt + chunk - 1) / chunk);
  for (int slot = 0; slot < nslots; ++slot) {
    clik_status st = ensure_scratch(s, slot, bytes);
    if (st != CLIK_OK) return st;
  }
  int slot = 0;
  for (int64_t i0 = lo; i0 < lo + cnt; i0 += chunk, slot = (slot + 1) % nslots) {
    const int64_t c = std::min<int64_t>(chunk, lo + cnt - i0);
    cudaStream_t st = s->scratch.stream[slot];
    char* base = (char*)s->scratch.dev[slot];
    for (size_t k = 0; k < NF; ++k) {
      const HostField& fl = f[k];
      p[k].p = present(k) ? base + off[k] : nullptr;
      if (!present(k) || fl.dir != IN) continue;
      if (fl.broadcast) {
        if (fl.rowmask & 1u) CK(cudaMemcpyAsync(p[k].p, fl.host, fl.elem, cudaMemcpyHostToDevice, st));
        continue;
      }
      clik_status cs = for_row_runs(fl.rows, fl.rowmask, [&](int r0, int nr) -> clik_status {
        CK(cudaMemcpy2DAsync(base + off[k] + (size_t)r0 * c * fl.elem, (size_t)c * fl.elem,
                             (const char*)fl.host + ((size_t)r0 * N + (size_t)i0) * fl.elem,
                             (size_t)N * fl.elem, (size_t)c * fl.elem, nr, cudaMemcpyHostToDevice, st));
        return CLIK_OK;
      });
      if (cs != CLIK_OK) return cs;
    }
    clik_status ls = launch(p, c, c, st, false);
    if (ls != CLIK_OK) return ls;
    for (size_t k = 0; k < NF; ++k) {
      const HostField& fl = f[k];
      if (!present(k) || fl.dir != OUT) continue;
      CK(cudaMemcpy2DAsync((char*)fl.host + (size_t)i0 * fl.elem, (size_t)N * fl.elem, base + off[k],
                           (size_t)c * fl.elem, (size_t)c * fl.elem, fl.rows, cudaMemcpyDeviceToHost, st));
    }
  }
  for (int k = 0; k < nslots; ++k) CK(cudaStreamSynchronize(s->scratch.stream[k]));
  return CLIK_OK;
}

}  // namespace

extern "C" {

const char* clik_last_error(void) { return g_err.c_str(); }
int32_t clik_abi_version(void) { return CLIK_ABI_VERSION; }

int32_t clik_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

clik_status clik_skill_load(const void* cubin, size_t len, const clik_skill_desc* desc,
                            clik_skill** out) {
  if (!cubin || len == 0 || !desc || !out) return fail(CLIK_ERR_INVALID, "NULL argument");
  if (desc->abi_version != CLIK_ABI_VERSION)
    return fail(CLIK_ERR_INVALID, "descriptor ABI version %d != library %d", desc->abi_version,
                CLIK_ABI_VERSION);
  if (desc->n_robot <= 0) return fail(CLIK_ERR_INVALID, "n_robot must be positive");
  *out = nullptr;
  ON_DEVICE(desc->device);
  clik_skill* s = new clik_skill();
  s->desc = *desc;
  cudaError_t e = cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, desc->device);
  if (e == cudaSuccess) e = cudaLibraryLoadData(&s->lib, cubin, nullptr, nullptr, 0, nullptr, nullptr, 0);
  if (e != cudaSuccess) {
    delete s;
    return fail(CLIK_ERR_IMAGE, "cannot load cubin (%zu bytes): %s", len, cudaGetErrorString(e));
  }
  // The image carries its own manifest (clik_sizes_kernel): sizes, which optional kernels it
  // holds, and which input rows its kernels read.  Refuse a descriptor that disagrees.
  clik_status st = CLIK_OK;
  int hsz[24] = {0};
  {
    cudaKernel_t probe;
    cudaError_t pe = cudaLibraryGetKernel(&probe, s->lib, "clik_sizes_kernel");
    if (pe != cudaSuccess) {
      st = fail(CLIK_ERR_IMAGE, "cubin has no clik_sizes_kernel manifest: %s", cudaGetErrorString(pe));
    } else {
      int* dsz = nullptr;
      cudaError_t le = cudaMalloc(&dsz, sizeof(hsz));
      // slots an image does not write (o[18], o[19] of older or pinv-only images) must read 0, not whatever the
      // allocation held before
      if (le == cudaSuccess) le = cudaMemset(dsz, 0, sizeof(hsz));
      if (le == cudaSuccess) {
        void* args[] = {&dsz};
        le = cudaLaunchKernel((const void*)probe, dim3(1), dim3(1), args, 0, nullptr);
        if (le == cudaSuccess) le = cudaMemcpy(hsz, dsz, sizeof(hsz), cudaMemcpyDeviceToHost);
        cudaFree(dsz);
      }
      if (le != cudaSuccess) {
        st = fail(CLIK_ERR_CUDA, "size probe failed: %s", cudaGetErrorString(le));
      } else if (hsz[0] != desc->n_robot || hsz[1] != desc->n_virtual || hsz[2] != desc->n_input ||
                 hsz[3] != desc->n_modes || hsz[4] != desc->qp_n || hsz[5] != desc->qp_m) {
        st = fail(CLIK_ERR_IMAGE,
                  "descriptor does not match cubin: image (n_robot %d, n_virtual %d, n_input %d, "
                  "n_modes %d, qp %dx%d)",
                  hsz[0], hsz[1], hsz[2], hsz[3], hsz[5], hsz[4]);
      }
    }
  }
  const int flags = hsz[7];   // bit 0: pinv TMA variant, bit 1: pinv rollout, bit 2: QP rollout
  if (st == CLIK_OK && desc->has_pinv) st = setup_kernel(s, "clik_pinv_kernel", &s->pinv);
  if (st == CLIK_OK && desc->has_pinv) {
    s->pinv.unroll = hsz[6] > 0 ? hsz[6] : 1;
    s->pinv_reads = ReadMask{(unsigned)hsz[8], (unsigned)hsz[9], (unsigned)hsz[10], (unsigned)hsz[11]};
    if (flags & 1) st = setup_kernel(s, "clik_pinv_tma_kernel", &s->pinv_tma);
    if (const char* e = getenv("CLIK_TMA")) s->use_tma = atoi(e) != 0;
    if (st == CLIK_OK && (flags & 2)) st = setup_kernel(s, "clik_pinv_rollout_kernel", &s->pinv_rollout);
    if (st == CLIK_OK && (flags & 64)) st = setup_kernel(s, "clik_pinv_fast_kernel", &s->pinv_fast);
    if (st == CLIK_OK && (flags & 32)) {
      st = setup_kernel(s, "clik_pinv_group_kernel", &s->pinv_group);
      s->pinv_group.block = hsz[17] > 0 ? hsz[17] : 64;
    }
    if (st == CLIK_OK) s->pinv_fast.unroll = s->pinv.unroll;
    s->n_static = hsz[16] > 0 ? hsz[16] : 1;
    if (const char* e = getenv("CLIK_PINV_SPLIT")) s->pinv_split = atoi(e) != 0;
    if (const char* e = getenv("CLIK_PINV_GROUP")) s->pinv_group_all = atoi(e) != 0;
  }
  if (st == CLIK_OK && desc->has_qp) st = setup_kernel(s, "clik_qp_kernel", &s->qp);
  if (st == CLIK_OK && desc->has_qp) {
    s->qp_reads = ReadMask{(unsigned)hsz[12], (unsigned)hsz[13], (unsigned)hsz[14], (unsigned)hsz[15]};
    if (flags & 4) st = setup_kernel(s, "clik_qp_rollout_kernel", &s->qp_rollout);
    if (st == CLIK_OK && (flags & 16)) st = setup_kernel(s, "clik_qp_fast_kernel", &s->qp_fast);
    if (st == CLIK_OK && (flags & 16)) st = setup_kernel(s, "clik_qp_tail_kernel", &s->qp_tail);
    if (st == CLIK_OK && (flags & 128)) st = setup_kernel(s, "clik_qp_tail_capped_kernel", &s->qp_tail_capped);
    if (const char* e = getenv("CLIK_QP_TAIL_PICK")) s->qp_tail_pick = atoi(e);
    if (const char* e = getenv("CLIK_QP_SPLIT")) s->qp_split = atoi(e) != 0;
  }
  if (st == CLIK_OK && (flags & 256)) {
    s->qp_reads = ReadMask{(unsigned)hsz[12], (unsigned)hsz[13], (unsigned)hsz[14], (unsigned)hsz[15]};
    st = setup_kernel(s, "clik_nlp_kernel", &s->nlp);
    if (st == CLIK_OK) st = setup_kernel(s, "clik_nlp_rollout_kernel", &s->nlp_rollout);
  }
  const int duals = hsz[18];   // multiplier kernels: bit 0 QP, bit 1 NLP
  if (st == CLIK_OK && (duals & 1)) st = setup_kernel(s, "clik_qp_duals_kernel", &s->qp_duals);
  if (st == CLIK_OK && (duals & 2)) st = setup_kernel(s, "clik_nlp_duals_kernel", &s->nlp_duals);
  const int vjp = hsz[19];     // VJP kernels (images built with emit_skill(..., vjp=True)): bit 0 QP, bit 1 NLP
  if (st == CLIK_OK && (vjp & 1)) st = setup_kernel(s, "clik_qp_vjp_kernel", &s->qp_vjp);
  if (st == CLIK_OK && (vjp & 2)) st = setup_kernel(s, "clik_nlp_vjp_kernel", &s->nlp_vjp);
  if (st != CLIK_OK) {
    cudaLibraryUnload(s->lib);
    delete s;
    return st;
  }
  if (const char* e = getenv("CLIK_PDL")) s->overlap = std::max(0, std::min(2, atoi(e)));
  *out = s;
  return CLIK_OK;
}

clik_status clik_skill_set_overlap(clik_skill* s, int32_t level) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  if (level < 0 || level > 2) return fail(CLIK_ERR_INVALID, "overlap level %d (0, 1 or 2)", (int)level);
  s->overlap = level;
  return CLIK_OK;
}

int32_t clik_skill_get_overlap(const clik_skill* s) { return s ? s->overlap : -1; }

clik_status clik_skill_set_staging(clik_skill* s, int32_t on) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  if (on && !s->pinv_tma.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the staged pinv kernel");
  s->use_tma = on != 0;
  return CLIK_OK;
}

int32_t clik_skill_get_staging(const clik_skill* s) { return s ? (s->use_tma && s->pinv_tma.kernel ? 1 : 0) : -1; }

void clik_skill_free(clik_skill* s) {
  if (!s) return;
  DeviceGuard guard(s->desc.device);
  if (s->one_host) cudaFreeHost(s->one_host);
  if (s->one_stream) cudaStreamDestroy(s->one_stream);
  for (int i = 0; i < NSLOTS; ++i) {
    if (s->scratch.dev[i]) cudaFree(s->scratch.dev[i]);
    if (s->scratch.stream[i]) cudaStreamDestroy(s->scratch.stream[i]);
  }
  if (s->lib) cudaLibraryUnload(s->lib);
  delete s;
}

clik_status clik_skill_launch_info(const clik_skill* s, int32_t which, int32_t* grid, int32_t* block,
                                   int32_t* regs, int32_t* local_bytes) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  const KernelInfo& k = which == 0 ? s->pinv : which == 2 ? s->pinv_tma : which == 3 ? s->qp_fast : which == 4 ? s->qp_tail
                        : which == 5 ? s->pinv_fast : which == 6 ? s->pinv_group : which == 7 ? s->qp_tail_capped : s->qp;
  if (!k.kernel) return fail(CLIK_ERR_INVALID, "skill has no such kernel");
  if (grid) *grid = k.grid;
  if (block) *block = k.block;
  if (regs) *regs = k.regs;
  if (local_bytes) *local_bytes = k.local_bytes;
  return CLIK_OK;
}

}  // extern "C"

namespace {
// `level`: overlap level of this call (the public entry points pass the skill's; the host-buffer pipelines,
// which order copies and kernels on their own streams, never more than 1)
clik_status pinv_step_impl(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                           const double* q, const double* x, const double* y, double* qdot,
                           double* xdot, int32_t* mode, void* stream, int level, bool staged_ok = true,
                           bool split_ok = true) {
  clik_status st = check_common(s, N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (ld < N) return fail(CLIK_ERR_INVALID, "row stride ld (%lld) < N (%lld)", (long long)ld, (long long)N);
  if (!s->pinv.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the pinv kernel");
  if (!qdot) return fail(CLIK_ERR_INVALID, "qdot is required");
  if (s->desc.n_virtual > 0 && !xdot) return fail(CLIK_ERR_INVALID, "xdot is required");
  ON_DEVICE(s->desc.device);
  long long n = N, l = ld;
  int ts = t_stride ? 1 : 0;
  void* args[] = {&n, &l, &t, &ts, &q, &x, &y, &qdot, &xdot, &mode};
  // bulk async copies need 16-byte aligned row segments: even stride and aligned bases
  const bool tma_ok = staged_ok && s->use_tma && s->pinv_tma.kernel && (ld % 2 == 0) && aligned16(t) && aligned16(q) &&
                      aligned16(x) && aligned16(y);
  const int64_t tiles = (N + clik::PINV_TAIL_TILE - 1) / clik::PINV_TAIL_TILE;
  const bool within = level >= 1, across = level >= 2;
  if (s->pinv_group_all && s->pinv_group.kernel) {
    // the whole step in the sub-warp mapping (from mode 0, every instance)
    int from = 0, pending_only = 0;
    void* gargs[] = {&n, &l, &t, &ts, &q, &x, &y, &qdot, &xdot, &mode, &from, &pending_only};
    CK(launch(s->pinv_group, (unsigned)std::min<int64_t>(tiles, 1 << 20), gargs, (cudaStream_t)stream, across));
  } else if (split_ok && s->pinv_split && s->pinv_fast.kernel && s->pinv_group.kernel && mode != nullptr) {
    // two launches: statically compiled modes for every instance (thread mapping, registers), then the
    // run-time tail of the activation map for the instances they all rejected (sub-warp mapping);
    // handed over through mode[] (transient value PINV_PENDING)
    CK(launch(s->pinv_fast, grid_for(s->pinv_fast, N), args, (cudaStream_t)stream, across));
    int from = s->n_static, pending_only = 1;
    void* gargs[] = {&n, &l, &t, &ts, &q, &x, &y, &qdot, &xdot, &mode, &from, &pending_only};
    CK(launch(s->pinv_group, (unsigned)std::min<int64_t>(tiles, 1 << 20), gargs, (cudaStream_t)stream, within));
  } else if (tma_ok) {
    // CLIK_TMA_TILES=T: one CTA per T tiles (hardware CTA scheduling, T tiles staged ahead) instead of the
    // balanced persistent grid
    int tiles_per_cta = 0;
    if (const char* e = getenv("CLIK_TMA_TILES")) tiles_per_cta = atoi(e);
    const int64_t ntiles = (N + s->pinv_tma.block - 1) / s->pinv_tma.block;
    const unsigned tgrid = tiles_per_cta > 0 ? (unsigned)std::max<int64_t>(1, (ntiles + tiles_per_cta - 1) / tiles_per_cta)
                                             : (unsigned)balanced_grid(s->pinv_tma, N);
    CK(launch(s->pinv_tma, tgrid, args, (cudaStream_t)stream, across));
  } else {
    CK(launch(s->pinv, grid_for(s->pinv, N), args, (cudaStream_t)stream, across));
  }
  return CLIK_OK;
}

}  // namespace

extern "C" {

clik_status clik_pinv_step_ld(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                              const double* q, const double* x, const double* y, double* qdot,
                              double* xdot, int32_t* mode, void* stream) {
  return pinv_step_impl(s, N, ld, t, t_stride, q, x, y, qdot, xdot, mode, stream, s ? s->overlap : 0);
}

clik_status clik_pinv_step(const clik_skill* s, int64_t N, const double* t, int32_t t_stride,
                           const double* q, const double* x, const double* y, double* qdot,
                           double* xdot, int32_t* mode, void* stream) {
  return pinv_step_impl(s, N, N, t, t_stride, q, x, y, qdot, xdot, mode, stream, s ? s->overlap : 0);
}

clik_status clik_pinv_rollout(const clik_skill* s, int64_t N, int32_t steps, double dt, const double* t0,
                              int32_t t_stride, double* q, double* x, const double* y,
                              double max_robot_speed, double max_virtual_speed, double* qdot_last,
                              double* xdot_last, int32_t* mode_last, int32_t* n_failed, void* stream) {
  clik_status st = check_common(s, N, t0, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!s->pinv_rollout.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the rollout kernel");
  if (steps < 0) return fail(CLIK_ERR_INVALID, "steps < 0");
  ON_DEVICE(s->desc.device);
  long long n = N, l = N;
  int ts = t_stride ? 1 : 0, k = steps;
  void* args[] = {&n, &l, &k, &dt, &t0, &ts, &q, &x, &y, &max_robot_speed, &max_virtual_speed,
                  &qdot_last, &xdot_last, &mode_last, &n_failed};
  CK(cudaLaunchKernel((const void*)s->pinv_rollout.kernel, dim3(grid_for(s->pinv_rollout, N)),
                      dim3(s->pinv_rollout.block), args, 0, (cudaStream_t)stream));
  return CLIK_OK;
}

}  // extern "C"

namespace {
clik_status qp_step_impl(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                         const double* q, const double* x, const double* y, const double* x0,
                         const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                         int32_t max_iter, void* stream, int level, bool split_ok = true) {
  clik_status st = check_common(s, N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (ld < N) return fail(CLIK_ERR_INVALID, "row stride ld (%lld) < N (%lld)", (long long)ld, (long long)N);
  if (!s->qp.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the QP kernel");
  if (!sol) return fail(CLIK_ERR_INVALID, "sol is required");
  ON_DEVICE(s->desc.device);
  long long n = N, l = ld;
  int ts = t_stride ? 1 : 0;
  int mi = max_iter > 0 ? max_iter : 10 * (s->desc.qp_n + s->desc.qp_m);
  void* args[] = {&n, &l, &t, &ts, &q, &x, &y, &x0, &active0, &sol, &status, &active, &mi};
  const bool within = level >= 1, across = level >= 2;
  if (split_ok && s->qp_fast.kernel && s->qp_tail.kernel && s->qp_split && status != nullptr) {
    // two launches: the working-set prediction for every instance (no Goldfarb-Idnani code in that
    // kernel: ~160 registers instead of 255 + spills), then the full solver for the few instances the
    // prediction could not certify; they are handed over through status[] (transient value 3).
    CK(launch(s->qp_fast, grid_for(s->qp_fast, N), args, (cudaStream_t)stream, across));
    const int64_t tiles = (N + clik::QP_TAIL_TILE - 1) / clik::QP_TAIL_TILE;
    // small batches (every tail CTA resident at once): the launch lasts as long as its slowest instance, which
    // the uncapped kernel (255 registers) runs fastest; more tiles than that: a throughput problem, the capped
    // kernel keeps twice the CTAs in flight and interleaves with other streams' fast passes (profiles/r2_ab10.txt)
    const bool capped = s->qp_tail_capped.kernel &&
                        (s->qp_tail_pick >= 0 ? s->qp_tail_pick != 0 : tiles > s->qp_tail.resident);
    CK(launch(capped ? s->qp_tail_capped : s->qp_tail, (unsigned)std::min<int64_t>(tiles, 1 << 20), args,
              (cudaStream_t)stream, within));
    return CLIK_OK;
  }
  CK(launch(s->qp, grid_for(s->qp, N), args, (cudaStream_t)stream, across));
  return CLIK_OK;
}

}  // namespace

extern "C" {

clik_status clik_qp_step_ld(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                            const double* q, const double* x, const double* y, const double* x0,
                            const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                            int32_t max_iter, void* stream) {
  return qp_step_impl(s, N, ld, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter, stream,
                      s ? s->overlap : 0);
}

clik_status clik_qp_step(const clik_skill* s, int64_t N, const double* t, int32_t t_stride,
                         const double* q, const double* x, const double* y, const double* x0,
                         const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                         int32_t max_iter, void* stream) {
  return qp_step_impl(s, N, N, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter, stream,
                      s ? s->overlap : 0);
}

clik_status clik_qp_rollout(const clik_skill* s, int64_t N, int32_t steps, double dt, const double* t0,
                            int32_t t_stride, double* q, double* x, const double* y,
                            double max_robot_speed, double max_virtual_speed, double* sol_last,
                            int32_t* n_failed, int32_t max_iter, void* stream) {
  clik_status st = check_common(s, N, t0, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!s->qp_rollout.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the QP rollout kernel");
  if (steps < 0) return fail(CLIK_ERR_INVALID, "steps < 0");
  ON_DEVICE(s->desc.device);
  long long n = N, l = N;
  int ts = t_stride ? 1 : 0, k = steps;
  int mi = max_iter > 0 ? max_iter : 10 * (s->desc.qp_n + s->desc.qp_m);
  void* args[] = {&n, &l, &k, &dt, &t0, &ts, &q, &x, &y, &max_robot_speed, &max_virtual_speed,
                  &sol_last, &n_failed, &mi};
  CK(cudaLaunchKernel((const void*)s->qp_rollout.kernel, dim3(grid_for(s->qp_rollout, N)),
                      dim3(s->qp_rollout.block), args, 0, (cudaStream_t)stream));
  return CLIK_OK;
}

clik_status clik_qp_dense(int32_t device, int64_t N, int32_t nx, int32_t m, const double* h,
                          const double* A, const double* lb, const double* ub, const double* x0,
                          double* sol, int32_t* status, uint32_t* active, int32_t max_iter,
                          void* stream) {
  if (N < 0 || nx <= 0 || m < 0) return fail(CLIK_ERR_INVALID, "bad sizes");
  if (nx > DENSE_NX2 || m > DENSE_M2)
    return fail(CLIK_ERR_INVALID, "clik_qp_dense supports nx <= %d, m <= %d (got %d x %d)", DENSE_NX2, DENSE_M2, m, nx);
  if (N == 0) return CLIK_OK;
  if (!h || (m > 0 && (!A || !lb || !ub)) || !sol) return fail(CLIK_ERR_INVALID, "NULL argument");
  ON_DEVICE(device);
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  const bool big = nx > DENSE_NX || m > DENSE_M;
  const int block = big ? 32 : 64;
  int grid = (int)std::min<int64_t>((N + block - 1) / block, (int64_t)sms * (big ? 2 : 8));
  int mi = max_iter > 0 ? max_iter : 10 * (nx + m);
  if (big)
    clik_qp_dense_kernel<DENSE_NX2, DENSE_M2><<<grid, block, 0, (cudaStream_t)stream>>>(N, nx, m, h, A, lb, ub, x0, sol,
                                                                                     status, active, mi);
  else
    clik_qp_dense_kernel<DENSE_NX, DENSE_M><<<grid, block, 0, (cudaStream_t)stream>>>(N, nx, m, h, A, lb, ub, x0, sol,
                                                                                   status, active, mi);
  CK(cudaGetLastError());
  return CLIK_OK;
}

}  // extern "C"

namespace {

// Contiguous shards of one host batch, one per skill handle (= per device), each on its own host
// thread; no exchange between devices (instances are independent), results land in the caller's arrays.
template <class Run>
clik_status run_sharded(const clik_skill* const* skills, int32_t n_skills, int64_t N, Run run) {
  if (!skills || n_skills < 1) return fail(CLIK_ERR_INVALID, "no skill handles");
  for (int k = 0; k < n_skills; ++k)
    if (!skills[k]) return fail(CLIK_ERR_INVALID, "skill handle %d is NULL", k);
  if (n_skills == 1 || N < n_skills) return run(const_cast<clik_skill*>(skills[0]), (int64_t)0, N);
  std::vector<clik_status> st(n_skills, CLIK_OK);
  std::vector<std::string> msg(n_skills);
  std::vector<std::thread> th;
  const int64_t base = N / n_skills, rem = N % n_skills;
  for (int k = 0; k < n_skills; ++k) {
    const int64_t lo = k * base + std::min<int64_t>(k, rem), cnt = base + (k < rem ? 1 : 0);
    th.emplace_back([&, k, lo, cnt] {
      st[k] = run(const_cast<clik_skill*>(skills[k]), lo, cnt);
      if (st[k] != CLIK_OK) msg[k] = g_err;      // g_err is per thread: carry the text back
    });
  }
  for (auto& t : th) t.join();
  for (int k = 0; k < n_skills; ++k)
    if (st[k] != CLIK_OK) return fail(st[k], "shard %d (device %d): %s", k, skills[k]->desc.device, msg[k].c_str());
  return CLIK_OK;
}

}  // namespace

extern "C" {

clik_status clik_pinv_step_host(const clik_skill* cs, int64_t N, const double* t, int32_t t_stride,
                                const double* q, const double* x, const double* y, double* qdot,
                                double* xdot, int32_t* mode) {
  return clik_pinv_step_host_multi(&cs, 1, N, t, t_stride, q, x, y, qdot, xdot, mode);
}

clik_status clik_pinv_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                      const double* t, int32_t t_stride, const double* q, const double* x,
                                      const double* y, double* qdot, double* xdot, int32_t* mode) {
  if (!skills || n_skills < 1 || !skills[0]) return fail(CLIK_ERR_INVALID, "no skill handles");
  clik_status st = check_common(skills[0], N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!qdot) return fail(CLIK_ERR_INVALID, "qdot is required");
  return run_sharded(skills, n_skills, N, [&](clik_skill* s, int64_t lo, int64_t cnt) {
    const clik_skill_desc& d = s->desc;
    const ReadMask& r = s->pinv_reads;
    const std::array<HostField, 7> f = {{{t, IN, 1, 8, t_stride == 0, r.t}, {q, IN, d.n_robot, 8, false, r.q},
                                         {x, IN, d.n_virtual, 8, false, r.x}, {y, IN, d.n_input, 8, false, r.y},
                                         {qdot, OUT, d.n_robot, 8}, {xdot, OUT, d.n_virtual, 8}, {mode, OUT, 1, 4}}};
    return run_host_batch(s, N, lo, cnt, f, [&](const std::array<DevPtr, 7>& p, int64_t n, int64_t ld,
                                                cudaStream_t stream, bool zero_copy) {
      auto [dt, dq, dx, dy, dqdot, dxdot, dmode] = p;
      // on mapped host memory: the staged kernel only on request (CLIK_ZC_STAGED), and no hand-over through
      // mode[] over PCIe
      return pinv_step_impl(s, n, ld, dt, t_stride, dq, dx, dy, dqdot, dxdot, dmode, stream, std::min(s->overlap, 1),
                            /*staged_ok=*/!zero_copy || zero_copy_staged(), /*split_ok=*/!zero_copy);
    });
  });
}

clik_status clik_qp_step_host(const clik_skill* cs, int64_t N, const double* t, int32_t t_stride,
                              const double* q, const double* x, const double* y, const double* x0,
                              const uint32_t* active0, double* sol, int32_t* status, uint32_t* active,
                              int32_t max_iter) {
  return clik_qp_step_host_multi(&cs, 1, N, t, t_stride, q, x, y, x0, active0, sol, status, active, max_iter);
}

clik_status clik_qp_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                    const double* t, int32_t t_stride, const double* q, const double* x,
                                    const double* y, const double* x0, const uint32_t* active0, double* sol,
                                    int32_t* status, uint32_t* active, int32_t max_iter) {
  if (!skills || n_skills < 1 || !skills[0]) return fail(CLIK_ERR_INVALID, "no skill handles");
  clik_status st = check_common(skills[0], N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!sol) return fail(CLIK_ERR_INVALID, "sol is required");
  return run_sharded(skills, n_skills, N, [&](clik_skill* s, int64_t lo, int64_t cnt) {
    const clik_skill_desc& d = s->desc;
    const ReadMask& r = s->qp_reads;
    const std::array<HostField, 9> f = {{{t, IN, 1, 8, t_stride == 0, r.t}, {q, IN, d.n_robot, 8, false, r.q},
                                         {x, IN, d.n_virtual, 8, false, r.x}, {y, IN, d.n_input, 8, false, r.y},
                                         {x0, IN, d.qp_n, 8}, {active0, IN, 2, 4}, {sol, OUT, d.qp_n, 8},
                                         {status, OUT, 1, 4}, {active, OUT, 2, 4}}};
    return run_host_batch(s, N, lo, cnt, f, [&](const std::array<DevPtr, 9>& p, int64_t n, int64_t ld,
                                                cudaStream_t stream, bool zero_copy) {
      auto [dt, dq, dx, dy, dx0, dactive0, dsol, dstatus, dactive] = p;
      // on mapped host memory one kernel: a tail pass would scan status[] and re-read the inputs of the pending
      // instances over PCIe (1.7e8 vs 4.4-4.8e8 steps/s for the UR5 problem, profiles/r2_ab19.txt)
      return qp_step_impl(s, n, ld, dt, t_stride, dq, dx, dy, dx0, dactive0, dsol, dstatus, dactive, max_iter, stream,
                          std::min(s->overlap, 1), /*split_ok=*/!zero_copy);
    });
  });
}

// ---- single instance (PseudoInverseController.solve / ReactiveQPController.solve as the reference calls
// them, one robot state at a time): HOST pointers to the vectors of ONE instance.  The instance goes
// through a page-locked slot mapped into the device address space: no allocation, no staging copies, no
// pointer queries per call — fill, launch on the skill's own stream, wait, read.
static clik_status one_slot(clik_skill* s, size_t doubles) {
  if (!s->one_stream) CK(cudaStreamCreateWithFlags(&s->one_stream, cudaStreamNonBlocking));
  if (s->one_doubles < doubles) {
    if (s->one_host) CK(cudaFreeHost(s->one_host));
    s->one_host = nullptr;
    s->one_doubles = 0;
    CK(cudaHostAlloc((void**)&s->one_host, doubles * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
    CK(cudaHostGetDevicePointer((void**)&s->one_dev, s->one_host, 0));
    s->one_doubles = doubles;
  }
  return CLIK_OK;
}

// The single-instance slot of `s`, locked (until the OneSlot goes out of scope) and sized for t | q | x | y followed
// by `own_cells` doubles of the caller's own cells, with the four inputs written.
struct OneSlot {
  std::unique_lock<std::mutex> lock;
  double* host = nullptr;   // the slot: host view ...
  double* dev = nullptr;    // ... and device view
  const double *t = nullptr, *q = nullptr, *x = nullptr, *y = nullptr;   // device pointers of the inputs
  size_t own = 0;           // first cell after the inputs: the caller's own cells start here
};

static clik_status fill_one_slot(clik_skill* s, size_t own_cells, double t, const double* q, const double* x,
                                 const double* y, OneSlot* o) {
  const int nq = s->desc.n_robot, nx = s->desc.n_virtual, ny = s->desc.n_input;
  o->lock = std::unique_lock<std::mutex>(s->mu);
  o->own = 1 + nq + nx + ny;
  clik_status st = one_slot(s, o->own + own_cells);
  if (st != CLIK_OK) return st;
  double *h = s->one_host, *dv = s->one_dev;
  h[0] = t;
  std::memcpy(h + 1, q, sizeof(double) * nq);
  if (nx) std::memcpy(h + 1 + nq, x, sizeof(double) * nx);
  if (ny) std::memcpy(h + 1 + nq + nx, y, sizeof(double) * ny);
  o->host = h;
  o->dev = dv;
  o->t = dv;
  o->q = dv + 1;
  o->x = nx ? dv + 1 + nq : nullptr;
  o->y = ny ? dv + 1 + nq + nx : nullptr;
  return CLIK_OK;
}

clik_status clik_pinv_solve_one(const clik_skill* cs, double t, const double* q, const double* x, const double* y,
                                double* qdot, double* xdot, int32_t* mode) {
  clik_skill* s = const_cast<clik_skill*>(cs);
  if (!s || !q || !qdot) return fail(CLIK_ERR_INVALID, "NULL argument");
  if (!s->pinv.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the pinv kernel");
  const clik_skill_desc& d = s->desc;
  if (d.n_virtual > 0 && (!x || !xdot)) return fail(CLIK_ERR_INVALID, "skill has virtual_var: x and xdot are required");
  if (d.n_input > 0 && !y) return fail(CLIK_ERR_INVALID, "skill reads input_var: y is required");
  ON_DEVICE(d.device);
  const int nq = d.n_robot, nx = d.n_virtual;
  OneSlot o;
  // slot: t | q | x | y | qdot | xdot | mode (as one double-sized cell)
  clik_status st = fill_one_slot(s, nq + nx + 1, t, q, x, y, &o);
  if (st != CLIK_OK) return st;
  long long n = 1, l = 1;
  int ts = 0;
  double *dqd = o.dev + o.own, *dxd = nx ? o.dev + o.own + nq : nullptr;
  int* dm = (int*)(o.dev + o.own + nq + nx);
  void* args[] = {&n, &l, &o.t, &ts, &o.q, &o.x, &o.y, &dqd, &dxd, &dm};
  CK(cudaLaunchKernel((const void*)s->pinv.kernel, dim3(1), dim3(32), args, 0, s->one_stream));
  CK(cudaStreamSynchronize(s->one_stream));
  const double* h = o.host + o.own;
  std::memcpy(qdot, h, sizeof(double) * nq);
  if (nx) std::memcpy(xdot, h + nq, sizeof(double) * nx);
  if (mode) *mode = *(const int*)(h + nq + nx);
  return CLIK_OK;
}

clik_status clik_qp_solve_one(const clik_skill* cs, double t, const double* q, const double* x, const double* y,
                              const double* x0, double* sol, int32_t* status, uint32_t* active, int32_t max_iter) {
  return clik_qp_solve_one_lam(cs, t, q, x, y, x0, sol, status, active, max_iter, nullptr);
}

clik_status clik_qp_solve_one_lam(const clik_skill* cs, double t, const double* q, const double* x, const double* y,
                                  const double* x0, double* sol, int32_t* status, uint32_t* active, int32_t max_iter,
                                  double* lam) {
  clik_skill* s = const_cast<clik_skill*>(cs);
  if (!s || !q || !sol) return fail(CLIK_ERR_INVALID, "NULL argument");
  if (!s->qp.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the QP kernel");
  if (lam && !s->qp_duals.kernel)
    return fail(CLIK_ERR_INVALID, "multipliers need at most 32 constraint rows (the skill has %d)", s->desc.qp_m);
  const clik_skill_desc& d = s->desc;
  if (d.n_virtual > 0 && !x) return fail(CLIK_ERR_INVALID, "skill has virtual_var: x is required");
  if (d.n_input > 0 && !y) return fail(CLIK_ERR_INVALID, "skill reads input_var: y is required");
  ON_DEVICE(d.device);
  const int qn = d.qp_n, qm = lam ? d.qp_m : 0;
  OneSlot o;
  // slot: t | q | x | y | x0 | sol | status, active_up, active_lo (three int cells in two doubles) | lam
  clik_status st = fill_one_slot(s, 2 * qn + 2 + qm, t, q, x, y, &o);
  if (st != CLIK_OK) return st;
  const size_t o_x0 = o.own, o_sol = o_x0 + qn, o_int = o_sol + qn, o_lam = o_int + 2;
  double *h = o.host, *dv = o.dev;
  if (x0) std::memcpy(h + o_x0, x0, sizeof(double) * qn);
  long long n = 1, l = 1;
  int ts = 0;
  int mi = max_iter > 0 ? max_iter : 10 * (d.qp_n + d.qp_m);
  const double* dx0 = x0 ? dv + o_x0 : nullptr;
  const unsigned* da0 = nullptr;
  double* dsol = dv + o_sol;
  int* dst = (int*)(dv + o_int);
  unsigned* dact = (unsigned*)(dv + o_int) + 1;      // active[0], active[ld = 1]
  void* args[] = {&n, &l, &o.t, &ts, &o.q, &o.x, &o.y, &dx0, &da0, &dsol, &dst, &dact, &mi};
  // one instance: the single full kernel (prediction + iteration in one launch)
  CK(cudaLaunchKernel((const void*)s->qp.kernel, dim3(1), dim3(32), args, 0, s->one_stream));
  if (lam) {
    // the multipliers at the step's output, same stream: one wait for both launches
    double* dlam = dv + o_lam;
    void* largs[] = {&n, &l, &o.t, &ts, &o.q, &o.x, &o.y, &dsol, &dst, &dact, &dlam};
    CK(cudaLaunchKernel((const void*)s->qp_duals.kernel, dim3(1), dim3(32), largs, 0, s->one_stream));
  }
  CK(cudaStreamSynchronize(s->one_stream));
  std::memcpy(sol, h + o_sol, sizeof(double) * qn);
  const int* hi = (const int*)(h + o_int);
  if (status) *status = hi[0];
  if (active) { active[0] = (uint32_t)hi[1]; active[1] = (uint32_t)hi[2]; }
  if (lam) std::memcpy(lam, h + o_lam, sizeof(double) * qm);
  return CLIK_OK;
}

}  // extern "C"

// ---- reactive NLP controller ------------------------------------------------------------------------------
namespace {

constexpr int NLP_DEFAULT_MAX_ITER = 50;

clik_status nlp_step_impl(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                          const double* q, const double* x, const double* y, const double* x0, double* sol,
                          int32_t* status, int32_t* iters, uint32_t* active, int32_t max_iter, void* stream) {
  clik_status st = check_common(s, N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (ld < N) return fail(CLIK_ERR_INVALID, "row stride ld (%lld) < N (%lld)", (long long)ld, (long long)N);
  if (!s->nlp.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the NLP kernel");
  if (!sol) return fail(CLIK_ERR_INVALID, "sol is required");
  ON_DEVICE(s->desc.device);
  long long n = N, l = ld;
  int ts = t_stride ? 1 : 0;
  int mi = max_iter > 0 ? max_iter : NLP_DEFAULT_MAX_ITER;
  void* args[] = {&n, &l, &t, &ts, &q, &x, &y, &x0, &sol, &status, &iters, &active, &mi};
  CK(launch(s->nlp, grid_for(s->nlp, N), args, (cudaStream_t)stream, false));
  return CLIK_OK;
}

}  // namespace

extern "C" {

clik_status clik_nlp_step(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                          const double* x, const double* y, const double* x0, double* sol, int32_t* status,
                          int32_t* iters, uint32_t* active, int32_t max_iter, void* stream) {
  return nlp_step_impl(s, N, N, t, t_stride, q, x, y, x0, sol, status, iters, active, max_iter, stream);
}

clik_status clik_nlp_step_ld(const clik_skill* s, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                             const double* q, const double* x, const double* y, const double* x0, double* sol,
                             int32_t* status, int32_t* iters, uint32_t* active, int32_t max_iter, void* stream) {
  return nlp_step_impl(s, N, ld, t, t_stride, q, x, y, x0, sol, status, iters, active, max_iter, stream);
}

clik_status clik_nlp_step_host(const clik_skill* cs, int64_t N, const double* t, int32_t t_stride,
                               const double* q, const double* x, const double* y, const double* x0,
                               double* sol, int32_t* status, int32_t* iters, uint32_t* active, int32_t max_iter) {
  return clik_nlp_step_host_multi(&cs, 1, N, t, t_stride, q, x, y, x0, sol, status, iters, active, max_iter);
}

clik_status clik_nlp_step_host_multi(const clik_skill* const* skills, int32_t n_skills, int64_t N,
                                     const double* t, int32_t t_stride, const double* q, const double* x,
                                     const double* y, const double* x0, double* sol, int32_t* status,
                                     int32_t* iters, uint32_t* active, int32_t max_iter) {
  if (!skills || n_skills < 1 || !skills[0]) return fail(CLIK_ERR_INVALID, "no skill handles");
  clik_status st = check_common(skills[0], N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!skills[0]->nlp.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the NLP kernel");
  if (!sol) return fail(CLIK_ERR_INVALID, "sol is required");
  return run_sharded(skills, n_skills, N, [&](clik_skill* s, int64_t lo, int64_t cnt) {
    const clik_skill_desc& d = s->desc;
    const ReadMask& r = s->qp_reads;
    const std::array<HostField, 9> f = {{{t, IN, 1, 8, t_stride == 0, r.t}, {q, IN, d.n_robot, 8, false, r.q},
                                         {x, IN, d.n_virtual, 8, false, r.x}, {y, IN, d.n_input, 8, false, r.y},
                                         {x0, IN, d.qp_n, 8}, {sol, OUT, d.qp_n, 8}, {status, OUT, 1, 4},
                                         {iters, OUT, 1, 4}, {active, OUT, 2, 4}}};
    return run_host_batch(s, N, lo, cnt, f, [&](const std::array<DevPtr, 9>& p, int64_t n, int64_t ld,
                                                cudaStream_t stream, bool) {
      auto [dt, dq, dx, dy, dx0, dsol, dstatus, diters, dactive] = p;
      return nlp_step_impl(s, n, ld, dt, t_stride, dq, dx, dy, dx0, dsol, dstatus, diters, dactive, max_iter, stream);
    });
  });
}

clik_status clik_nlp_solve_one(const clik_skill* cs, double t, const double* q, const double* x, const double* y,
                               const double* x0, double* sol, int32_t* status, int32_t* iters, uint32_t* active,
                               int32_t max_iter) {
  return clik_nlp_solve_one_lam(cs, t, q, x, y, x0, sol, status, iters, active, max_iter, nullptr);
}

clik_status clik_nlp_solve_one_lam(const clik_skill* cs, double t, const double* q, const double* x, const double* y,
                                   const double* x0, double* sol, int32_t* status, int32_t* iters, uint32_t* active,
                                   int32_t max_iter, double* lam) {
  clik_skill* s = const_cast<clik_skill*>(cs);
  if (!s || !q || !sol) return fail(CLIK_ERR_INVALID, "NULL argument");
  if (!s->nlp.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the NLP kernel");
  if (lam && !s->nlp_duals.kernel)
    return fail(CLIK_ERR_INVALID, "multipliers need at most 32 constraint rows (the skill has %d)", s->desc.qp_m);
  const clik_skill_desc& d = s->desc;
  if (d.n_virtual > 0 && !x) return fail(CLIK_ERR_INVALID, "skill has virtual_var: x is required");
  if (d.n_input > 0 && !y) return fail(CLIK_ERR_INVALID, "skill reads input_var: y is required");
  ON_DEVICE(d.device);
  const int qn = d.qp_n, qm = lam ? d.qp_m : 0;
  OneSlot o;
  // slot: t | q | x | y | x0 | sol | status, iters, active_up, active_lo (four int cells in two doubles) | lam
  clik_status st = fill_one_slot(s, 2 * qn + 2 + qm, t, q, x, y, &o);
  if (st != CLIK_OK) return st;
  const size_t o_x0 = o.own, o_sol = o_x0 + qn, o_int = o_sol + qn, o_lam = o_int + 2;
  double *h = o.host, *dv = o.dev;
  if (x0) std::memcpy(h + o_x0, x0, sizeof(double) * qn);
  long long n = 1, l = 1;
  int ts = 0;
  int mi = max_iter > 0 ? max_iter : NLP_DEFAULT_MAX_ITER;
  const double* dx0 = x0 ? dv + o_x0 : nullptr;
  double* dsol = dv + o_sol;
  int* dst = (int*)(dv + o_int);
  int* dit = dst + 1;
  unsigned* dact = (unsigned*)(dst + 2);      // active[0], active[ld = 1]
  void* args[] = {&n, &l, &o.t, &ts, &o.q, &o.x, &o.y, &dx0, &dsol, &dst, &dit, &dact, &mi};
  CK(cudaLaunchKernel((const void*)s->nlp.kernel, dim3(1), dim3(32), args, 0, s->one_stream));
  if (lam) {
    double* dlam = dv + o_lam;
    void* largs[] = {&n, &l, &o.t, &ts, &o.q, &o.x, &o.y, &dsol, &dst, &dact, &dlam};
    CK(cudaLaunchKernel((const void*)s->nlp_duals.kernel, dim3(1), dim3(32), largs, 0, s->one_stream));
  }
  CK(cudaStreamSynchronize(s->one_stream));
  std::memcpy(sol, h + o_sol, sizeof(double) * qn);
  const int* hi = (const int*)(h + o_int);
  if (status) *status = hi[0];
  if (iters) *iters = hi[1];
  if (active) { active[0] = (uint32_t)hi[2]; active[1] = (uint32_t)hi[3]; }
  if (lam) std::memcpy(lam, h + o_lam, sizeof(double) * qm);
  return CLIK_OK;
}

clik_status clik_nlp_rollout(const clik_skill* s, int64_t N, int32_t steps, double dt, const double* t0,
                             int32_t t_stride, double* q, double* x, const double* y, double max_robot_speed,
                             double max_virtual_speed, double* sol_last, int32_t* n_failed, int32_t max_iter,
                             void* stream) {
  clik_status st = check_common(s, N, t0, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!s->nlp_rollout.kernel) return fail(CLIK_ERR_INVALID, "skill was built without the NLP rollout kernel");
  if (steps < 0) return fail(CLIK_ERR_INVALID, "steps < 0");
  ON_DEVICE(s->desc.device);
  long long n = N, l = N;
  int ts = t_stride ? 1 : 0, k = steps;
  int mi = max_iter > 0 ? max_iter : NLP_DEFAULT_MAX_ITER;
  void* args[] = {&n, &l, &k, &dt, &t0, &ts, &q, &x, &y, &max_robot_speed, &max_virtual_speed,
                  &sol_last, &n_failed, &mi};
  CK(cudaLaunchKernel((const void*)s->nlp_rollout.kernel, dim3(grid_for(s->nlp_rollout, N)),
                      dim3(s->nlp_rollout.block), args, 0, (cudaStream_t)stream));
  return CLIK_OK;
}

}  // extern "C"

// ---- constraint multipliers of a step's output (clik_duals.cuh) -------------------------------------------
namespace {

// Arguments of a multiplier call; CLIK_OK with nothing to do when N == 0.
clik_status duals_check(const clik_skill* s, bool nlp, int64_t N, const double* t, const double* q, const double* x,
                        const double* y, const double* sol, const int32_t* status, const uint32_t* active,
                        const double* lam) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  if (!(nlp ? s->nlp.kernel : s->qp.kernel))
    return fail(CLIK_ERR_INVALID, "skill was built without the %s kernel", nlp ? "NLP" : "QP");
  if (!(nlp ? s->nlp_duals.kernel : s->qp_duals.kernel))
    return fail(CLIK_ERR_INVALID, "multipliers need at most 32 constraint rows (the skill has %d)", s->desc.qp_m);
  clik_status st = check_common(s, N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!sol || !status || !active || !lam) return fail(CLIK_ERR_INVALID, "sol, status, active and lam are required");
  return CLIK_OK;
}

clik_status duals_impl(const clik_skill* s, bool nlp, int64_t N, int64_t ld, const double* t, int32_t t_stride,
                       const double* q, const double* x, const double* y, const double* sol, const int32_t* status,
                       const uint32_t* active, double* lam, void* stream) {
  clik_status st = duals_check(s, nlp, N, t, q, x, y, sol, status, active, lam);
  if (st != CLIK_OK || N == 0) return st;
  if (ld < N) return fail(CLIK_ERR_INVALID, "row stride ld (%lld) < N (%lld)", (long long)ld, (long long)N);
  const KernelInfo& k = nlp ? s->nlp_duals : s->qp_duals;
  ON_DEVICE(s->desc.device);
  long long n = N, l = ld;
  int ts = t_stride ? 1 : 0;
  void* args[] = {&n, &l, &t, &ts, &q, &x, &y, &sol, &status, &active, &lam};
  CK(launch(k, grid_for(k, N), args, (cudaStream_t)stream, false));
  return CLIK_OK;
}

// Host arrays: the kernel on mapped memory when every buffer is page-locked, else the chunked copy pipeline.
clik_status duals_host(clik_skill* s, bool nlp, int64_t N, const double* t, int32_t t_stride, const double* q,
                       const double* x, const double* y, const double* sol, const int32_t* status,
                       const uint32_t* active, double* lam) {
  clik_status st = duals_check(s, nlp, N, t, q, x, y, sol, status, active, lam);
  if (st != CLIK_OK || N == 0) return st;
  const clik_skill_desc& d = s->desc;
  const ReadMask& r = s->qp_reads;
  const std::array<HostField, 8> f = {{{t, IN, 1, 8, t_stride == 0, r.t}, {q, IN, d.n_robot, 8, false, r.q},
                                       {x, IN, d.n_virtual, 8, false, r.x}, {y, IN, d.n_input, 8, false, r.y},
                                       {sol, IN, d.qp_n, 8}, {status, IN, 1, 4}, {active, IN, 2, 4},
                                       {lam, OUT, d.qp_m, 8}}};
  return run_host_batch(s, N, 0, N, f, [&](const std::array<DevPtr, 8>& p, int64_t n, int64_t ld,
                                           cudaStream_t stream, bool) {
    auto [dt, dq, dx, dy, dsol, dstatus, dactive, dlam] = p;
    return duals_impl(s, nlp, n, ld, dt, t_stride, dq, dx, dy, dsol, dstatus, dactive, dlam, stream);
  });
}

}  // namespace

extern "C" {

clik_status clik_qp_duals(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                          const double* x, const double* y, const double* sol, const int32_t* status,
                          const uint32_t* active, double* lam, void* stream) {
  return duals_impl(s, false, N, N, t, t_stride, q, x, y, sol, status, active, lam, stream);
}

clik_status clik_nlp_duals(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                           const double* x, const double* y, const double* sol, const int32_t* status,
                           const uint32_t* active, double* lam, void* stream) {
  return duals_impl(s, true, N, N, t, t_stride, q, x, y, sol, status, active, lam, stream);
}

clik_status clik_qp_duals_host(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                               const double* x, const double* y, const double* sol, const int32_t* status,
                               const uint32_t* active, double* lam) {
  return duals_host(const_cast<clik_skill*>(s), false, N, t, t_stride, q, x, y, sol, status, active, lam);
}

clik_status clik_nlp_duals_host(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                                const double* x, const double* y, const double* sol, const int32_t* status,
                                const uint32_t* active, double* lam) {
  return duals_host(const_cast<clik_skill*>(s), true, N, t, t_stride, q, x, y, sol, status, active, lam);
}

}  // extern "C"

// ---- reverse-mode derivative of a step's output (clik_vjp.cuh) -------------------------------------------
namespace {

clik_status vjp_impl(const clik_skill* s, bool nlp, int64_t N, const double* t, int32_t t_stride, const double* q,
                     const double* x, const double* y, const double* sol, const int32_t* status,
                     const uint32_t* active, const double* sol_bar, double* t_bar, double* q_bar, double* x_bar,
                     double* y_bar, void* stream) {
  if (!s) return fail(CLIK_ERR_INVALID, "skill is NULL");
  const KernelInfo& k = nlp ? s->nlp_vjp : s->qp_vjp;
  if (!k.kernel)
    return fail(CLIK_ERR_INVALID, "skill image has no %s VJP kernel (build it with emit_skill(..., vjp=True); at most "
                "32 constraint rows)", nlp ? "NLP" : "QP");
  clik_status st = check_common(s, N, t, q, x, y);
  if (st != CLIK_OK || N == 0) return st;
  if (!sol || !status || !active || !sol_bar || !t_bar || !q_bar)
    return fail(CLIK_ERR_INVALID, "sol, status, active, sol_bar, t_bar and q_bar are required");
  if (s->desc.n_virtual > 0 && !x_bar) return fail(CLIK_ERR_INVALID, "skill has virtual_var: x_bar is required");
  if (s->desc.n_input > 0 && !y_bar) return fail(CLIK_ERR_INVALID, "skill reads input_var: y_bar is required");
  ON_DEVICE(s->desc.device);
  long long n = N, l = N;
  int ts = t_stride ? 1 : 0;
  void* args[] = {&n, &l, &t, &ts, &q, &x, &y, &sol, &status, &active, &sol_bar, &t_bar, &q_bar, &x_bar, &y_bar};
  CK(launch(k, grid_for(k, N), args, (cudaStream_t)stream, false));
  return CLIK_OK;
}

}  // namespace

extern "C" {

clik_status clik_qp_vjp(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                        const double* x, const double* y, const double* sol, const int32_t* status,
                        const uint32_t* active, const double* sol_bar, double* t_bar, double* q_bar, double* x_bar,
                        double* y_bar, void* stream) {
  return vjp_impl(s, false, N, t, t_stride, q, x, y, sol, status, active, sol_bar, t_bar, q_bar, x_bar, y_bar, stream);
}

clik_status clik_nlp_vjp(const clik_skill* s, int64_t N, const double* t, int32_t t_stride, const double* q,
                         const double* x, const double* y, const double* sol, const int32_t* status,
                         const uint32_t* active, const double* sol_bar, double* t_bar, double* q_bar, double* x_bar,
                         double* y_bar, void* stream) {
  return vjp_impl(s, true, N, t, t_stride, q, x, y, sol, status, active, sol_bar, t_bar, q_bar, x_bar, y_bar, stream);
}

clik_status clik_measure_fp64_peak(int32_t device, int32_t iters, double* tflops) {
  if (!tflops || iters <= 0) return fail(CLIK_ERR_INVALID, "bad argument");
  ON_DEVICE(device);
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  const int block = 256, grid = sms * 8;
  double* out = nullptr;
  CK(cudaMalloc(&out, (size_t)grid * block * sizeof(double)));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CK(cudaEventRecord(e0));
    dfma_peak_kernel<<<grid, block>>>(out, iters, 0.999999, 1e-7);
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8.0 * (double)iters * grid * block;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  *tflops = best;
  return CLIK_OK;
}

clik_status clik_flush_l2(int32_t device, void* stream) {
  if (device < 0 || device >= 64) return fail(CLIK_ERR_INVALID, "bad device");
  ON_DEVICE(device);
  {
    std::lock_guard<std::mutex> lock(g_flush_mu);
    if (!g_flush_buf[device]) CK(cudaMalloc(&g_flush_buf[device], FLUSH_BYTES));
  }
  fill_kernel<<<1184, 256, 0, (cudaStream_t)stream>>>(g_flush_buf[device], FLUSH_BYTES / 8, 0.0);
  CK(cudaGetLastError());
  return CLIK_OK;
}

}  // extern "C"
