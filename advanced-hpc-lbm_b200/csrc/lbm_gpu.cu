// lbm_gpu.cu -- host side of liblbm_b200.so: the C-ABI declared in include/lbm_gpu.h.
//
// Replaces the step loop of the reference's main() (d2q9-bgk.c:180-201) and the device
// side of initialise()/finalise() (d2q9-bgk.c:2787-2857, :2871-2890).  No PyTorch, no
// CPU fallback: every entry point either runs the CUDA path or returns an error.
#include "lbm_gpu.h"
#include "lbm_kernels.cuh"
#include "lbm_cluster.cuh"
#include "lbm_tb2.cuh"
#include "lbm_tb3.cuh"
#include "lbm_pairs.cuh"
#include "lbm_f16.cuh"

#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

namespace {

thread_local std::string g_error;

struct CachedWindow { int device; size_t bytes; char* ptr; };
std::mutex g_window_mutex;
std::vector<CachedWindow> g_window_cache;     // windows of destroyed LBM_GPU_POOL lattices
struct CachedIpcMapping { cudaIpcMemHandle_t handle; int device; void* ptr; };
std::vector<CachedIpcMapping> g_ipc_cache;    // neighbours' windows opened by LBM_GPU_POOL lattices (kept mapped)

int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_error = buf;
  return 1;
}

struct CudaError {
  std::string what;
};

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      char b_[512];                                                                           \
      snprintf(b_, sizeof b_, "CUDA error %s (%s) at %s:%d: %s", cudaGetErrorName(e_),        \
               cudaGetErrorString(e_), __FILE__, __LINE__, #call);                            \
      throw CudaError{b_};                                                                    \
    }                                                                                         \
  } while (0)

inline long long round_up(long long v, long long m) { return (v + m - 1) / m * m; }

inline bool env_on(const char* name) { const char* e = getenv(name); return e && e[0] == '1'; }   // kill switches

// The one LBM_GPU_KERNEL_* flag the caller forced, or 0; two or more are refused, by name.
unsigned forced_kernel(unsigned flags) {
  // LBM_GPU_KERNEL_<name> == 1 << index
  static const char* const names[] = {nullptr, nullptr, "SCALAR", "TMA", "VEC4", nullptr, "PERSISTENT", nullptr, "CLUSTER", "TB2", nullptr, "PAIRS", "TB3"};
  unsigned k = 0;
  std::string msg = "more than one kernel forced, pass at most one of:";
  for (int b = 0; b < 13; b++)
    if (names[b] && (flags >> b & 1)) { k |= 1u << b; msg += std::string(" LBM_GPU_KERNEL_") + names[b]; }
  if (k & (k - 1)) throw CudaError{msg};
  return k;
}

constexpr int kPersistScalarBlocks = 296;      // measured, profiles/r01_small_grids.md
constexpr long long kPersistMaxCells = 1280 * 1024;   // K5 up to here (1024^2: 109 GLUPS against 63 for K7); from 1280^2 on K7 wins (profiles/r02_kernel_variants.md)
constexpr size_t kStagingBytes = 64u << 20;   // device staging for AoS<->SoA / mask / fields

// descriptor exchanged between processes (lbm_gpu_ipc_export / _connect)
struct IpcDesc {
  uint32_t magic;
  int32_t elem_size;
  int32_t device;
  int32_t pid;
  int32_t nx, pitch, rows;
  int32_t pad_;
  long long row0;
  unsigned long long win_addr;        // only meaningful inside the exporting process
  unsigned long long win_bytes;
  unsigned long long off_sync;        // byte offset of the sync words inside the window
  unsigned long long off_gmask;       // byte offset of the ghost mask rows inside the window
  unsigned long long steps_done;
  unsigned long long passes_done;     // kernel passes so far: the unit of the flag protocol
  long long local_free_cells;
  int32_t cur;                        // lattice buffer holding the current state
  int32_t tb2_ok;                     // this slab could run the two-step kernel
  cudaIpcMemHandle_t handle;          // of the window (the lattice itself is never shared)
  char gpu_uuid[16];                  // physical GPU: two flag-ordered slabs must not share one
};
static_assert(sizeof(IpcDesc) <= LBM_GPU_IPC_DESC_BYTES, "descriptor too large");
constexpr uint32_t kIpcMagic = 0x4c424d31u;   // "LBM1"

enum SyncWord { kFlagFromBelow = 0, kFlagFromAbove = 1, kBoundaryDone = 2, kScratch0 = 3, kScratch1 = 4,
                kScratch2 = 5, kGridBarrier = 6, kAbort = 7, kSyncError = 8 /* must follow kAbort */,
                kAvScratch = 16 /* kAvWords words */, kSyncWords = 16 + 128 };
constexpr int kTb2MinRows = 8;                             // per slab, for the two-step kernel
constexpr int kTb3MinRows = 12;                            // for the three-step kernel (one slab)
constexpr double kTb3MinWaves = 2.0;                       // K10 by default from this many waves of its blocks on
constexpr int kTb3OverlapSegRows = 192;                    // K10 segment height when passes overlap
constexpr int kAvWords = LBM_AV_STRIDE * LBM_AV_SLOTS;     // words of one step's |u| sums (1 KiB)
constexpr int kMaxSegmentSteps = 1 << 16;                  // 64 MiB of sums per run segment

struct GridBase {
  virtual ~GridBase() {}
  virtual bool is_f64() const = 0;
};

template <typename real>
struct Slab {
  int device = 0;
  long long row0 = 0;   // first global row
  int rows = 0;         // local rows
  int accel_row = LBM_NO_ROW;   // local row of global row ny-2, or LBM_NO_ROW
  char* base = nullptr; // lattice[2] | side[2] | mask (private to this GPU)
  size_t bytes = 0;
  size_t off_lattice[2] = {0, 0}, off_side[2] = {0, 0}, off_mask = 0;
  real* lattice[2] = {nullptr, nullptr};
  real* side[2] = {nullptr, nullptr};
  uint32_t* mask = nullptr;
  // window: ghost rows [parity 2][direction 2][depth 2][9 planes][pitch], ghost mask rows, sync words.
  // The only memory neighbours (other GPUs / processes) read or write.
  char* win = nullptr;
  size_t win_bytes = 0, off_sync = 0, off_gmask = 0;
  unsigned long long* sync = nullptr;
  uint32_t* ghost_mask = nullptr;     // inside the window: mask words of row -1, then of row `rows`
  unsigned long long* av = nullptr;   // per step LBM_AV_SLOTS x {sum of low halves, sum of high halves}
  unsigned long long* av_compact = nullptr;
  size_t av_cap = 0;                  // steps
  void* staging = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;            // host <-> staging copies, overlapped with the kernels on `stream`
  cudaEvent_t stage_filled[2] = {nullptr, nullptr};   // a staging half is ready for its consumer
  cudaEvent_t stage_drained[2] = {nullptr, nullptr};  // ... and has been consumed
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t step_ev[2] = {nullptr, nullptr};   // "step t finished", alternating by parity
  long long free_cells = 0;
  // neighbour views: the windows of the slab above (holds global row row0+rows) and below
  char* up_win = nullptr;
  char* dn_win = nullptr;
  unsigned long long* up_flag = nullptr;      // neighbour above's kFlagFromBelow
  unsigned long long* dn_flag = nullptr;      // neighbour below's kFlagFromAbove
  unsigned long long* up_abort = nullptr;     // the neighbours' kAbort words
  unsigned long long* dn_abort = nullptr;
  uint32_t* up_gmask = nullptr;               // neighbour above's copy of the mask of its row -1
  uint32_t* dn_gmask = nullptr;               // neighbour below's copy of the mask of its row `rows`
  void* ipc_mapped[2] = {nullptr, nullptr};   // pointers to close on destroy
  bool pooled = false;                        // base/staging came from the stream-ordered pool
  alignas(64) CUtensorMap tmap[2];            // K1c: (x, row, plane) view of lattice[0], lattice[1], row boxes
  alignas(64) CUtensorMap tmap_halo[2];       // same view, 4-element boxes (the x halo of a tile)
};

template <typename real> struct ParamT;
template <> struct ParamT<float> { typedef lbm_param type; };
template <> struct ParamT<double> { typedef lbm_param_f64 type; };

template <typename real>
class Grid : public GridBase {
 public:
  typedef typename ParamT<real>::type Param;
  Param prm;
  unsigned flags = 0;
  int kernel = 0;              // LBM_GPU_KERNEL_* that runs: set by select_kernel() only
  int persistent_vec = 4;      // cells per thread of the persistent kernel (4, or 1 for tiny grids)
  int cluster_ctas = 0;        // K6: CTAs of the cluster (16 or 8), 0 = not applicable
  int cluster_rows = 0;        // K6: rows per CTA
  size_t cluster_smem = 0;     // K6: dynamic shared memory per CTA
  int pitch = 0, mask_pitch = 0;
  bool slab_mode = false;      // one process per GPU: neighbours are other processes
  bool connected = false;      // neighbour views are set
  bool multi = false;          // more than one slab in the whole grid
  bool use_flags = false;      // cross-slab ordering by device-side flags (else: CUDA events)
  long long global_free_cells = -1;
  long long steps_done = 0;
  long long passes_done = 0;   // kernel passes (one or two timesteps each): the unit of the flag protocol
  int cur = 0;                 // lattice buffer / window parity holding the current state (flips per pass)
  int tb2_strips = 0, tb2_wout = 0, tb2_seg_rows = 0, tb2_span = 0, tb2_threads = 0;
  int tb2_tail_rows = 16, tb2_tail_segs = 0;   // K7: height and number of the short segments that end a launch
  int tb3_seg_rows = 0;        // K10: rows per segment
  bool tb3_overlap = false;    // K10: consecutive passes overlap, ordered per tile (lbm_tb3.cuh)
  uint32_t* tb3_done = nullptr;   // K10: per tile, the passes it has completed (tb3_overlap only)
  int pairs_tile_rows = 0;     // K9: rows per block
  bool f16 = false;            // LBM_GPU_STORE_F16: the lattice buffers hold shifted binary16 (lbm_f16.cuh)
  bool failed = false;         // a neighbour never arrived: the lattice contents are void
  bool loaded_unprepared = false;   // a slab handle took rows from lbm_gpu_load_rows: lbm_gpu_ipc_prepare must come first
  unsigned long long timeout_ns = 10000000000ULL;
  long long launches = 0;
  double last_run_ms = 0.0, last_step_ms = 0.0;
  std::vector<Slab<real>> slabs;

  bool is_f64() const override { return sizeof(real) == 8; }

  ~Grid() override {
    for (auto& s : slabs) {
      cudaSetDevice(s.device);
      if (s.stream) cudaStreamSynchronize(s.stream);
      for (int i = 0; i < 2; i++)
        if (s.ipc_mapped[i]) cudaIpcCloseMemHandle(s.ipc_mapped[i]);
      pool_free(s.av, s);
      pool_free(s.staging, s);
      pool_free(s.base, s);
      if (s.stream) cudaStreamSynchronize(s.stream);
      window_free(s);
      if (s.ev0) cudaEventDestroy(s.ev0);
      if (s.ev1) cudaEventDestroy(s.ev1);
      for (int i = 0; i < 2; i++) {
        if (s.stage_filled[i]) cudaEventDestroy(s.stage_filled[i]);
        if (s.stage_drained[i]) cudaEventDestroy(s.stage_drained[i]);
      }
      if (s.copy_stream) { cudaStreamSynchronize(s.copy_stream); cudaStreamDestroy(s.copy_stream); }
      for (int i = 0; i < 2; i++)
        if (s.step_ev[i]) cudaEventDestroy(s.step_ev[i]);
      if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (tb3_done) { cudaSetDevice(slabs[0].device); cudaFree(tb3_done); }
  }

  // LBM_GPU_POOL: the lattice and the staging buffer come from the device's stream-ordered
  // memory pool with an unlimited release threshold, so destroying a lattice and creating
  // the next one of a similar size (parameter sweeps, bench.py's end-to-end leg) reuses
  // the pages instead of paying cudaFree + cudaMalloc of ~20 GB each time (25-80 ms).
  // Not the default: the pool's first growth is slower than one cudaMalloc (0.4 s for
  // 19 GB), which a one-shot CLI run would pay for nothing, and the memory stays with the
  // process after lbm_gpu_destroy.  The window is always a plain allocation (CUDA IPC).
  bool use_pool() const { return (flags & LBM_GPU_POOL) != 0; }
  void pool_alloc(void** p, size_t bytes, Slab<real>& s) {
    if (use_pool()) {
      int supported = 0;
      CK(cudaDeviceGetAttribute(&supported, cudaDevAttrMemoryPoolsSupported, s.device));
      if (supported) {
        cudaMemPool_t pool;
        CK(cudaDeviceGetDefaultMemPool(&pool, s.device));
        unsigned long long keep = ~0ULL;
        CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        CK(cudaMallocAsync(p, bytes, s.stream));
        s.pooled = true;
        return;
      }
    }
    CK(cudaMalloc(p, bytes));
  }
  static void pool_free(void* p, Slab<real>& s) {
    if (!p) return;
    if (s.pooled) cudaFreeAsync(p, s.stream);
    else cudaFree(p);
  }
  // The window must be a plain cudaMalloc allocation (CUDA IPC), and a plain cudaFree
  // is a device-wide synchronisation that was measured to take up to 0.6 s when it follows
  // large transfers.  With LBM_GPU_POOL a destroyed lattice parks its window in a small
  // per-process cache instead and the next lattice of the same width picks it up.
  void window_alloc(Slab<real>& s) {
    if (use_pool()) {
      std::lock_guard<std::mutex> lock(g_window_mutex);
      for (size_t i = 0; i < g_window_cache.size(); i++)
        if (g_window_cache[i].device == s.device && g_window_cache[i].bytes == s.win_bytes) {
          s.win = g_window_cache[i].ptr;
          g_window_cache.erase(g_window_cache.begin() + i);
          return;
        }
    }
    CK(cudaMalloc((void**)&s.win, s.win_bytes));
  }
  void window_free(Slab<real>& s) {
    if (!s.win) return;
    if (use_pool()) {
      std::lock_guard<std::mutex> lock(g_window_mutex);
      g_window_cache.push_back({s.device, s.win_bytes, s.win});
    } else {
      cudaFree(s.win);
    }
    s.win = nullptr;
  }

  // ---------------------------------------------------------------- allocation ----
  void alloc_slab(Slab<real>& s) {
    CK(cudaSetDevice(s.device));
    const long long plane = (long long)s.rows * pitch;
    const size_t lat = (size_t)9 * plane * (f16 ? sizeof(__half) : sizeof(real));
    const size_t side = (size_t)6 * pitch * sizeof(real);
    const size_t maskb = (size_t)s.rows * mask_pitch * sizeof(uint32_t);
    size_t off = 0;
    for (int i = 0; i < 2; i++) { s.off_lattice[i] = off; off = round_up(off + lat, 256); }
    for (int i = 0; i < 2; i++) { s.off_side[i] = off; off = round_up(off + side, 256); }
    s.off_mask = off; off = round_up(off + maskb, 256);
    s.bytes = off;
    CK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&s.copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
      CK(cudaEventCreateWithFlags(&s.stage_filled[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&s.stage_drained[i], cudaEventDisableTiming));
    }
    pool_alloc((void**)&s.base, s.bytes, s);
    for (int i = 0; i < 2; i++) {
      s.lattice[i] = (real*)(s.base + s.off_lattice[i]);
      s.side[i] = (real*)(s.base + s.off_side[i]);
    }
    s.mask = (uint32_t*)(s.base + s.off_mask);
    // the window gets its own allocation, a multiple of 2 MiB so that it never shares a
    // driver block with anything else (it is exported over CUDA IPC)
    s.off_gmask = round_up((size_t)LBM_GHOST_PLANE_ROWS * pitch * sizeof(real), 256);
    s.off_sync = round_up(s.off_gmask + (size_t)2 * mask_pitch * sizeof(uint32_t), 256);
    s.win_bytes = round_up(s.off_sync + kSyncWords * sizeof(unsigned long long), 2u << 20);
    window_alloc(s);
    s.ghost_mask = (uint32_t*)(s.win + s.off_gmask);
    s.sync = (unsigned long long*)(s.win + s.off_sync);
    CK(cudaEventCreate(&s.ev0));
    CK(cudaEventCreate(&s.ev1));
    for (int i = 0; i < 2; i++) CK(cudaEventCreateWithFlags(&s.step_ev[i], cudaEventDisableTiming));
    CK(cudaMemsetAsync(s.base + s.off_side[0], 0, s.bytes - s.off_side[0], s.stream));
    CK(cudaMemsetAsync(s.win, 0, s.win_bytes, s.stream));
    void* st = nullptr;
    pool_alloc(&st, kStagingBytes, s);
    s.staging = st;
  }

  // K1c: one 3-D tensor map (x, row, plane) per lattice buffer, box = one row of a tile
  void make_tensor_maps(Slab<real>& s) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                 const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                 CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) throw CudaError{"cuTensorMapEncodeTiled is not available in this driver"};
    const cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)s.rows, 9};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * sizeof(real), (cuuint64_t)plane_stride(s) * sizeof(real)};
    const cuuint32_t box[3] = {LBM_TMA_BOX, 1, 1};
    const cuuint32_t hbox[3] = {4, 1, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    for (int b = 0; b < 2; b++) {
      for (int h = 0; h < 2; h++) {
        const CUresult r = ((EncodeFn)fn)(h ? &s.tmap_halo[b] : &s.tmap[b], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, s.lattice[b],
                                          dims, strides, h ? hbox : box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
          char msg[96];
          snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
          throw CudaError{msg};
        }
      }
    }
  }

  // ghost rows of a window: parity b, direction d (0 = "from below", 1 = "from above")
  real* win_section(char* win, int b, int d) const { return (real*)win + lbm::ghost_offset(pitch, b, d); }

  long long plane_stride(const Slab<real>& s) const { return (long long)s.rows * pitch; }

  // LBM_GPU_STORE_F16: the binary16 view of a lattice buffer, and the shift of each speed
  // (the rest state, computed as load_slab computes it)
  __half* hlat(const Slab<real>& s, int b) const { return reinterpret_cast<__half*>(s.lattice[b]); }
  lbm::RestShift rest() const {
    lbm::RestShift r;
    r.w0 = (float)(prm.density * (real)4 / (real)9);
    r.w1 = (float)(prm.density / (real)9);
    r.w2 = (float)(prm.density / (real)36);
    return r;
  }

  void setup_geometry(int nx) {
    pitch = (int)round_up(nx, 32);
    mask_pitch = pitch / 32;
    if (const char* e = getenv("LBM_GPU_SYNC_TIMEOUT_MS")) {      // longest wait for a neighbouring slab
      const double ms = atof(e);
      if (ms > 0) timeout_ns = (unsigned long long)(ms * 1e6);
    }
  }

  // launch shape shared by the step kernels: blockDim (bx, by), tiles of bx*vec x by cells
  void tile_shape(int vec, int& bx, int& by) const {
    const int nxv = (prm.nx + vec - 1) / vec;
    bx = (int)std::min<long long>(LBM_BLOCK_THREADS, round_up(nxv, 32));
    if (kernel == LBM_GPU_KERNEL_TMA) bx = LBM_BLOCK_THREADS;     // one row of LBM_TMA_TILE cells per block
    by = LBM_BLOCK_THREADS / bx;
  }

  // blocks of lbm_steps_persistent that can be resident at once on the slab's GPU
  const void* persistent_fn() const {
    const bool strict = (flags & LBM_GPU_STRICT) != 0;
    if (persistent_vec == 1)
      return strict ? (const void*)lbm::lbm_steps_persistent<real, true, 1> : (const void*)lbm::lbm_steps_persistent<real, false, 1>;
    return strict ? (const void*)lbm::lbm_steps_persistent<real, true, 4> : (const void*)lbm::lbm_steps_persistent<real, false, 4>;
  }

  int persistent_capacity(const Slab<real>& s) {
    int per_sm = 0, sms = 0, coop = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, persistent_fn(), LBM_BLOCK_THREADS, 0));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s.device));
    CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, s.device));
    return coop ? per_sm * sms : 0;
  }

  const void* cluster_fn() const {
    return (flags & LBM_GPU_STRICT) ? (const void*)lbm::lbm_steps_cluster<true> : (const void*)lbm::lbm_steps_cluster<false>;
  }

  // K6 applies to a single fp32 slab whose double-buffered lattice fits in the shared memory
  // of one cluster (16 CTAs if the device schedules such a cluster, else 8).
  bool cluster_fits() {
    if (sizeof(real) != 4 || slabs.size() != 1 || slab_mode) return false;
    Slab<real>& s = slabs[0];
    int max_smem = 0;
    CK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, s.device));
    for (int c : {16, 8}) {
      const int rows = (s.rows + c - 1) / c;
      const size_t smem = (size_t)2 * 9 * rows * prm.nx * sizeof(float);
      if (smem > (size_t)max_smem) continue;
      if (cudaFuncSetAttribute(cluster_fn(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
          cudaFuncSetAttribute(cluster_fn(), cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
        continue;
      }
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(c);
      cfg.blockDim = dim3(LBM_CLUSTER_THREADS);
      cfg.dynamicSmemBytes = smem;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = c; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      int nclusters = 0;
      if (cudaOccupancyMaxActiveClusters(&nclusters, cluster_fn(), &cfg) != cudaSuccess || nclusters < 1) {
        cudaGetLastError();
        continue;
      }
      cluster_ctas = c;
      cluster_rows = rows;
      cluster_smem = smem;
      return true;
    }
    return false;
  }

  // K5 on the single slab: one or four cells per thread; false without cooperative launch
  bool persistent_fits() {
    // tiny grids: one cell per thread (4x the threads on the step's dependent-latency chain)
    // as long as that does not put more than kPersistScalarBlocks blocks on the grid barrier
    int bx, by;
    tile_shape(1, bx, by);
    const long long tiles = (long long)((prm.nx + bx - 1) / bx) * ((slabs[0].rows + by - 1) / by);
    persistent_vec = 1;
    int cap = persistent_capacity(slabs[0]);
    long long scalar_limit = std::min<long long>(cap, kPersistScalarBlocks);
    if (const char* e = getenv("LBM_PERSIST_VEC"))      // measurement knob of profiles/r01_small_grids.md
      scalar_limit = (atoi(e) == 1) ? cap : 0;
    if (tiles > scalar_limit) {
      persistent_vec = 4;
      cap = persistent_capacity(slabs[0]);
    }
    return cap >= 1;
  }

  // K7 (two timesteps per pass) needs fp32, a width the 16-byte bulk copies can cut (multiple
  // of 4; of 8 for binary16 rows), slabs tall enough for two-row ghost zones, and no other
  // kernel forced by the caller.  Every slab of the grid must come to the same answer: the
  // ghost-row pushes and the flag protocol count passes, not timesteps.
  bool k7_fits(int rows_min) const {
    const unsigned k = forced_kernel(flags);
    if (k != 0 && k != LBM_GPU_KERNEL_TB2 && k != LBM_GPU_KERNEL_TB3) return false;
    if (f16) return prm.nx % 8 == 0 && prm.nx >= 32 && rows_min >= kTb2MinRows;
    return sizeof(real) == 4 && !env_on("LBM_GPU_NO_TB2") && prm.nx % 4 == 0 && prm.nx >= 32 && rows_min >= kTb2MinRows;
  }

  void configure_tb2() {
    if constexpr (sizeof(real) == 4) {
      for (auto& s : slabs) {
        CK(cudaSetDevice(s.device));
        if (f16) {
          for (const void* fn : {(const void*)lbm::lbm_step2_tb_f16<false>, (const void*)lbm::lbm_step2_tb_f16<true>})
            CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(lbm::Tb2hSmem)));
          continue;
        }
        for (const void* fn : {(const void*)lbm::lbm_step2_tb<false, false>, (const void*)lbm::lbm_step2_tb<false, true>,
                               (const void*)lbm::lbm_step2_tb<true, false>, (const void*)lbm::lbm_step2_tb<true, true>})
          CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(lbm::Tb2Smem)));
      }
      // K7-f16 has a halo of 8 columns and owns multiples of 8 (16-byte bulk copies of binary16)
      const int pad = f16 ? LBM_TB2H_PAD : LBM_TB2_PAD, max_wout = f16 ? LBM_TB2H_MAX_WOUT : LBM_TB2_MAX_WOUT;
      if (prm.nx + 2 * pad <= LBM_TB2_SPAN) {      // narrow grid: one strip, the whole width plus halo
        tb2_strips = 1;
        tb2_wout = prm.nx;
        tb2_span = prm.nx + 2 * pad;
      } else {
        tb2_strips = (prm.nx + max_wout - 1) / max_wout;
        tb2_wout = (int)round_up((prm.nx + tb2_strips - 1) / tb2_strips, f16 ? 8 : 4);
        tb2_span = LBM_TB2_SPAN;
      }
      tb2_threads = (int)round_up(tb2_span / 4, 32);
      // segment height: every segment recomputes two rows of the first sub-step, so tall is cheap
      int rows_max = 0;
      for (auto& s : slabs) rows_max = std::max(rows_max, s.rows);
      const double resident = (double)LBM_TB2_MIN_BLOCKS * sm_count();
      tb2_seg_rows = best_segment_rows(rows_max, resident, 2, 128);
      if (const char* e = getenv("LBM_TB2_SEG_ROWS")) tb2_seg_rows = std::max(2, atoi(e));   // tuning knob
      // A block lives (segment height) x ~2.6 us; the last blocks of a launch to be scheduled
      // leave the other SMs idle for about half of that.  So the launch ENDS with short
      // segments -- one set of resident blocks' worth, given the highest block indices -- and the
      // SMs drain together (tall slabs only: the short segments pay 2 halo rows per 16).
      tb2_tail_segs = (int)((resident + tb2_strips - 1) / tb2_strips) + 1;
      if (const char* e = getenv("LBM_TB2_TAIL_ROWS")) tb2_tail_rows = atoi(e);                // tuning knob, 0 = off
      if (tb2_tail_rows < 2) tb2_tail_segs = 0;
    }
  }

  int sm_count() const {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, slabs[0].device);
    return sms;
  }
  // blocks of a launch of `rows` rows in segments of h rows, in waves of `resident` blocks
  double tb_waves(int rows, int h, double resident) const { return (double)tb2_strips * ((rows + h - 1) / h) / resident; }
  // Segment height of K7 (extra = 2 recomputed rows) and K10 (4).  The blocks of a launch run
  // in "waves" of the resident blocks and a last wave that is nearly empty leaves the SMs idle
  // (16384 rows in 64-row segments: 19.03 waves of K7).  Score each height by
  // (rows / (rows + extra)) x (waves / ceil(waves)) and take the best; grids with few blocks
  // prefer short segments so that there are several waves at all.
  int best_segment_rows(int rows, double resident, int extra, int h_max) const {
    double best = -1.0;
    int best_h = 64;
    for (int h = 16; h <= h_max; h++) {
      const double waves = tb_waves(rows, h, resident);
      const double score = (double)h / (h + extra) * waves / std::ceil(waves) * (waves >= 4.0 ? 1.0 : 0.25 * waves);
      if (score > best + 1e-9) { best = score; best_h = h; }
    }
    return best_h;
  }

  // K10 (three timesteps per pass) on top of K7: one slab that holds the whole grid (its
  // rows beyond the ends are its own, so no three-deep ghost zones are needed), at least
  // kTb3MinRows rows, fp32 storage, and the K7 conditions.
  bool k10_fits() const {
    return slabs.size() == 1 && slabs[0].rows == prm.ny && slabs[0].row0 == 0 && !f16 && k7_fits(slabs[0].rows) &&
           slabs[0].rows >= kTb3MinRows && !env_on("LBM_GPU_NO_TB3");
  }
  // Default: K10 where its blocks fill at least two waves of the SMs.  At four blocks per SM it
  // measured faster than K7 on every size swept (1.15 x at 16384 x 2048, 2.4 waves;
  // profiles/r07_k10_four_blocks.md); below two waves (4096^2: 1.2) K7 stays, where the launch
  // tail of K10's longer blocks weighs most.
  bool tb3_pays() const {
    const double resident = (double)LBM_TB3_MIN_BLOCKS * sm_count();
    return tb_waves(slabs[0].rows, 64, resident) >= kTb3MinWaves;
  }
  void configure_tb3() {
    if constexpr (sizeof(real) == 4) {
      Slab<real>& s = slabs[0];
      CK(cudaSetDevice(s.device));
      for (const void* fn : {(const void*)lbm::lbm_step3_tb<false>, (const void*)lbm::lbm_step3_tb<true>})
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(lbm::Tb3Smem)));
      const double resident = (double)LBM_TB3_MIN_BLOCKS * sm_count();
      // Passes that do not overlap end in a tail: the wave score picks 88 rows at 16384^2, where
      // 80-112 rows are within 0.7 % of each other (profiles/r07_k10_four_blocks.md).  Overlapped
      // passes have no tail between them, so taller segments pay less halo: 192 rows measured
      // 2.3 % faster than 88 at 16384^2 (profiles/r08_k10_overlap.md); the wave score stays for
      // launches of fewer than two waves at that height.
      const bool overlap = use_pdl() && !env_on("LBM_GPU_NO_TB3_OVERLAP");
      tb3_seg_rows = (overlap && tb_waves(s.rows, kTb3OverlapSegRows, resident) >= 2.0)
                         ? kTb3OverlapSegRows : best_segment_rows(s.rows, resident, 4, 96);
      if (const char* e = getenv("LBM_TB3_SEG_ROWS")) tb3_seg_rows = std::max(1, atoi(e));   // tuning knob
      tb3_overlap = overlap && tb3_overlap_fits(s.rows);
      if (tb3_overlap && !tb3_done) {
        const size_t bytes = (size_t)tb2_strips * tb3_segments(s.rows).n_big * sizeof(uint32_t);
        CK(cudaMalloc((void**)&tb3_done, bytes));
        // No reset is needed later (upload, a K7 or K1a pass in between): the first K10 pass after
        // anything else waits for the whole previous grid and then publishes every tile.
        CK(cudaMemset(tb3_done, 0, bytes));
      }
    }
  }
  // Overlapped K10 passes order a tile after the 3 x 3 neighbourhood of its tile in the previous
  // pass.  That neighbourhood holds every tile whose cells it reads (rows R0-3 .. R1+2, the
  // staged columns) and, the relation being symmetric, every tile that reads the cells it
  // writes, if no tile reads beyond the strips and segments next to it: false for segments of
  // fewer than three rows, or a last strip narrower than the halo.
  bool tb3_overlap_fits(int rows) const {
    const Tb2Segments g = tb3_segments(rows);
    auto near = [](int a, int b, int n) { const int d = (a - b + n) % n; return d <= 1 || d == n - 1; };
    for (int seg = 0; seg < g.n_big; seg++) {
      const int r0 = seg * g.seg_rows, r1 = std::min(r0 + g.seg_rows, rows);
      for (int r = r0 - 3; r < r1 + 3; r++)
        if (!near(((r % rows) + rows) % rows / g.seg_rows, seg, g.n_big)) return false;
    }
    for (int strip = 0; strip < tb2_strips; strip++)
      for (int c = strip * tb2_wout - LBM_TB2_PAD; c < strip * tb2_wout - LBM_TB2_PAD + tb2_span; c++)
        if (!near(((c % prm.nx) + prm.nx) % prm.nx / tb2_wout, strip, tb2_strips)) return false;
    return true;
  }

  // segments of a slab for K7: n_big segments of equal height, then (tall slabs) n_tail short
  // ones; the last segment keeps at least two rows (the rows that push into the neighbour
  // above must sit in an edge segment)
  struct Tb2Segments { int seg_rows, n_big, big_rows, seg_rows_tail, n_tail; };
  Tb2Segments tb2_segments(int rows) const {
    Tb2Segments g;
    // measured (profiles/r02_kernel_variants.md): +1.2 % on 16384 rows, nothing on 8192, -2 % on 2048
    const long long min_rows = (long long)tb2_tail_segs * tb2_tail_rows * (tb2_tail_rows >= 8 ? 32 : 4);
    g.n_tail = (tb2_tail_segs > 0 && min_rows <= rows) ? tb2_tail_segs : 0;
    g.seg_rows_tail = tb2_tail_rows;
    g.big_rows = rows - g.n_tail * g.seg_rows_tail;
    int nsegs = std::max(1, (g.big_rows + tb2_seg_rows - 1) / tb2_seg_rows);
    for (;;) {
      g.seg_rows = (g.big_rows + nsegs - 1) / nsegs;
      nsegs = (g.big_rows + g.seg_rows - 1) / g.seg_rows;
      if (nsegs == 1 || g.n_tail > 0 || g.big_rows - (nsegs - 1) * g.seg_rows >= 2) break;
      nsegs--;
    }
    g.n_big = nsegs;
    return g;
  }

  // segments of the slab for K10: equal heights (one slab: no rows need to sit in edge segments)
  Tb2Segments tb3_segments(int rows) const {
    Tb2Segments g;
    const int nsegs = (rows + tb3_seg_rows - 1) / tb3_seg_rows;
    g.seg_rows = g.seg_rows_tail = (rows + nsegs - 1) / nsegs;
    g.n_big = (rows + g.seg_rows - 1) / g.seg_rows;
    g.big_rows = rows;
    g.n_tail = 0;
    return g;
  }

  // K9 (two timesteps per grid barrier) for the small grids the persistent kernel K5 would
  // take: single GPU, fp32, nx a multiple of 4 and at most 256, every block resident.  pairs_fit()
  // checks them and sets the tile rows.
  const void* pairs_fn() const {
    if constexpr (sizeof(real) == 4)
      return (flags & LBM_GPU_STRICT) ? (const void*)lbm::lbm_steps_pairs<true> : (const void*)lbm::lbm_steps_pairs<false>;
    return nullptr;
  }
  dim3 pairs_block() const { return dim3((unsigned)round_up(prm.nx / 4, 32), (unsigned)(pairs_tile_rows + 2)); }
  size_t pairs_smem() const { return (size_t)(pairs_tile_rows + 2) * 9 * prm.nx * sizeof(float); }

  bool pairs_fit() {
    if (!(sizeof(real) == 4 && slabs.size() == 1 && !slab_mode && prm.nx % 4 == 0 && prm.nx >= 4 &&
          prm.nx <= LBM_PAIRS_MAX_NX && slabs[0].rows >= 4))
      return false;
    Slab<real>& s = slabs[0];
    int sms = 0, coop = 0, per_sm = 0;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s.device));
    CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, s.device));
    // one block per SM if the grid allows it: the fewest rows per block that still fits
    pairs_tile_rows = std::min(LBM_PAIRS_MAX_TILE_ROWS, std::max(1, (s.rows + sms - 1) / sms));
    if (const char* e = getenv("LBM_PAIRS_TILE_ROWS"))                      // tuning knob
      pairs_tile_rows = std::min(LBM_PAIRS_MAX_TILE_ROWS, std::max(1, atoi(e)));
    pairs_tile_rows = std::min(pairs_tile_rows, s.rows - 2);
    const dim3 b = pairs_block();
    const bool ok = coop && cudaFuncSetAttribute(pairs_fn(), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pairs_smem()) == cudaSuccess &&
                    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pairs_fn(), (int)(b.x * b.y), pairs_smem()) == cudaSuccess &&
                    (long long)per_sm * sms >= (s.rows + pairs_tile_rows - 1) / pairs_tile_rows;
    cudaGetLastError();
    return ok;
  }

  // ------------------------------------------------------------ kernel choice ----
  // Which kernel runs the lattice, and its launch configuration: the only code that sets
  // `kernel`.  Runs before anything is allocated, and again when a slab handle joins a ring of
  // processes (`ring_k7`: lbm_gpu_ipc_connect_all found that every rank can run K7):
  //   0. refused on flags and shape alone: two kernels, TMA in fp64, binary16 outside one fp32
  //      lbm_gpu_create slab or with a kernel other than VEC4 or TB2;
  //   1. a forced kernel where its conditions hold, otherwise a refusal;
  //   2. a ring: K7 where every rank can run it, otherwise K1a;
  //   3. one lbm_gpu_create slab in L2 (kPersistMaxCells): K9 where it fits (unless LBM_GPU_NO_PAIRS), else K5;
  //   4. K7 (K7-f16) where it fits, but not yet on a slab handle that holds part of the grid; K10
  //      instead on the whole grid in one slab with enough waves of blocks (unless LBM_GPU_NO_TB3);
  //   5. K1a (K1a-f16).
  void select_kernel(bool ring = false, bool ring_k7 = false) {
    const unsigned forced = forced_kernel(flags);
    if (f16) {
      if (slab_mode) throw CudaError{"LBM_GPU_STORE_F16 is for lbm_gpu_create lattices only, not slab handles"};
      if (sizeof(real) != 4) throw CudaError{"LBM_GPU_STORE_F16 is for fp32 lattices only"};
      if (slabs.size() != 1) throw CudaError{"LBM_GPU_STORE_F16 needs n_gpus == 1 (got " + std::to_string(slabs.size()) + ")"};
      if (forced & ~(LBM_GPU_KERNEL_VEC4 | LBM_GPU_KERNEL_TB2)) {
        char msg[160];
        snprintf(msg, sizeof msg, "LBM_GPU_STORE_F16 runs LBM_GPU_KERNEL_VEC4 or LBM_GPU_KERNEL_TB2 only; "
                 "another kernel was forced (flags 0x%x)", forced);
        throw CudaError{msg};
      }
    }
    if (forced == LBM_GPU_KERNEL_TMA && sizeof(real) != 4) throw CudaError{"the TMA kernel is built for single precision only"};
    const bool one_slab = slabs.size() == 1 && !slab_mode;
    const bool partial = slab_mode && slabs[0].rows != prm.ny;
    int rows_min = slabs[0].rows;
    for (auto& s : slabs) rows_min = std::min(rows_min, s.rows);
    CK(cudaSetDevice(slabs[0].device));
    bool k7 = false;
    switch (forced) {
      case 0:
        if (!ring && !f16 && one_slab && (long long)prm.nx * slabs[0].rows <= kPersistMaxCells && persistent_fits()) {
          kernel = (!env_on("LBM_GPU_NO_PAIRS") && pairs_fit()) ? LBM_GPU_KERNEL_PAIRS : LBM_GPU_KERNEL_PERSISTENT;
          return;
        }
        k7 = ring ? ring_k7 : !partial && k7_fits(rows_min);
        break;
      case LBM_GPU_KERNEL_PERSISTENT:
        if (!one_slab) throw CudaError{"the persistent kernel handles a single slab only"};
        if (!persistent_fits()) throw CudaError{"cooperative launch is not available on this device"};
        break;
      // K6 is opt-in only: 16 SMs doing all the arithmetic are no faster than K5 spreading it
      // over the whole chip (profiles/r01_small_grids.md).
      case LBM_GPU_KERNEL_CLUSTER:
        if (!cluster_fits()) throw CudaError{"the cluster kernel needs a single-GPU fp32 lattice that fits in one cluster's shared memory"};
        break;
      case LBM_GPU_KERNEL_PAIRS:
        if (!pairs_fit()) throw CudaError{"the pairs kernel needs a single-GPU fp32 lattice with nx a multiple of 4 and <= 256 whose blocks are all resident"};
        break;
      case LBM_GPU_KERNEL_TB2:
        if (ring && !ring_k7)
          throw CudaError{"the two-step kernel needs lbm_gpu_ipc_connect_all and fp32, nx a multiple of 4 and >= 32, "
                          ">= 8 rows on every rank"};
        if (!ring && !partial && !k7_fits(rows_min))
          throw CudaError{f16 ? "the two-step kernel with LBM_GPU_STORE_F16 needs nx a multiple of 8 and >= 32, and >= 8 rows"
                              : "the two-step kernel needs fp32, nx a multiple of 4 and >= 32, and >= 8 rows per slab"};
        k7 = ring || !partial;
        break;
      case LBM_GPU_KERNEL_TB3:
        if (ring) throw CudaError{"the three-step kernel needs the whole grid in one slab"};
        if (!k10_fits()) throw CudaError{"the three-step kernel needs fp32, nx a multiple of 4 and >= 32, the whole grid in one slab, and >= 12 rows"};
        k7 = true;
        break;
    }
    if (!k7) {
      kernel = (forced && forced != LBM_GPU_KERNEL_TB2) ? forced : LBM_GPU_KERNEL_VEC4;
      return;
    }
    configure_tb2();
    kernel = LBM_GPU_KERNEL_TB2;
    if (forced == LBM_GPU_KERNEL_TB3 || (!forced && !ring && k10_fits() && tb3_pays())) {
      configure_tb3();
      kernel = LBM_GPU_KERNEL_TB3;
    }
  }

  // timesteps of the kernel's longest pass: K10 three, K7 and K7-f16 two, the others one
  int max_pass_steps() const { return kernel == LBM_GPU_KERNEL_TB3 ? 3 : kernel == LBM_GPU_KERNEL_TB2 ? 2 : 1; }

  // ------------------------------------------------------------- lattice input ----
  // cells: AoS rows for this slab (or NULL -> rest state); obstacles: rows for this slab
  void load_slab(Slab<real>& s, const real* cells_aos, const void* obstacles, int cur) {
    CK(cudaSetDevice(s.device));
    const int nx = prm.nx;
    if (cells_aos) {
      upload_cells(s, cells_aos, cur);
    } else if (f16) {
      CK(cudaMemsetAsync(s.lattice[cur], 0, (size_t)9 * plane_stride(s) * sizeof(__half), s.stream));   // the rest state
    } else {
      const real w0 = prm.density * (real)4 / (real)9;     // d2q9-bgk.c:2802-2804
      const real w1 = prm.density / (real)9;
      const real w2 = prm.density / (real)36;
      const long long total = plane_stride(s);
      lbm::lbm_init_rest<real><<<(unsigned)((total + 255) / 256), 256, 0, s.stream>>>(
          s.lattice[cur], plane_stride(s), pitch, nx, s.rows, w0, w1, w2);
      CK(cudaGetLastError());
      launches++;
    }
    // mask
    unsigned long long* counter = s.sync + kScratch0;
    CK(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), s.stream));
    if (obstacles) {
      // host rows -> one half of the staging buffer (copy stream) -> packed into the mask
      // (kernel stream); the copy of chunk i+1 overlaps the packing of chunk i, one
      // synchronisation per call
      const bool bits = (flags & LBM_GPU_OBST_BITS) != 0;
      const int wpr = (nx + 31) / 32;
      const size_t row_bytes = bits ? (size_t)wpr * 4 : (size_t)nx * 4;
      const size_t half = kStagingBytes / 2;
      if (row_bytes > half) throw CudaError{"nx too large for the obstacle staging buffer"};
      const int chunk_rows = (int)(half / row_bytes);
      CK(cudaEventRecord(s.stage_drained[0], s.stream));       // orders the first copies behind the memsets above
      CK(cudaEventRecord(s.stage_drained[1], s.stream));
      int i = 0;
      for (int r = 0; r < s.rows; r += chunk_rows, i++) {
        const int n = std::min(chunk_rows, s.rows - r);
        const int b = i & 1;
        char* st = (char*)s.staging + (size_t)b * half;
        CK(cudaStreamWaitEvent(s.copy_stream, s.stage_drained[b], 0));
        CK(cudaMemcpyAsync(st, (const char*)obstacles + (size_t)r * row_bytes, (size_t)n * row_bytes,
                           cudaMemcpyHostToDevice, s.copy_stream));
        CK(cudaEventRecord(s.stage_filled[b], s.copy_stream));
        CK(cudaStreamWaitEvent(s.stream, s.stage_filled[b], 0));
        if (bits) {
          const long long words = (long long)n * wpr;
          lbm::lbm_copy_mask_bits<<<(unsigned)((words + 255) / 256), 256, 0, s.stream>>>(
              (const uint32_t*)st, s.mask, mask_pitch, nx, r, n, counter);
        } else {
          const long long threads = (long long)n * wpr * 32;
          lbm::lbm_pack_mask<<<(unsigned)((threads + 255) / 256), 256, 0, s.stream>>>(
              (const int*)st, s.mask, mask_pitch, nx, r, n, counter);
        }
        CK(cudaGetLastError());
        launches++;
        CK(cudaEventRecord(s.stage_drained[b], s.stream));
      }
    }
    unsigned long long blocked = 0;
    CK(cudaMemcpyAsync(&blocked, counter, sizeof blocked, cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    s.free_cells = (long long)s.rows * nx - (long long)blocked;
  }

  void upload_cells(Slab<real>& s, const real* cells_aos, int cur) {
    CK(cudaSetDevice(s.device));
    const int nx = prm.nx;
    const size_t row_bytes = (size_t)nx * 9 * sizeof(real);
    const int chunk_rows = (int)std::max<size_t>(1, kStagingBytes / row_bytes);
    if (row_bytes > kStagingBytes) throw CudaError{"nx too large for the AoS staging buffer"};
    for (int r = 0; r < s.rows; r += chunk_rows) {
      const int n = std::min(chunk_rows, s.rows - r);
      const long long ncells = (long long)n * nx;
      CK(cudaMemcpyAsync(s.staging, (const char*)cells_aos + (size_t)r * row_bytes, (size_t)n * row_bytes,
                         cudaMemcpyHostToDevice, s.stream));
      if (f16)
        lbm::lbm_aos_to_soa<real, __half><<<(unsigned)((ncells * 9 + 255) / 256), 256, 0, s.stream>>>(
            (const real*)s.staging, hlat(s, cur), plane_stride(s), pitch, nx, r, ncells, rest());
      else
        lbm::lbm_aos_to_soa<real><<<(unsigned)((ncells * 9 + 255) / 256), 256, 0, s.stream>>>(
            (const real*)s.staging, s.lattice[cur], plane_stride(s), pitch, nx, r, ncells);
      CK(cudaGetLastError());
      launches++;
      CK(cudaStreamSynchronize(s.stream));
    }
  }

  // ------------------------------------------------------------------ wiring ----
  // all slabs live in this process: neighbours are reached through peer access
  void connect_local() {
    const int n = (int)slabs.size();
    for (int i = 0; i < n; i++) {
      Slab<real>& s = slabs[i];
      Slab<real>& up = slabs[(i + 1) % n];
      Slab<real>& dn = slabs[(i + n - 1) % n];
      CK(cudaSetDevice(s.device));
      for (Slab<real>* o : {&up, &dn}) {
        if (o->device != s.device) {
          int can = 0;
          CK(cudaDeviceCanAccessPeer(&can, s.device, o->device));
          if (!can) throw CudaError{"peer access between the selected GPUs is not available"};
          cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
          if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
          cudaGetLastError();
        }
      }
      s.up_win = up.win;
      s.dn_win = dn.win;
      s.up_flag = up.sync + kFlagFromBelow;
      s.dn_flag = dn.sync + kFlagFromAbove;
      s.up_abort = up.sync + kAbort;
      s.dn_abort = dn.sync + kAbort;
      s.up_gmask = up.ghost_mask;
      s.dn_gmask = dn.ghost_mask + mask_pitch;
    }
    multi = n > 1;
    // Slabs of one process are ordered by the device-side flag protocol (edge blocks wait,
    // interior blocks never do) whenever every slab has a GPU of its own; slabs that share a
    // GPU (tests on a one-GPU box) cannot wait on one another inside kernels and are ordered
    // by CUDA events, as is everything when LBM_GPU_SYNC_EVENTS asks for it.
    bool distinct = true;
    for (int i = 0; i < n; i++)
      for (int j = i + 1; j < n; j++)
        if (slabs[i].device == slabs[j].device) distinct = false;
    if ((flags & LBM_GPU_SYNC_FLAGS) && multi && !distinct)
      throw CudaError{"LBM_GPU_SYNC_FLAGS needs every slab on its own GPU (kernels that wait on "
                      "one another must not share a device)"};
    use_flags = multi && distinct && !(flags & LBM_GPU_SYNC_EVENTS);
    connected = true;
  }

  void prepare() {
    if (!connected) throw CudaError{"lattice is not connected to its neighbours yet"};
    if (f16) {            // one slab that holds the whole grid: no ghost rows, only the side row
      Slab<real>& s = slabs[0];
      CK(cudaSetDevice(s.device));
      lbm::lbm_prepare_f16<<<(prm.nx + 127) / 128, 128, 0, s.stream>>>(
          hlat(s, cur), (float*)s.side[cur], s.mask, plane_stride(s), prm.nx, pitch, mask_pitch, s.accel_row, rest(),
          (float)(prm.density * prm.accel / (real)9), (float)(prm.density * prm.accel / (real)36));
      CK(cudaGetLastError());
      launches++;
      CK(cudaStreamSynchronize(s.stream));
      return;
    }
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      lbm::PrepareArgs<real> a;
      a.cur = s.lattice[cur];
      a.side_cur = s.side[cur];
      a.mask = s.mask;
      a.push_up = win_section(s.up_win, cur, 0);
      a.push_dn = win_section(s.dn_win, cur, 1);
      a.mask_up = s.up_gmask;
      a.mask_dn = s.dn_gmask;
      a.plane_stride = plane_stride(s);
      a.nx = prm.nx; a.rows = s.rows; a.pitch = pitch; a.mask_pitch = mask_pitch; a.accel_row = s.accel_row;
      a.deep = max_pass_steps() > 1 ? 1 : 0;   // K10 reads the source lattice directly: K7's ghost rows are enough
      a.aw1 = prm.density * prm.accel / (real)9;      // d2q9-bgk.c:230-231
      a.aw2 = prm.density * prm.accel / (real)36;
      lbm::lbm_prepare<real><<<(std::max(prm.nx, mask_pitch) + 127) / 128, 128, 0, s.stream>>>(a);
      CK(cudaGetLastError());
      launches++;
    }
    for (auto& s : slabs) { CK(cudaSetDevice(s.device)); CK(cudaStreamSynchronize(s.stream)); }
    loaded_unprepared = false;
  }

  // -------------------------------------------------------------------- run ----
  template <bool STRICT, bool MULTI>
  void launch_step(Slab<real>& s, const lbm::StepArgs<real>& a, dim3 grid, dim3 block, int src) {
    if (kernel == LBM_GPU_KERNEL_SCALAR)
      lbm::lbm_step_scalar<real, STRICT, MULTI><<<grid, block, 0, s.stream>>>(a);
    else if (kernel == LBM_GPU_KERNEL_TMA)
      launch_tma<STRICT, MULTI>(s, a, grid, block, src);
    else
      launch_vec4<STRICT, MULTI>(s, a, grid, block);
  }
  // Step kernels go out with programmatic stream serialization (PDL): the next pass's grid
  // is set up while the current one drains, which hides the launch gap on mid-size grids.
  static bool use_pdl() {
    static const bool pdl = !(getenv("LBM_GPU_NO_PDL") && getenv("LBM_GPU_NO_PDL")[0] == '1');
    return pdl;
  }
  template <typename Kernel, typename Args>
  void launch_pdl(Slab<real>& s, Kernel k, const Args& a, dim3 grid, dim3 block, size_t smem) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s.stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = use_pdl() ? 1 : 0;
    CK(cudaLaunchKernelEx(&cfg, k, a));
  }
  template <bool STRICT, bool MULTI>
  void launch_vec4(Slab<real>& s, const lbm::StepArgs<real>& a, dim3 grid, dim3 block) {
    launch_pdl(s, lbm::lbm_step_vec4<real, STRICT, MULTI>, a, grid, block, 0);
  }
  template <bool STRICT, bool MULTI>
  void launch_tma(Slab<real>& s, const lbm::StepArgs<real>& a, dim3 grid, dim3 block, int src) {
    if constexpr (sizeof(real) == 4)
      lbm::lbm_step_tma<STRICT, MULTI><<<grid, block, 0, s.stream>>>(a, s.tmap[src], s.tmap_halo[src]);
  }
  template <bool STRICT, bool MULTI>
  void launch_tb2(Slab<real>& s, const lbm::Tb2Args& ta, dim3 grid) {
    if constexpr (sizeof(real) == 4)
      launch_pdl(s, lbm::lbm_step2_tb<STRICT, MULTI>, ta, grid, dim3(tb2_threads), sizeof(lbm::Tb2Smem));
  }
  template <bool STRICT>
  void launch_tb3(Slab<real>& s, const lbm::Tb2Args& ta, dim3 grid) {
    if constexpr (sizeof(real) == 4)
      launch_pdl(s, lbm::lbm_step3_tb<STRICT>, ta, grid, dim3(tb2_threads), sizeof(lbm::Tb3Smem));
  }

  void launch_cluster(int n_steps, bool strict) {
    if constexpr (sizeof(real) == 4) {
      Slab<real>& s = slabs[0];
      CK(cudaSetDevice(s.device));
      lbm::ClusterArgs a;
      a.src = s.lattice[cur];
      a.dst = s.lattice[(cur + n_steps) & 1];
      a.mask = s.mask;
      a.av = s.av;
      a.plane_stride = plane_stride(s);
      a.nx = prm.nx; a.ny = s.rows; a.pitch = pitch; a.mask_pitch = mask_pitch;
      a.rows_per_cta = cluster_rows;
      a.n_steps = n_steps;
      a.omega = prm.omega;
      a.aw1 = prm.density * prm.accel / 9.f;
      a.aw2 = prm.density * prm.accel / 36.f;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(cluster_ctas);
      cfg.blockDim = dim3(LBM_CLUSTER_THREADS);
      cfg.dynamicSmemBytes = cluster_smem;
      cfg.stream = s.stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = cluster_ctas; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      if (strict) CK(cudaLaunchKernelEx(&cfg, lbm::lbm_steps_cluster<true>, a));
      else CK(cudaLaunchKernelEx(&cfg, lbm::lbm_steps_cluster<false>, a));
      launches++;
    }
    (void)n_steps; (void)strict;
  }

  // The per-step sums take 1 KiB of device memory per step, so very long runs are cut into
  // segments of kMaxSegmentSteps (one sync + one read-back per segment, no other effect).
  void run(int n_steps, double* sums_out) {
    if (!connected) throw CudaError{"lattice is not connected to its neighbours yet"};
    if (failed) throw CudaError{"an earlier run of this lattice was abandoned (a neighbouring slab never arrived); "
                                "its contents are void"};
    if (loaded_unprepared)
      throw CudaError{"rows were loaded into this slab handle with lbm_gpu_load_rows and its neighbours' ghost rows are "
                      "stale: pass a host barrier over all ranks, lbm_gpu_ipc_prepare, and a second barrier first"};
    double ms = 0.0;
    const int total = n_steps;
    for (int done = 0; done < total; done += kMaxSegmentSteps) {
      const int n = std::min(kMaxSegmentSteps, total - done);
      run_segment(n, sums_out ? sums_out + done : nullptr);
      ms += last_run_ms;
    }
    if (total > 0) {
      last_run_ms = ms;
      last_step_ms = ms / total;
    }
  }

  // arguments common to every kernel of one pass on one slab: reads buffer `cur`, writes cur^1
  void fill_step_args(lbm::StepArgs<real>& a, Slab<real>& s, int t_in_segment) {
    const int src = cur, dst = cur ^ 1;
    a.src = s.lattice[src];
    a.dst = s.lattice[dst];
    a.side_src = s.side[src];
    a.side_dst = s.side[dst];
    a.mask = s.mask;
    a.av = s.av + (size_t)t_in_segment * kAvWords;
    a.ghost_s = win_section(s.win, src, 0);
    a.ghost_n = win_section(s.win, src, 1);
    a.push_up = win_section(s.up_win, dst, 0);
    a.push_dn = win_section(s.dn_win, dst, 1);
    a.flag_from_below = s.sync + kFlagFromBelow;
    a.flag_from_above = s.sync + kFlagFromAbove;
    a.up_flag = s.up_flag;
    a.dn_flag = s.dn_flag;
    a.boundary_done = s.sync + kBoundaryDone;
    a.abort_word = s.sync + kAbort;
    a.up_abort = s.up_abort;
    a.dn_abort = s.dn_abort;
    a.pass = (unsigned long long)passes_done;
    a.timeout_ns = timeout_ns;
    a.plane_stride = plane_stride(s);
    a.nx = prm.nx; a.rows = s.rows; a.pitch = pitch; a.mask_pitch = mask_pitch;
    a.accel_row = s.accel_row;
    a.tiles_x = a.tiles_y = 0;
    a.edge_tiles = 1;
    a.deep = 0;
    a.omega = prm.omega;
    a.aw1 = prm.density * prm.accel / (real)9;       // d2q9-bgk.c:230-231
    a.aw2 = prm.density * prm.accel / (real)36;
  }

  // one pass over every slab: one timestep (K1a/K1b/K1c), two (K7) or three (K10)
  // K1a-f16 (one step) or K7-f16 (two) on the single slab of a LBM_GPU_STORE_F16 lattice
  void launch_pass_f16(int t_in_segment, int steps) {
    if constexpr (sizeof(real) == 4) {
      Slab<real>& s = slabs[0];
      CK(cudaSetDevice(s.device));
      lbm::F16Args a;
      memset(&a, 0, sizeof a);
      a.src = hlat(s, cur);
      a.dst = hlat(s, cur ^ 1);
      a.side_src = s.side[cur];
      a.side_dst = s.side[cur ^ 1];
      a.mask = s.mask;
      a.av = s.av + (size_t)t_in_segment * kAvWords;
      a.av2 = a.av + kAvWords;
      a.plane_stride = plane_stride(s);
      a.nx = prm.nx; a.rows = s.rows; a.pitch = pitch; a.mask_pitch = mask_pitch; a.accel_row = s.accel_row;
      a.omega = prm.omega;
      a.aw1 = prm.density * prm.accel / 9.f;          // d2q9-bgk.c:230-231
      a.aw2 = prm.density * prm.accel / 36.f;
      a.rest = rest();
      const bool strict = (flags & LBM_GPU_STRICT) != 0;
      if (steps == 2) {
        const Tb2Segments sg = tb2_segments(s.rows);
        a.tiles_x = tb2_strips;
        a.tiles_y = sg.n_big + sg.n_tail;
        a.wout = tb2_wout; a.span = tb2_span;
        a.seg_rows = sg.seg_rows; a.n_big = sg.n_big; a.big_rows = sg.big_rows; a.seg_rows_tail = sg.seg_rows_tail;
        const dim3 grid((unsigned)((long long)a.tiles_x * a.tiles_y));
        if (strict) launch_pdl(s, lbm::lbm_step2_tb_f16<true>, a, grid, dim3(tb2_threads), sizeof(lbm::Tb2hSmem));
        else        launch_pdl(s, lbm::lbm_step2_tb_f16<false>, a, grid, dim3(tb2_threads), sizeof(lbm::Tb2hSmem));
      } else {
        int bx, by;
        tile_shape(4, bx, by);
        a.tiles_x = ((prm.nx + 3) / 4 + bx - 1) / bx;
        a.tiles_y = (s.rows + by - 1) / by;
        const dim3 grid((unsigned)((long long)a.tiles_x * a.tiles_y)), block(bx, by);
        if (strict) launch_pdl(s, lbm::lbm_step_vec4_f16<true>, a, grid, block, 0);
        else        launch_pdl(s, lbm::lbm_step_vec4_f16<false>, a, grid, block, 0);
      }
      CK(cudaGetLastError());
      launches++;
    }
    passes_done++;
    cur ^= 1;
  }

  void launch_pass(int t_in_segment, int pass_in_segment, int steps) {
    if (f16) { launch_pass_f16(t_in_segment, steps); return; }
    const bool strict = (flags & LBM_GPU_STRICT) != 0;
    const int nslabs = (int)slabs.size();
    const int vec = (kernel == LBM_GPU_KERNEL_SCALAR) ? 1 : 4;
    int bx, by;
    tile_shape(vec, bx, by);
    const int nxv = (prm.nx + vec - 1) / vec;
    for (int si = 0; si < nslabs; si++) {
      Slab<real>& s = slabs[si];
      CK(cudaSetDevice(s.device));
      if (multi && !use_flags && pass_in_segment > 0) {
        // slabs sharing a GPU: pass p needs the neighbours' pass p-1 (their pushes into this
        // slab's ghost rows, and their reads of the ghost rows this pass overwrites)
        const int up = (si + 1) % nslabs, dn = (si + nslabs - 1) % nslabs;
        CK(cudaStreamWaitEvent(s.stream, slabs[up].step_ev[(pass_in_segment - 1) & 1], 0));
        if (dn != up) CK(cudaStreamWaitEvent(s.stream, slabs[dn].step_ev[(pass_in_segment - 1) & 1], 0));
      }
      lbm::StepArgs<real> a;
      fill_step_args(a, s, t_in_segment);
      if (steps == 3) {
        if constexpr (sizeof(real) == 4) {
          lbm::Tb2Args ta;
          const Tb2Segments sg = tb3_segments(s.rows);
          a.tiles_x = tb2_strips;
          a.tiles_y = sg.n_big;
          ta.s = a;
          ta.ghost_mask = nullptr;
          ta.av2 = a.av + kAvWords;
          ta.av3 = a.av + 2 * kAvWords;
          ta.wout = tb2_wout;
          ta.span = tb2_span;
          ta.seg_rows = sg.seg_rows;
          ta.n_big = sg.n_big;
          ta.big_rows = sg.big_rows;
          ta.seg_rows_tail = sg.seg_rows_tail;
          ta.tile_done = tb3_overlap ? tb3_done : nullptr;
          // a K10 pass is preceded in its run segment by K10 passes only (a shorter last pass comes last)
          ta.wait_tiles = tb3_overlap && pass_in_segment > 0;
          const dim3 grid((unsigned)((long long)tb2_strips * sg.n_big));
          if (strict) launch_tb3<true>(s, ta, grid);
          else        launch_tb3<false>(s, ta, grid);
        }
      } else if (steps == 2) {
        if constexpr (sizeof(real) == 4) {
          lbm::Tb2Args ta;
          const Tb2Segments sg = tb2_segments(s.rows);
          const int nsegs = sg.n_big + sg.n_tail;
          a.tiles_x = tb2_strips;
          a.tiles_y = nsegs;
          a.edge_tiles = 1;
          a.deep = 1;
          ta.s = a;
          ta.ghost_mask = s.ghost_mask;
          ta.av2 = a.av + kAvWords;
          ta.av3 = nullptr;
          ta.wout = tb2_wout;
          ta.span = tb2_span;
          ta.seg_rows = sg.seg_rows;
          ta.n_big = sg.n_big;
          ta.big_rows = sg.big_rows;
          ta.seg_rows_tail = sg.seg_rows_tail;
          const dim3 grid((unsigned)((long long)tb2_strips * nsegs));
          if (strict) { if (use_flags) launch_tb2<true, true>(s, ta, grid); else launch_tb2<true, false>(s, ta, grid); }
          else        { if (use_flags) launch_tb2<false, true>(s, ta, grid); else launch_tb2<false, false>(s, ta, grid); }
        }
      } else {
        a.tiles_x = (nxv + bx - 1) / bx;
        a.tiles_y = (s.rows + by - 1) / by;
        a.deep = max_pass_steps() > 1 ? 1 : 0;     // a lone step between multi-step passes keeps their ghost rows filled
        a.edge_tiles = a.deep ? (2 + by - 1) / by : 1;   // the tile rows that hold the slab's two edge rows   // the tile rows that hold the slab's two edge rows
        const dim3 grid((unsigned)((long long)a.tiles_x * a.tiles_y));
        const dim3 block(bx, by);
        if (strict) { if (use_flags) launch_step<true, true>(s, a, grid, block, cur); else launch_step<true, false>(s, a, grid, block, cur); }
        else        { if (use_flags) launch_step<false, true>(s, a, grid, block, cur); else launch_step<false, false>(s, a, grid, block, cur); }
      }
      CK(cudaGetLastError());
      launches++;
      if (multi && !use_flags) CK(cudaEventRecord(s.step_ev[pass_in_segment & 1], s.stream));
    }
    passes_done++;
    cur ^= 1;
  }

  // room for the per-step sums of n_steps steps (the caller zeroes them)
  void reserve_av(Slab<real>& s, int n_steps) {
    if (s.av_cap >= (size_t)n_steps) return;
    pool_free(s.av, s);
    s.av = nullptr;
    s.av_cap = std::max<size_t>((size_t)n_steps, 1024);
    void* av = nullptr;
    pool_alloc(&av, s.av_cap * (kAvWords + 2) * sizeof(unsigned long long), s);
    s.av = (unsigned long long*)av;
    s.av_compact = s.av + s.av_cap * kAvWords;      // {low, high} per step, filled after the run
  }

  void run_segment(int n_steps, double* sums_out) {
    if (n_steps <= 0) return;
    const bool strict = (flags & LBM_GPU_STRICT) != 0;
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      reserve_av(s, n_steps);
      CK(cudaMemsetAsync(s.av, 0, (size_t)n_steps * kAvWords * sizeof(unsigned long long), s.stream));
    }
    for (auto& s : slabs) { CK(cudaSetDevice(s.device)); CK(cudaEventRecord(s.ev0, s.stream)); }

    if (kernel == LBM_GPU_KERNEL_CLUSTER) {
      launch_cluster(n_steps, strict);
      cur = (cur + n_steps) & 1;
    } else if (kernel == LBM_GPU_KERNEL_PERSISTENT) {
      const int vec = persistent_vec;
      int bx, by;
      tile_shape(vec, bx, by);
      const int nxv = (prm.nx + vec - 1) / vec;
      Slab<real>& s = slabs[0];
      CK(cudaSetDevice(s.device));
      lbm::PersistArgs<real> pa;
      memset(&pa, 0, sizeof pa);
      fill_step_args(pa.s, s, 0);
      lbm::StepArgs<real>& a = pa.s;
      a.tiles_x = (nxv + bx - 1) / bx;
      a.tiles_y = (s.rows + by - 1) / by;
      for (int b = 0; b < 2; b++) { pa.lattice[b] = s.lattice[b]; pa.side[b] = s.side[b]; }
      pa.window = (real*)s.win;
      pa.av = s.av;
      pa.barrier = s.sync + kGridBarrier;
      pa.first_parity = cur;
      pa.n_steps = n_steps;
      pa.n_tiles = a.tiles_x * a.tiles_y;
      const int cap = persistent_capacity(s);
      const int rounds = (pa.n_tiles + cap - 1) / cap;
      const int nblocks = (pa.n_tiles + rounds - 1) / rounds;
      CK(cudaMemsetAsync(pa.barrier, 0, sizeof(unsigned long long), s.stream));
      void* kargs[] = {(void*)&pa};
      CK(cudaLaunchCooperativeKernel(persistent_fn(), dim3(nblocks), dim3(bx, by), kargs, 0, s.stream));
      launches++;
      cur = (cur + n_steps) & 1;
    } else if (kernel == LBM_GPU_KERNEL_PAIRS) {
      const int n_pairs = n_steps / 2;
      if constexpr (sizeof(real) == 4) {
        if (n_pairs > 0) {
          Slab<real>& s = slabs[0];
          CK(cudaSetDevice(s.device));
          lbm::PairsArgs pa;
          memset(&pa, 0, sizeof pa);
          fill_step_args(pa.s, s, 0);
          for (int b = 0; b < 2; b++) { pa.lattice[b] = s.lattice[b]; pa.side[b] = s.side[b]; }
          pa.window = (real*)s.win;
          pa.av = s.av;
          pa.barrier = s.sync + kGridBarrier;
          pa.first_parity = cur;
          pa.n_pairs = n_pairs;
          pa.tile_rows = pairs_tile_rows;
          CK(cudaMemsetAsync(pa.barrier, 0, sizeof(unsigned long long), s.stream));
          void* kargs[] = {(void*)&pa};
          CK(cudaLaunchCooperativeKernel(pairs_fn(), dim3((unsigned)((s.rows + pairs_tile_rows - 1) / pairs_tile_rows)),
                                         pairs_block(), kargs, pairs_smem(), s.stream));
          launches++;
          cur = (cur + n_pairs) & 1;
          passes_done += n_pairs;
        }
      }
      if (n_steps & 1) launch_pass(n_steps - 1, 0, 1);     // the odd last step: K1a
    } else {
      int t = 0, p = 0;
      while (t < n_steps) {
        const int steps = std::min(max_pass_steps(), n_steps - t);
        launch_pass(t, p, steps);
        t += steps;
        p++;
      }
      if (use_flags) {
        // end of the run: wait (on the device, bounded) until both neighbours are as far
        for (auto& s : slabs) {
          CK(cudaSetDevice(s.device));
          lbm::StepArgs<real> a;
          fill_step_args(a, s, 0);
          lbm::lbm_wait_neighbours<real><<<1, 32, 0, s.stream>>>(a);
          CK(cudaGetLastError());
          launches++;
        }
      }
    }
    double ms_max = 0.0;
    for (auto& s : slabs) { CK(cudaSetDevice(s.device)); CK(cudaEventRecord(s.ev1, s.stream)); }
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      CK(cudaStreamSynchronize(s.stream));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, s.ev0, s.ev1));
      ms_max = std::max(ms_max, (double)ms);
    }
    last_run_ms = ms_max;
    last_step_ms = ms_max / n_steps;
    steps_done += n_steps;
    if (use_flags || (kernel == LBM_GPU_KERNEL_TB3 && tb3_overlap)) check_sync_errors();
    if (kernel == LBM_GPU_KERNEL_CLUSTER) prepare();     // side row + ghost rows of the new state
    if (sums_out) read_sums(n_steps, sums_out);
  }

  // The per-step sums of the last n_steps steps (device words -> exact 128-bit totals ->
  // double; NaN for a step that met a non-finite cell).  After the steps have finished.
  void read_sums(int n_steps, double* sums_out) {
    std::vector<unsigned long long> words((size_t)n_steps * 2);
    std::vector<unsigned __int128> tot(n_steps, 0);
    std::vector<char> bad(n_steps, 0);
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      lbm::lbm_compact_av<<<(n_steps + 255) / 256, 256, 0, s.stream>>>(s.av, s.av_compact, n_steps);
      CK(cudaGetLastError());
      launches++;
      CK(cudaMemcpyAsync(words.data(), s.av_compact, words.size() * sizeof(unsigned long long),
                         cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      for (int t = 0; t < n_steps; t++) {
        const unsigned long long lo = words[2 * (size_t)t], hi = words[2 * (size_t)t + 1];
        if (hi & LBM_NONFINITE_MARK) bad[t] = 1;
        tot[t] += ((unsigned __int128)(hi & ~LBM_NONFINITE_MARK) << 32) + lo;
      }
    }
    for (int t = 0; t < n_steps; t++)
      sums_out[t] = bad[t] ? std::nan("") : (double)((long double)tot[t] / (long double)LBM_FIX_SCALE);
  }

  // The flag protocol gave up (see boundary_wait): say why, in the reference's die() spirit.
  void check_sync_errors() {
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      unsigned long long w[2] = {0, 0};
      CK(cudaMemcpyAsync(w, s.sync + kAbort, sizeof w, cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      if (w[0] == 0ULL) continue;
      failed = true;
      const unsigned long long why = w[1] >> 56, pass = w[1] & 0xffffffffffffffULL;
      char msg[256];
      if (why == LBM_SYNC_TILE_TIMEOUT)
        snprintf(msg, sizeof msg, "three-step kernel: a tile of pass %llu did not complete within %.1f s; run abandoned",
                 pass - 1, (double)timeout_ns * 1e-9);
      else if (why == LBM_SYNC_TIMEOUT)
        snprintf(msg, sizeof msg, "rows [%lld,%lld): a neighbouring slab did not complete pass %llu within %.1f s "
                 "(its process died, or it was asked for a different number of steps); run abandoned",
                 s.row0, s.row0 + s.rows, pass, (double)timeout_ns * 1e-9);
      else
        snprintf(msg, sizeof msg, "rows [%lld,%lld): run abandoned because a neighbouring slab gave up%s",
                 s.row0, s.row0 + s.rows, why == LBM_SYNC_ABORTED ? " (abort word set)" : "");
      throw CudaError{msg};
    }
  }

  long long local_free_cells() const {
    long long n = 0;
    for (auto& s : slabs) n += s.free_cells;
    return n;
  }
  long long divisor() const { return global_free_cells >= 0 ? global_free_cells : local_free_cells(); }

  // ---------------------------------------------------------------- outputs ----
  Slab<real>& slab_of_row(long long grow) {
    for (auto& s : slabs)
      if (grow >= s.row0 && grow < s.row0 + s.rows) return s;
    throw CudaError{"row is not held by this process"};
  }

  // Refuse a row range that leaves the rows held here before anything is enqueued, so that a
  // refused call leaves no copy in flight into the caller's buffers or the staging buffer.
  void check_rows(long long row0, long long nrows) {
    long long held = 0;
    for (auto& s : slabs) held += s.rows;
    if (nrows > 0 && (row0 < slabs[0].row0 || row0 + nrows > slabs[0].row0 + held))
      throw CudaError{"row range is not held by this process"};
  }

  void download_rows(long long row0, long long nrows, real* out) {
    const int nx = prm.nx;
    const size_t row_bytes = (size_t)nx * 9 * sizeof(real);
    if (row_bytes > kStagingBytes) throw CudaError{"nx too large for the AoS staging buffer"};
    check_rows(row0, nrows);
    const int chunk_rows = (int)std::max<size_t>(1, kStagingBytes / row_bytes);
    long long g = row0;
    while (g < row0 + nrows) {
      Slab<real>& s = slab_of_row(g);
      CK(cudaSetDevice(s.device));
      const int n = (int)std::min<long long>({(long long)chunk_rows, s.row0 + s.rows - g, row0 + nrows - g});
      const long long ncells = (long long)n * nx;
      if (f16)
        lbm::lbm_soa_to_aos<real, __half><<<(unsigned)((ncells * 9 + 255) / 256), 256, 0, s.stream>>>(
            hlat(s, cur), (real*)s.staging, plane_stride(s), pitch, nx, (int)(g - s.row0), ncells, rest());
      else
        lbm::lbm_soa_to_aos<real><<<(unsigned)((ncells * 9 + 255) / 256), 256, 0, s.stream>>>(
            s.lattice[cur], (real*)s.staging, plane_stride(s), pitch, nx, (int)(g - s.row0), ncells);
      CK(cudaGetLastError());
      launches++;
      CK(cudaMemcpyAsync((char*)out + (size_t)(g - row0) * row_bytes, s.staging, (size_t)n * row_bytes,
                         cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      g += n;
    }
  }

  // lbm_gpu_save_rows / lbm_gpu_load_rows: the stored lattice as cell-major records of 9 stored
  // elements (lbm_pack_rows, lbm_unpack_rows), nothing decoded or rounded
  size_t rec_bytes() const { return f16 ? sizeof(__half) : sizeof(real); }

  template <typename T>
  void launch_rec(bool save, Slab<real>& s, void* st, int r, int n) {
    const long long ncells = (long long)n * prm.nx;
    const dim3 grid((unsigned)((ncells + lbm::kRecCells - 1) / lbm::kRecCells));
    T* planes = reinterpret_cast<T*>(s.lattice[cur]);
    T* rec = static_cast<T*>(st);
    const bool vec = prm.nx % (int)(16 / sizeof(T)) == 0;
    if (save && vec)  lbm::lbm_pack_rows<T, true><<<grid, lbm::kRecThreads, 0, s.stream>>>(planes, rec, plane_stride(s), pitch, prm.nx, r, ncells);
    if (save && !vec) lbm::lbm_pack_rows<T, false><<<grid, lbm::kRecThreads, 0, s.stream>>>(planes, rec, plane_stride(s), pitch, prm.nx, r, ncells);
    if (!save && vec)  lbm::lbm_unpack_rows<T, true><<<grid, lbm::kRecThreads, 0, s.stream>>>(rec, planes, plane_stride(s), pitch, prm.nx, r, ncells);
    if (!save && !vec) lbm::lbm_unpack_rows<T, false><<<grid, lbm::kRecThreads, 0, s.stream>>>(rec, planes, plane_stride(s), pitch, prm.nx, r, ncells);
    CK(cudaGetLastError());
    launches++;
  }

  // Rows [row0, row0+nrows) between the lattice and the host's records, chunk by chunk through
  // the two halves of the staging buffer: the kernel of chunk i+1 overlaps the copy of chunk i on
  // copy_stream, one synchronisation per call.  A range that crosses slabs is cut at their
  // boundaries.  After a load the side row and the ghost rows of the new contents are rebuilt
  // (prepare), except on a slab handle that holds part of the grid: its pushes reach other
  // processes' windows, so there lbm_gpu_ipc_prepare between two host barriers does it.
  void move_rows(bool save, long long row0, long long nrows, void* host) {
    const size_t row_bytes = (size_t)prm.nx * 9 * rec_bytes();
    const size_t half = kStagingBytes / 2;
    if (row_bytes > half) throw CudaError{"nx too large for the record staging buffer"};
    check_rows(row0, nrows);
    if (nrows == 0) return;
    const int chunk_rows = (int)(half / row_bytes);
    std::vector<Slab<real>*> used;
    long long g = row0;
    int i = 0;
    while (g < row0 + nrows) {
      Slab<real>& s = slab_of_row(g);
      CK(cudaSetDevice(s.device));
      if (used.empty() || used.back() != &s) {
        used.push_back(&s);
        i = 0;
        CK(cudaEventRecord(s.stage_drained[0], s.stream));     // the halves are free once earlier work is done
        CK(cudaEventRecord(s.stage_drained[1], s.stream));
      }
      const int n = (int)std::min<long long>({(long long)chunk_rows, s.row0 + s.rows - g, row0 + nrows - g});
      const int b = i & 1;
      char* st = (char*)s.staging + (size_t)b * half;
      char* h = (char*)host + (size_t)(g - row0) * row_bytes;
      const size_t bytes = (size_t)n * row_bytes;
      const int r = (int)(g - s.row0);
      if (save) {
        CK(cudaStreamWaitEvent(s.stream, s.stage_drained[b], 0));
        if (f16) launch_rec<uint16_t>(true, s, st, r, n);
        else if (sizeof(real) == 8) launch_rec<uint64_t>(true, s, st, r, n);
        else launch_rec<uint32_t>(true, s, st, r, n);
        CK(cudaEventRecord(s.stage_filled[b], s.stream));
        CK(cudaStreamWaitEvent(s.copy_stream, s.stage_filled[b], 0));
        CK(cudaMemcpyAsync(h, st, bytes, cudaMemcpyDeviceToHost, s.copy_stream));
        CK(cudaEventRecord(s.stage_drained[b], s.copy_stream));
      } else {
        CK(cudaStreamWaitEvent(s.copy_stream, s.stage_drained[b], 0));
        CK(cudaMemcpyAsync(st, h, bytes, cudaMemcpyHostToDevice, s.copy_stream));
        CK(cudaEventRecord(s.stage_filled[b], s.copy_stream));
        CK(cudaStreamWaitEvent(s.stream, s.stage_filled[b], 0));
        if (f16) launch_rec<uint16_t>(false, s, st, r, n);
        else if (sizeof(real) == 8) launch_rec<uint64_t>(false, s, st, r, n);
        else launch_rec<uint32_t>(false, s, st, r, n);
        CK(cudaEventRecord(s.stage_drained[b], s.stream));
      }
      g += n;
      i++;
    }
    for (Slab<real>* s : used) {
      CK(cudaSetDevice(s->device));
      CK(cudaStreamSynchronize(s->copy_stream));
      CK(cudaStreamSynchronize(s->stream));
    }
    if (save) return;
    if (!slab_mode || slabs[0].rows == prm.ny) prepare();
    else loaded_unprepared = true;
  }

  // Fields of rows [row0, row0+nrows): computed chunk by chunk into one half of the staging
  // buffer (kernel stream) and copied out from the other half (copy stream): the kernel of
  // chunk i+1 overlaps the device-to-host copies of chunk i, one synchronisation per call.
  void final_fields(long long row0, long long nrows, real* ux, real* uy, real* u, real* p) {
    const int nx = prm.nx;
    const size_t row_bytes = (size_t)nx * sizeof(real);
    const size_t half = kStagingBytes / 2;
    if (4 * row_bytes > half) throw CudaError{"nx too large for the fields staging buffer"};
    check_rows(row0, nrows);
    const int chunk_rows = (int)(half / (4 * row_bytes));
    std::vector<Slab<real>*> used;
    long long g = row0;
    int i = 0;
    while (g < row0 + nrows) {
      Slab<real>& s = slab_of_row(g);
      CK(cudaSetDevice(s.device));
      if (used.empty() || used.back() != &s) {
        used.push_back(&s);
        i = 0;
      }
      const int n = (int)std::min<long long>({(long long)chunk_rows, s.row0 + s.rows - g, row0 + nrows - g});
      const long long ncells = (long long)n * nx;
      const int b = i & 1;
      real* st = (real*)((char*)s.staging + (size_t)b * half);
      real* d_ux = ux ? st : nullptr;
      real* d_uy = uy ? st + ncells : nullptr;
      real* d_u = u ? st + 2 * ncells : nullptr;
      real* d_p = p ? st + 3 * ncells : nullptr;
      if (i >= 2) CK(cudaStreamWaitEvent(s.stream, s.stage_drained[b], 0));
      if (f16)
        lbm::lbm_fields<real, __half><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            hlat(s, cur), s.mask, plane_stride(s), pitch, mask_pitch, nx, (int)(g - s.row0), n,
            prm.density, d_ux, d_uy, d_u, d_p, nullptr, rest());
      else
        lbm::lbm_fields<real><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            s.lattice[cur], s.mask, plane_stride(s), pitch, mask_pitch, nx, (int)(g - s.row0), n,
            prm.density, d_ux, d_uy, d_u, d_p, nullptr);
      CK(cudaGetLastError());
      launches++;
      CK(cudaEventRecord(s.stage_filled[b], s.stream));
      CK(cudaStreamWaitEvent(s.copy_stream, s.stage_filled[b], 0));
      const size_t off = (size_t)(g - row0) * nx;
      if (ux) CK(cudaMemcpyAsync(ux + off, d_ux, ncells * sizeof(real), cudaMemcpyDeviceToHost, s.copy_stream));
      if (uy) CK(cudaMemcpyAsync(uy + off, d_uy, ncells * sizeof(real), cudaMemcpyDeviceToHost, s.copy_stream));
      if (u) CK(cudaMemcpyAsync(u + off, d_u, ncells * sizeof(real), cudaMemcpyDeviceToHost, s.copy_stream));
      if (p) CK(cudaMemcpyAsync(p + off, d_p, ncells * sizeof(real), cudaMemcpyDeviceToHost, s.copy_stream));
      CK(cudaEventRecord(s.stage_drained[b], s.copy_stream));
      g += n;
      i++;
    }
    for (Slab<real>* s : used) {
      CK(cudaSetDevice(s->device));
      CK(cudaStreamSynchronize(s->copy_stream));
      CK(cudaStreamSynchronize(s->stream));
    }
  }

  // Block means of the fields (lbm_gpu_coarse_fields; the arithmetic is in lbm_coarse_fields).
  // Coarse rows that lie wholly in one slab go through the staging buffer as final_fields'
  // rows do: chunk by chunk into one half (kernel stream), copied out from the other (copy
  // stream), one synchronisation per call.  A coarse row cut by a boundary between two slabs
  // of this process (at most one per boundary) comes after them: each slab's integer sums are
  // copied back and added here, and the host computes the same means the kernel would.
  template <typename out_t>
  void launch_coarse(Slab<real>& s, int factor, int nc, long long J0, int n, out_t* const (&d)[4],
                     unsigned long long* raw) {
    const int ncx = (prm.nx + factor - 1) / factor;
    const dim3 grid((unsigned)((ncx + nc - 1) / nc), (unsigned)n);
    const unsigned threads = (unsigned)round_up((nc * factor + 3) / 4, 32);
    const size_t smem = factor == 1 ? 0 : (size_t)nc * (4 * sizeof(unsigned long long) + sizeof(unsigned));
    if (f16)
      lbm::lbm_coarse_fields<__half, out_t><<<grid, threads, smem, s.stream>>>(
          hlat(s, cur), s.mask, plane_stride(s), pitch, mask_pitch, prm.nx, prm.ny, s.row0, s.rows, factor, nc, ncx,
          J0, (float)prm.density, rest(), d[0], d[1], d[2], d[3], raw);
    else
      lbm::lbm_coarse_fields<float, out_t><<<grid, threads, smem, s.stream>>>(
          (const float*)s.lattice[cur], s.mask, plane_stride(s), pitch, mask_pitch, prm.nx, prm.ny, s.row0, s.rows,
          factor, nc, ncx, J0, (float)prm.density, rest(), d[0], d[1], d[2], d[3], raw);
    CK(cudaGetLastError());
    launches++;
  }

  void coarse_fields(int factor, bool half_out, long long crow0, long long ncrows, void* const (&out)[4]) {
    const int nx = prm.nx;
    const long long ny = prm.ny;
    const int ncx = (nx + factor - 1) / factor;
    const long long ncy = (ny + factor - 1) / factor;
    if (ncrows == 0) return;
    if (crow0 < 0 || crow0 + ncrows > ncy)
      throw CudaError{"coarse rows [" + std::to_string(crow0) + ", " + std::to_string(crow0 + ncrows) +
                      ") are not all in the grid's " + std::to_string(ncy) + " coarse rows"};
    long long held = 0;
    for (auto& s : slabs) held += s.rows;
    const long long h0 = slabs[0].row0, h1 = h0 + held;
    const long long first = crow0 * factor < h0 ? crow0 : (std::min((crow0 + ncrows) * factor, ny) > h1 ? std::max(crow0, h1 / factor) : -1);
    if (first >= 0) {
      char b[256];
      snprintf(b, sizeof b, "coarse row %lld needs global rows [%lld, %lld), and this process holds rows [%lld, %lld)",
               first, first * factor, std::min(first * factor + factor, ny), h0, h1);
      throw CudaError{b};
    }
    if (factor == 1 && !half_out) {                   // the per-cell fields themselves
      final_fields(crow0, ncrows, (real*)out[0], (real*)out[1], (real*)out[2], (real*)out[3]);
      return;
    }
    const size_t es = half_out ? sizeof(__half) : sizeof(float);
    const size_t half = kStagingBytes / 2;
    const size_t row_bytes = 4 * (size_t)ncx * es;
    if (row_bytes > half || (slabs.size() > 1 && (size_t)ncx * lbm::kCoarseRawWords * 8 > kStagingBytes))
      throw CudaError{"nx too large for the coarse fields staging buffer"};
    // coarse columns per block: nc * factor <= kCoarseSpan and a multiple of 4 (aligned quads)
    int nc = lbm::kCoarseSpan / factor;
    nc -= nc % (4 / std::gcd(factor, 4));
    nc = std::min(nc, ncx);
    const int chunk = (int)std::min<size_t>(half / row_bytes, 65535);
    std::vector<Slab<real>*> used;
    std::vector<long long> cut;
    long long J = crow0;
    int i = 0;
    while (J < crow0 + ncrows) {
      Slab<real>& s = slab_of_row(J * factor);
      const long long s_end = s.row0 + s.rows;
      if (std::min(J * factor + factor, ny) > s_end) { cut.push_back(J++); continue; }
      const long long whole_end = s_end == ny ? ncy : s_end / factor;     // first coarse row not wholly in s
      const int n = (int)std::min<long long>({(long long)chunk, whole_end - J, crow0 + ncrows - J});
      CK(cudaSetDevice(s.device));
      if (used.empty() || used.back() != &s) {
        used.push_back(&s);
        i = 0;
      }
      const int b = i & 1;
      char* st = (char*)s.staging + (size_t)b * half;
      const size_t plane = (size_t)n * ncx * es;
      void* d[4];
      for (int k = 0; k < 4; k++) d[k] = out[k] ? st + k * plane : nullptr;
      if (i >= 2) CK(cudaStreamWaitEvent(s.stream, s.stage_drained[b], 0));
      if (half_out) {
        __half* const dh[4] = {(__half*)d[0], (__half*)d[1], (__half*)d[2], (__half*)d[3]};
        launch_coarse<__half>(s, factor, nc, J, n, dh, nullptr);
      } else {
        float* const df[4] = {(float*)d[0], (float*)d[1], (float*)d[2], (float*)d[3]};
        launch_coarse<float>(s, factor, nc, J, n, df, nullptr);
      }
      CK(cudaEventRecord(s.stage_filled[b], s.stream));
      CK(cudaStreamWaitEvent(s.copy_stream, s.stage_filled[b], 0));
      const size_t off = (size_t)(J - crow0) * ncx * es;
      for (int k = 0; k < 4; k++)
        if (out[k]) CK(cudaMemcpyAsync((char*)out[k] + off, d[k], plane, cudaMemcpyDeviceToHost, s.copy_stream));
      CK(cudaEventRecord(s.stage_drained[b], s.copy_stream));
      J += n;
      i++;
    }
    for (Slab<real>* s : used) {
      CK(cudaSetDevice(s->device));
      CK(cudaStreamSynchronize(s->copy_stream));
      CK(cudaStreamSynchronize(s->stream));
    }
    if (cut.empty()) return;
    const float p0 = (float)prm.density * (1.0f / 3.0f);
    std::vector<unsigned long long> tot(ncx * lbm::kCoarseRawWords), part(tot.size());
    for (const long long Jc : cut) {
      const long long g0 = Jc * factor, g1 = std::min(g0 + factor, ny);
      std::fill(tot.begin(), tot.end(), 0ULL);
      for (auto& s : slabs) {
        if (s.row0 >= g1 || s.row0 + s.rows <= g0) continue;
        CK(cudaSetDevice(s.device));
        float* const none[4] = {nullptr, nullptr, nullptr, nullptr};
        launch_coarse<float>(s, factor, nc, Jc, 1, none, (unsigned long long*)s.staging);
        CK(cudaMemcpyAsync(part.data(), s.staging, part.size() * 8, cudaMemcpyDeviceToHost, s.stream));
        CK(cudaStreamSynchronize(s.stream));
        for (size_t w = 0; w < tot.size(); w++)
          tot[w] = (w % lbm::kCoarseRawWords == 4) ? (tot[w] | part[w]) : tot[w] + part[w];
      }
      for (int C = 0; C < ncx; C++) {
        const unsigned long long* w = &tot[(size_t)C * lbm::kCoarseRawWords];
        const double cells = (double)((g1 - g0) * (long long)std::min(factor, nx - C * factor));
        const size_t o = (size_t)(Jc - crow0) * ncx + C;
        for (int k = 0; k < 4; k++) {
          if (!out[k]) continue;
          const float m = ((w[4] >> k) & 1) ? std::nanf("") : (float)((double)(long long)w[k] * 0x1p-32 / cells);
          if (half_out) ((__half*)out[k])[o] = __float2half_rn(k == 3 ? m - p0 : m);
          else ((float*)out[k])[o] = m;
        }
      }
    }
  }

  double av_velocity_sum() {
    unsigned __int128 tot = 0;
    bool bad = false;
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      unsigned long long* av = s.sync + kAvScratch;       // 128-byte aligned inside the sync block
      CK(cudaMemsetAsync(av, 0, kAvWords * sizeof(unsigned long long), s.stream));
      const long long ncells = (long long)s.rows * prm.nx;
      if (f16)
        lbm::lbm_fields<real, __half><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            hlat(s, cur), s.mask, plane_stride(s), pitch, mask_pitch, prm.nx, 0, s.rows, prm.density,
            nullptr, nullptr, nullptr, nullptr, av, rest());
      else
        lbm::lbm_fields<real><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            s.lattice[cur], s.mask, plane_stride(s), pitch, mask_pitch, prm.nx, 0, s.rows, prm.density,
            nullptr, nullptr, nullptr, nullptr, av);
      CK(cudaGetLastError());
      launches++;
      unsigned long long w[kAvWords];
      CK(cudaMemcpyAsync(w, av, sizeof w, cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      for (int k = 0; k < LBM_AV_SLOTS; k++) {
        const unsigned long long hi = w[LBM_AV_STRIDE * k + 1];
        if (hi & LBM_NONFINITE_MARK) bad = true;
        tot += ((unsigned __int128)(hi & ~LBM_NONFINITE_MARK) << 32) + w[LBM_AV_STRIDE * k];
      }
    }
    if (bad) return std::nan("");                // a NaN or blown-up cell, as in read_sums
    return (double)((long double)tot / (long double)LBM_FIX_SCALE);
  }

  // exact digest of the rows held by this process (see lbm_digest)
  void digest(double* total_density, unsigned long long* checksum) {
    unsigned long long mass = 0, sum = 0;
    bool bad = false;
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      unsigned long long* out = s.sync + kScratch0;         // kScratch0..2: mass, checksum, mark
      CK(cudaMemsetAsync(out, 0, 3 * sizeof(unsigned long long), s.stream));
      const long long ncells = (long long)s.rows * prm.nx;
      if (f16)
        lbm::lbm_digest<real, __half><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            hlat(s, cur), plane_stride(s), pitch, prm.nx, 0, s.rows, s.row0, out, rest());
      else
        lbm::lbm_digest<real><<<(unsigned)((ncells + 255) / 256), 256, 0, s.stream>>>(
            s.lattice[cur], plane_stride(s), pitch, prm.nx, 0, s.rows, s.row0, out);
      CK(cudaGetLastError());
      launches++;
      unsigned long long w[3];
      CK(cudaMemcpyAsync(w, out, sizeof w, cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      mass += w[0];
      sum += w[1];
      bad = bad || w[2] != 0;
    }
    if (total_density) *total_density = bad ? std::nan("") : (double)(long long)mass / 4294967296.0;
    if (checksum) *checksum = sum;
  }

  // Momentum-exchange force on the solid cells of each box (lbm_gpu_obstacle_force; the arithmetic
  // is in lbm_obstacle_force).  boxes: n x {x0, y0, x1, y1}, already checked.  Each slab sums the
  // solid cells of its rows; the slabs' 128-bit integer sums are added here before the one
  // conversion to double, so any split of the rows over this process's slabs gives the same bits.
  void obstacle_force(int n, const int* boxes, double* out) {
    if (failed) throw CudaError{"an earlier run of this lattice was abandoned (a neighbouring slab never arrived); "
                                "its contents are void"};
    if (loaded_unprepared)
      throw CudaError{"rows were loaded into this slab handle with lbm_gpu_load_rows and its ghost rows are stale: "
                      "pass a host barrier over all ranks, lbm_gpu_ipc_prepare, and a second barrier first"};
    if (!connected) throw CudaError{"lattice is not connected to its neighbours yet (its ghost rows are not filled)"};
    const size_t table_bytes = (size_t)lbm::kForceMaxBoxes * sizeof(lbm::ForceBox);
    const size_t out_words = (size_t)n * lbm::kForceOutWords;
    std::vector<unsigned __int128> sum((size_t)2 * n, 0);
    std::vector<char> bad(n, 0);
    std::vector<unsigned long long> w(out_words);
    std::vector<lbm::ForceBox> table(n);
    for (auto& s : slabs) {
      CK(cudaSetDevice(s.device));
      // each box gets the blocks its mask words in this slab need, at most one resident wave
      const long long cap = force_resident_blocks(s);
      int total = 0;
      for (int j = 0; j < n; j++) {
        const int* q = boxes + 4 * j;
        lbm::ForceBox& t = table[j];
        const long long r0 = std::max<long long>(q[1], s.row0), r1 = std::min<long long>(q[3], s.row0 + s.rows);
        t.x0 = q[0];
        t.x1 = q[2];
        t.r0 = (int)(r0 - s.row0);
        t.w0 = q[0] / 32;
        t.nw = q[2] > q[0] ? (q[2] + 31) / 32 - t.w0 : 0;
        t.words = r1 > r0 ? (r1 - r0) * t.nw : 0;
        t.first = total;
        t.blocks = (int)std::min<long long>(cap, (t.words + lbm::kForceThreads - 1) / lbm::kForceThreads);
        total += t.blocks;
      }
      lbm::ForceBox* d_table = (lbm::ForceBox*)s.staging;
      unsigned long long* d_out = (unsigned long long*)((char*)s.staging + table_bytes);
      CK(cudaMemsetAsync(d_out, 0, out_words * sizeof(unsigned long long), s.stream));
      if (total > 0) {
        CK(cudaMemcpyAsync(d_table, table.data(), (size_t)n * sizeof(lbm::ForceBox), cudaMemcpyHostToDevice, s.stream));
        const bool whole = s.rows == prm.ny;
        if (f16) {
          lbm::ForceArgs<__half, float> a;
          a.buf = hlat(s, cur);
          a.side = (const float*)s.side[cur];
          a.ghost_s = a.ghost_n = nullptr;      // a binary16 lattice is one slab that holds the whole grid
          fill_force_args(a, s, whole, d_table, d_out, n);
          lbm::lbm_obstacle_force<__half, float><<<total, lbm::kForceThreads, 0, s.stream>>>(a);
        } else {
          lbm::ForceArgs<real, real> a;
          a.buf = s.lattice[cur];
          a.side = s.side[cur];
          a.ghost_s = whole ? nullptr : win_section(s.win, cur, 0);
          a.ghost_n = whole ? nullptr : win_section(s.win, cur, 1);
          fill_force_args(a, s, whole, d_table, d_out, n);
          lbm::lbm_obstacle_force<real, real><<<total, lbm::kForceThreads, 0, s.stream>>>(a);
        }
        CK(cudaGetLastError());
        launches++;
      }
      CK(cudaMemcpyAsync(w.data(), d_out, out_words * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s.stream));
      CK(cudaStreamSynchronize(s.stream));
      for (int j = 0; j < n; j++) {
        const unsigned long long* o = &w[(size_t)j * lbm::kForceOutWords];
        for (int c = 0; c < 2; c++) sum[2 * j + c] += ((unsigned __int128)o[2 * c + 1] << 64) | o[2 * c];
        bad[j] |= o[4] != 0;
      }
    }
    for (int j = 0; j < n; j++)
      for (int c = 0; c < 2; c++)
        out[2 * j + c] = bad[j] ? std::nan("") : std::ldexp((double)(__int128)sum[2 * j + c], -32);
  }
  // blocks of K14 resident on the slab's GPU at once (its register count decides)
  long long force_resident_blocks(const Slab<real>& s) const {
    int per_sm = 0, sms = 0;
    if (f16) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lbm::lbm_obstacle_force<__half, float>, lbm::kForceThreads, 0));
    else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lbm::lbm_obstacle_force<real, real>, lbm::kForceThreads, 0));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s.device));
    return std::max<long long>(1, (long long)per_sm * sms);
  }
  template <typename A>
  void fill_force_args(A& a, const Slab<real>& s, bool whole, const lbm::ForceBox* d_table, unsigned long long* d_out, int n) {
    a.mask = s.mask;
    a.ghost_mask = s.ghost_mask;
    a.boxes = d_table;
    a.out = d_out;
    a.plane_stride = plane_stride(s);
    a.nx = prm.nx; a.rows = s.rows; a.pitch = pitch; a.mask_pitch = mask_pitch; a.accel_row = s.accel_row;
    a.n_boxes = n;
    a.whole = whole;
    a.rest = rest();
  }
};

// split ny rows over n slabs: remainder spread over the first slabs
void split_rows(long long ny, int n, std::vector<long long>& row0, std::vector<int>& rows) {
  row0.resize(n);
  rows.resize(n);
  const long long base = ny / n, rem = ny % n;
  long long r = 0;
  for (int i = 0; i < n; i++) {
    rows[i] = (int)(base + (i < rem ? 1 : 0));
    row0[i] = r;
    r += rows[i];
  }
}

template <typename real>
int create_impl(const typename ParamT<real>::type* params, const real* cells_aos, const void* obstacles,
                int n_gpus, const int* device_ids, unsigned flags, lbm_gpu** out) {
  if (!params || !out) return fail("lbm_gpu_create: NULL argument");
  *out = nullptr;
  if (params->nx < 1 || params->ny < 2) return fail("lbm_gpu_create: need nx >= 1 and ny >= 2 (got %d x %d)", params->nx, params->ny);
  if (n_gpus < 1) return fail("lbm_gpu_create: n_gpus must be >= 1");
  if (params->ny < n_gpus) return fail("lbm_gpu_create: fewer rows (%d) than GPUs (%d)", params->ny, n_gpus);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return fail("lbm_gpu_create: no CUDA device available (this library has no CPU fallback)");
  }
  std::unique_ptr<Grid<real>> g(new Grid<real>());
  try {
    g->prm = *params;
    g->flags = flags;
    g->f16 = (flags & LBM_GPU_STORE_F16) != 0;
    g->setup_geometry(params->nx);
    std::vector<long long> row0;
    std::vector<int> rows;
    split_rows(params->ny, n_gpus, row0, rows);
    g->slabs.resize(n_gpus);
    for (int i = 0; i < n_gpus; i++) {
      Slab<real>& s = g->slabs[i];
      s.device = device_ids ? device_ids[i] : i;
      if (s.device < 0 || s.device >= ndev) return fail("lbm_gpu_create: device %d not available (%d visible)", s.device, ndev);
      s.row0 = row0[i];
      s.rows = rows[i];
      const long long ar = (long long)params->ny - 2;
      s.accel_row = (ar >= s.row0 && ar < s.row0 + s.rows) ? (int)(ar - s.row0) : LBM_NO_ROW;
    }
    g->select_kernel();
    const size_t cell_row = (size_t)params->nx * 9;
    const size_t obst_row_bytes = (flags & LBM_GPU_OBST_BITS) ? (size_t)((params->nx + 31) / 32) * 4 : (size_t)params->nx * 4;
    for (Slab<real>& s : g->slabs) {
      g->alloc_slab(s);
      if (g->kernel == LBM_GPU_KERNEL_TMA) g->make_tensor_maps(s);
      g->load_slab(s, cells_aos ? cells_aos + (size_t)s.row0 * cell_row : nullptr,
                   obstacles ? (const char*)obstacles + (size_t)s.row0 * obst_row_bytes : nullptr, 0);
    }
    g->connect_local();
    g->prepare();
  } catch (const CudaError& e) {
    return fail("lbm_gpu_create: %s", e.what.c_str());
  } catch (const std::exception& e) {      // e.g. std::bad_alloc: never let it cross the C boundary
    return fail("lbm_gpu_create: %s", e.what());
  }
  *out = reinterpret_cast<lbm_gpu*>(static_cast<GridBase*>(g.release()));
  return 0;
}

template <typename real>
Grid<real>* as_grid(lbm_gpu* h, const char* fn) {
  if (!h) { fail("%s: NULL handle", fn); return nullptr; }
  GridBase* b = reinterpret_cast<GridBase*>(h);
  if (b->is_f64() != (sizeof(real) == 8)) {
    fail("%s: handle was created for %s", fn, b->is_f64() ? "double precision (use the _f64 entry points)" : "single precision");
    return nullptr;
  }
  return static_cast<Grid<real>*>(b);
}

template <typename real, typename F>
int guarded(lbm_gpu* h, const char* fn, F&& body) {
  Grid<real>* g = as_grid<real>(h, fn);
  if (!g) return 1;
  try {
    body(*g);
  } catch (const CudaError& e) {
    return fail("%s: %s", fn, e.what.c_str());
  } catch (const std::exception& e) {
    return fail("%s: %s", fn, e.what());
  }
  return 0;
}

template <typename real>
int run_impl(lbm_gpu* h, int n_steps, real* av_out, double* sums_out, const char* fn) {
  if (n_steps < 0) return fail("%s: negative step count", fn);
  return guarded<real>(h, fn, [&](Grid<real>& g) {
    std::vector<double> sums;
    double* sp = sums_out;
    if (!sp && av_out) { sums.resize(std::max(n_steps, 1)); sp = sums.data(); }
    g.run(n_steps, sp);
    if (av_out) {
      const double div = (double)g.divisor();
      for (int t = 0; t < n_steps; t++) av_out[t] = (real)(sp[t] / div);
    }
  });
}

// ----------------------------------------------------------------- batches (K11) ----
// lbm_gpu_run_batch: many K9 lattices of one shape advanced by one kernel, blockIdx.y = member.
constexpr int kBatchMaxTileRows = 32;
// Cost model of one K11 launch per pair of timesteps, fitted to the tile sweep at 128^2
// (profiles/r04_batch.md): a fixed part (barrier, launch share) plus the larger of
//   latency     loop iterations of a thread row x one dependent L2 round trip, which grows with
//               the warps of a block that meet at its __syncthreads, and
//   throughput  warp-iterations the busiest SM has to issue.
constexpr double kBatchFixedNs = 2100.0, kBatchIterNs = 500.0, kBatchIterPerWarpNs = 70.0, kBatchWarpIterNs = 100.0;

struct BatchShape {
  int tile_rows = 0, thread_rows = 0, blocks_per_member = 0, members_per_launch = 0;
  size_t smem = 0;
};

const void* batch_fn(bool strict) {
  return strict ? (const void*)lbm::lbm_steps_pairs_batch<true> : (const void*)lbm::lbm_steps_pairs_batch<false>;
}

// Tile rows H and thread rows T of K11 for n members of nx x rows.  A launch holds as many
// members as have all their blocks resident at once (cooperative launch); bigger batches take
// several launches.  Every (H, T) whose blocks fit is scored with the cost model above and the
// cheapest wins; ties go to fewer launches, then to taller tiles (fewer halo rows recomputed).
BatchShape batch_shape(int device, int nx, int rows, bool strict, int n) {
  struct Entry { int device, nx, rows, n; bool strict; BatchShape shape; };
  static std::mutex mu;
  static std::vector<Entry> cache;
  std::lock_guard<std::mutex> lock(mu);
  for (const Entry& e : cache)
    if (e.device == device && e.nx == nx && e.rows == rows && e.n == n && e.strict == strict) return e.shape;
  int sms = 0, coop = 0, max_smem = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device));
  CK(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  if (!coop) throw CudaError{"cooperative launch is not available on this device"};
  const void* fn = batch_fn(strict);
  cudaFuncAttributes fa;
  CK(cudaFuncGetAttributes(&fa, fn));
  const int max_dyn = max_smem - (int)fa.sharedSizeBytes;     // the block's table entry is static shared memory
  CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  CK(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  const int bx = (int)round_up(nx / 4, 32), wpr = bx / 32;
  const int h_knob = getenv("LBM_BATCH_TILE_ROWS") ? atoi(getenv("LBM_BATCH_TILE_ROWS")) : 0;     // tuning knobs
  const int t_knob = getenv("LBM_BATCH_THREAD_ROWS") ? atoi(getenv("LBM_BATCH_THREAD_ROWS")) : 0;
  BatchShape best;
  double best_cost = 0.0;
  long long best_launches = 0;
  for (int H = 1; H <= std::min(kBatchMaxTileRows, rows - 2); H++) {
    if (h_knob > 0 && H != h_knob) continue;
    const size_t smem = (size_t)(H + 2) * 9 * nx * sizeof(float);
    if (smem > (size_t)max_dyn) break;
    const int bpm = (rows + H - 1) / H;
    for (int T = 1; T <= H + 2 && bx * T <= LBM_BATCH_MAX_THREADS; T++) {
      if (t_knob > 0 && T != t_knob) continue;
      int per_sm = 0;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, bx * T, smem));
      const long long fit = (long long)per_sm * sms / bpm;
      if (fit < 1) continue;
      const long long launches = (n + fit - 1) / fit;
      const long long members = (n + launches - 1) / launches;
      const long long blocks_on_sm = (members * bpm + sms - 1) / sms;
      const int iters = (H + 2 + T - 1) / T + (H + T - 1) / T;
      const double latency = iters * (kBatchIterNs + kBatchIterPerWarpNs * T * wpr);
      const double issue = (double)(blocks_on_sm * T * wpr * iters) * kBatchWarpIterNs;
      const double cost = (double)launches * (kBatchFixedNs + std::max(latency, issue));
      const bool better = best.tile_rows == 0 || cost < best_cost - 1e-6 ||
                          (cost < best_cost + 1e-6 && (launches < best_launches ||
                                                       (launches == best_launches && H > best.tile_rows)));
      if (better) {
        best.tile_rows = H;
        best.thread_rows = T;
        best.blocks_per_member = bpm;
        best.members_per_launch = (int)members;
        best.smem = smem;
        best_cost = cost;
        best_launches = launches;
      }
    }
  }
  if (best.tile_rows == 0) throw CudaError{"no tile shape of the batch kernel keeps one member's blocks resident"};
  if (getenv("LBM_BATCH_VERBOSE") && getenv("LBM_BATCH_VERBOSE")[0] == '1')     // measurement aid
    fprintf(stderr, "lbm_gpu_run_batch: %d x %d, %d members: tile_rows %d, thread_rows %d, %d members per launch\n",
            nx, rows, n, best.tile_rows, best.thread_rows, best.members_per_launch);
  cache.push_back({device, nx, rows, n, strict, best});
  return best;
}

// One segment (at most kMaxSegmentSteps steps) of every member, in order on the first
// member's stream; the other members' streams are ordered before and after it with events
// (each single-slab member's step_ev[], which only multi-slab handles use otherwise).
// Returns the device time; sums[i] (or NULL) receives member i's raw per-step sums.
double run_batch_segment(const std::vector<Grid<float>*>& gs, const BatchShape& shape, int n_steps,
                         const std::vector<double*>& sums) {
  const int n = (int)gs.size();
  Grid<float>& g0 = *gs[0];
  Slab<float>& s0 = g0.slabs[0];
  CK(cudaSetDevice(s0.device));
  const cudaStream_t st = s0.stream;
  for (Grid<float>* g : gs) g->reserve_av(g->slabs[0], n_steps);
  for (int i = 1; i < n; i++) {
    Slab<float>& s = gs[i]->slabs[0];
    CK(cudaEventRecord(s.step_ev[0], s.stream));
    CK(cudaStreamWaitEvent(st, s.step_ev[0], 0));
  }
  CK(cudaEventRecord(s0.ev0, st));
  for (Grid<float>* g : gs) {
    Slab<float>& s = g->slabs[0];
    CK(cudaMemsetAsync(s.av, 0, (size_t)n_steps * kAvWords * sizeof(unsigned long long), st));
  }
  const int n_pairs = n_steps / 2;
  if (n_pairs > 0) {
    // the member table goes to the first member's staging buffer (idle during runs)
    std::vector<lbm::BatchMember> table(n);
    for (int i = 0; i < n; i++) {
      Grid<float>& g = *gs[i];
      Slab<float>& s = g.slabs[0];
      lbm::StepArgs<float> a;
      g.fill_step_args(a, s, 0);
      lbm::BatchMember& m = table[i];
      for (int b = 0; b < 2; b++) { m.lattice[b] = s.lattice[b]; m.side[b] = s.side[b]; }
      m.window = (float*)s.win;
      m.mask = s.mask;
      m.av = s.av;
      m.barrier = s.sync + kGridBarrier;
      m.first_parity = g.cur;
      m.omega = a.omega;
      m.aw1 = a.aw1;
      m.aw2 = a.aw2;
      CK(cudaMemsetAsync(m.barrier, 0, sizeof(unsigned long long), st));
    }
    lbm::BatchMember* dtable = (lbm::BatchMember*)s0.staging;
    CK(cudaMemcpyAsync(dtable, table.data(), table.size() * sizeof(lbm::BatchMember), cudaMemcpyHostToDevice, st));
    lbm::BatchArgs ba;
    memset(&ba, 0, sizeof ba);
    g0.fill_step_args(ba.s, s0, 0);          // geometry; every pointer and constant is the member's
    ba.n_pairs = n_pairs;
    ba.tile_rows = shape.tile_rows;
    const dim3 block((unsigned)round_up(g0.prm.nx / 4, 32), (unsigned)shape.thread_rows);
    const bool strict = (g0.flags & LBM_GPU_STRICT) != 0;
    for (int first = 0; first < n; first += shape.members_per_launch) {
      const int count = std::min(shape.members_per_launch, n - first);
      ba.members = dtable + first;
      void* kargs[] = {(void*)&ba};
      CK(cudaLaunchCooperativeKernel(batch_fn(strict), dim3((unsigned)shape.blocks_per_member, (unsigned)count), block,
                                     kargs, shape.smem, st));
    }
    for (Grid<float>* g : gs) {
      g->launches++;                          // the launch that held its blocks
      g->cur = (g->cur + n_pairs) & 1;
      g->passes_done += n_pairs;
    }
  }
  if (n_steps & 1) {
    // the odd last step: each member's one-step pass (K1a) on its own stream, as run_segment does
    CK(cudaEventRecord(s0.step_ev[1], st));
    for (int i = 0; i < n; i++) {
      Slab<float>& s = gs[i]->slabs[0];
      if (i > 0) CK(cudaStreamWaitEvent(s.stream, s0.step_ev[1], 0));
      gs[i]->launch_pass(n_steps - 1, 0, 1);
      if (i > 0) {
        CK(cudaEventRecord(s.step_ev[1], s.stream));
        CK(cudaStreamWaitEvent(st, s.step_ev[1], 0));
      }
    }
  }
  CK(cudaEventRecord(s0.ev1, st));
  CK(cudaEventRecord(s0.step_ev[0], st));
  for (int i = 1; i < n; i++) CK(cudaStreamWaitEvent(gs[i]->slabs[0].stream, s0.step_ev[0], 0));
  CK(cudaStreamSynchronize(st));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, s0.ev0, s0.ev1));
  for (int i = 0; i < n; i++) {
    gs[i]->steps_done += n_steps;
    if (sums[i]) gs[i]->read_sums(n_steps, sums[i]);
  }
  return ms;
}

int run_batch_impl(lbm_gpu* const* handles, int n, int n_steps, float* av_out) {
  const char* fn = "lbm_gpu_run_batch";
  if (!handles) return fail("%s: NULL handle array", fn);
  if (n < 1) return fail("%s: need at least one member (n = %d)", fn, n);
  if (n_steps < 0) return fail("%s: negative step count", fn);
  std::vector<Grid<float>*> gs(n);
  for (int i = 0; i < n; i++) {
    if (!handles[i]) return fail("%s: member %d is a NULL handle", fn, i);
    for (int j = 0; j < i; j++)
      if (handles[j] == handles[i]) return fail("%s: members %d and %d are the same handle (duplicate)", fn, j, i);
    GridBase* b = reinterpret_cast<GridBase*>(handles[i]);
    if (b->is_f64()) return fail("%s: member %d is double precision; batches run fp32 lattices only", fn, i);
    Grid<float>& g = *static_cast<Grid<float>*>(b);
    if (g.slab_mode) return fail("%s: member %d is a slab handle (lbm_gpu_create_slab); members must be single-slab lattices", fn, i);
    if (g.slabs.size() != 1)
      return fail("%s: member %d is split into %d slabs; members must be single-slab lattices", fn, i, (int)g.slabs.size());
    if (g.failed) return fail("%s: member %d is failed (an earlier run was abandoned)", fn, i);
    if (g.kernel != LBM_GPU_KERNEL_PAIRS)
      return fail("%s: member %d does not run the pairs kernel (LBM_GPU_KERNEL_PAIRS), the only one batched", fn, i);
    gs[i] = &g;
    const Grid<float>& g0 = *gs[0];
    if (g.slabs[0].device != g0.slabs[0].device)
      return fail("%s: member %d is on device %d and member 0 on device %d; members must share one device", fn, i,
                  g.slabs[0].device, g0.slabs[0].device);
    if (g.prm.nx != g0.prm.nx || g.prm.ny != g0.prm.ny)
      return fail("%s: member %d is %d x %d and member 0 is %d x %d; members must have the same nx and ny", fn, i,
                  g.prm.nx, g.prm.ny, g0.prm.nx, g0.prm.ny);
    if ((g.flags & LBM_GPU_STRICT) != (g0.flags & LBM_GPU_STRICT))
      return fail("%s: member %d and member 0 differ in LBM_GPU_STRICT; members must share it", fn, i);
  }
  try {
    Grid<float>& g0 = *gs[0];
    CK(cudaSetDevice(g0.slabs[0].device));
    const BatchShape shape = batch_shape(g0.slabs[0].device, g0.prm.nx, g0.slabs[0].rows,
                                         (g0.flags & LBM_GPU_STRICT) != 0, n);
    std::vector<double> sums(av_out ? (size_t)n * n_steps : 0);
    std::vector<double*> at(n, nullptr);
    double ms = 0.0;
    for (int done = 0; done < n_steps; done += kMaxSegmentSteps) {
      const int seg = std::min(kMaxSegmentSteps, n_steps - done);
      for (int i = 0; i < n && av_out; i++) at[i] = sums.data() + (size_t)i * n_steps + done;
      ms += run_batch_segment(gs, shape, seg, at);
    }
    if (n_steps > 0)
      for (Grid<float>* g : gs) {
        g->last_run_ms = ms;
        g->last_step_ms = ms / n_steps;
      }
    if (av_out)
      for (int i = 0; i < n; i++) {
        const double div = (double)gs[i]->divisor();
        for (int t = 0; t < n_steps; t++) av_out[(size_t)i * n_steps + t] = (float)(sums[(size_t)i * n_steps + t] / div);
      }
  } catch (const CudaError& e) {
    return fail("%s: %s", fn, e.what.c_str());
  } catch (const std::exception& e) {
    return fail("%s: %s", fn, e.what());
  }
  return 0;
}

}  // namespace

// ======================================================================= C-ABI ====
extern "C" {

int lbm_gpu_abi_version(void) { return 2; }

const char* lbm_gpu_last_error(void) { return g_error.c_str(); }

int lbm_gpu_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return -1; }
  return n;
}

int lbm_gpu_create(const lbm_param* params, const float* cells_aos, const void* obstacles, int n_gpus,
                   const int* device_ids, unsigned flags, lbm_gpu** out) {
  return create_impl<float>(params, cells_aos, obstacles, n_gpus, device_ids, flags, out);
}
int lbm_gpu_create_f64(const lbm_param_f64* params, const double* cells_aos, const void* obstacles, int n_gpus,
                       const int* device_ids, unsigned flags, lbm_gpu** out) {
  return create_impl<double>(params, cells_aos, obstacles, n_gpus, device_ids, flags, out);
}

int lbm_gpu_create_slab(const lbm_param* params, long long row0, long long nrows, int device,
                        const float* cells_aos_rows, const void* obstacles_rows, unsigned flags, lbm_gpu** out) {
  if (!params || !out) return fail("lbm_gpu_create_slab: NULL argument");
  *out = nullptr;
  if (params->nx < 1 || params->ny < 2) return fail("lbm_gpu_create_slab: need nx >= 1 and ny >= 2");
  if (row0 < 0 || nrows < 1 || row0 + nrows > params->ny) return fail("lbm_gpu_create_slab: rows [%lld,%lld) outside the grid", row0, row0 + nrows);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    cudaGetLastError();
    return fail("lbm_gpu_create_slab: no CUDA device available (this library has no CPU fallback)");
  }
  if (device < 0 || device >= ndev) return fail("lbm_gpu_create_slab: device %d not available (%d visible)", device, ndev);
  std::unique_ptr<Grid<float>> g(new Grid<float>());
  try {
    g->prm = *params;
    g->flags = flags;
    g->f16 = (flags & LBM_GPU_STORE_F16) != 0;
    g->slab_mode = true;
    g->setup_geometry(params->nx);
    g->slabs.resize(1);
    Slab<float>& s = g->slabs[0];
    s.device = device;
    s.row0 = row0;
    s.rows = (int)nrows;
    const long long ar = (long long)params->ny - 2;
    s.accel_row = (ar >= row0 && ar < row0 + nrows) ? (int)(ar - row0) : LBM_NO_ROW;
    g->select_kernel();
    g->alloc_slab(s);
    if (g->kernel == LBM_GPU_KERNEL_TMA) g->make_tensor_maps(s);
    g->load_slab(s, cells_aos_rows, obstacles_rows, 0);
    if (nrows == params->ny) { g->connect_local(); g->prepare(); }   // whole grid in one slab
  } catch (const CudaError& e) {
    return fail("lbm_gpu_create_slab: %s", e.what.c_str());
  } catch (const std::exception& e) {
    return fail("lbm_gpu_create_slab: %s", e.what());
  }
  *out = reinterpret_cast<lbm_gpu*>(static_cast<GridBase*>(g.release()));
  return 0;
}

int lbm_gpu_ipc_export(lbm_gpu* h, void* desc) {
  if (!desc) return fail("lbm_gpu_ipc_export: NULL descriptor");
  return guarded<float>(h, "lbm_gpu_ipc_export", [&](Grid<float>& g) {
    if (g.slabs.size() != 1) throw CudaError{"only a one-slab handle can be exported"};
    if (g.f16) throw CudaError{"a LBM_GPU_STORE_F16 lattice cannot be shared between processes"};
    Slab<float>& s = g.slabs[0];
    CK(cudaSetDevice(s.device));
    IpcDesc d;
    memset(&d, 0, sizeof d);
    d.magic = kIpcMagic;
    d.elem_size = 4;
    d.device = s.device;
    d.pid = (int32_t)getpid();
    d.nx = g.prm.nx; d.pitch = g.pitch; d.rows = s.rows;
    d.row0 = s.row0;
    d.win_addr = (unsigned long long)(uintptr_t)s.win;
    d.win_bytes = s.win_bytes;
    d.off_sync = s.off_sync;
    d.off_gmask = s.off_gmask;
    d.steps_done = (unsigned long long)g.steps_done;
    d.passes_done = (unsigned long long)g.passes_done;
    d.local_free_cells = s.free_cells;
    d.cur = g.cur;
    d.tb2_ok = g.k7_fits(s.rows) ? 1 : 0;
    CK(cudaIpcGetMemHandle(&d.handle, s.win));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, s.device));
    memcpy(d.gpu_uuid, prop.uuid.bytes, 16);
    memset(desc, 0, LBM_GPU_IPC_DESC_BYTES);
    memcpy(desc, &d, sizeof d);
  });
}

namespace {
// wire a one-slab handle to the slabs below and above it; `ring_k7`: every slab of the ring
// can run (and therefore will run) the two-step kernel
void ipc_connect_impl(Grid<float>& g, const IpcDesc& dn, const IpcDesc& up, bool ring_k7) {
  if (g.slabs.size() != 1) throw CudaError{"only a one-slab handle can be connected"};
  if (g.f16) throw CudaError{"a LBM_GPU_STORE_F16 lattice cannot be shared between processes"};
  Slab<float>& s = g.slabs[0];
  CK(cudaSetDevice(s.device));
  const long long ny = g.prm.ny;
  for (const IpcDesc* d : {&dn, &up}) {
    if (d->magic != kIpcMagic || d->elem_size != 4) throw CudaError{"bad neighbour descriptor"};
    if (d->nx != g.prm.nx || d->pitch != g.pitch) throw CudaError{"neighbour descriptor is for another grid width"};
    if (d->steps_done != (unsigned long long)g.steps_done || d->passes_done != (unsigned long long)g.passes_done ||
        d->cur != g.cur)
      throw CudaError{"neighbour is at a different timestep"};
  }
  cudaDeviceProp my_prop;
  CK(cudaGetDeviceProperties(&my_prop, s.device));
  for (const IpcDesc* d : {&dn, &up})
    if (memcmp(d->gpu_uuid, my_prop.uuid.bytes, 16) == 0 &&
        !(d->pid == (int32_t)getpid() && d->win_addr == (unsigned long long)(uintptr_t)s.win))
      throw CudaError{"a neighbouring slab runs on the same physical GPU: kernels that wait on one another "
                      "must not share a device (use lbm_gpu_create with n_gpus slabs in one process instead)"};
  if ((dn.row0 + dn.rows) % ny != s.row0 % ny) throw CudaError{"descriptor 'below' does not hold row0-1"};
  if ((s.row0 + s.rows) % ny != up.row0 % ny) throw CudaError{"descriptor 'above' does not hold row0+nrows"};
  auto map = [&](const IpcDesc& d, int slot) -> char* {
    if (d.pid == (int32_t)getpid()) {
      // exported by this very process (tests, or a host that drives several GPUs through
      // slab handles): the address is valid here, no IPC mapping needed
      char* p = (char*)(uintptr_t)d.win_addr;
      if (p == s.win) return p;
      if (d.device == s.device)
        throw CudaError{"two slabs ordered by device-side flags must not share a GPU"};
      int can = 0;
      CK(cudaDeviceCanAccessPeer(&can, s.device, d.device));
      if (!can) throw CudaError{"peer access between the selected GPUs is not available"};
      cudaError_t e = cudaDeviceEnablePeerAccess(d.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
      cudaGetLastError();
      return p;
    }
    // LBM_GPU_POOL: the neighbour parks its window in its cache and exports the same
    // allocation again next time, so the mapping is kept too (cudaIpcCloseMemHandle is
    // as slow as cudaFree: up to 0.4 s measured)
    if (g.use_pool()) {
      std::lock_guard<std::mutex> lock(g_window_mutex);
      for (auto& c : g_ipc_cache)
        if (c.device == s.device && memcmp(&c.handle, &d.handle, sizeof d.handle) == 0) return (char*)c.ptr;
    }
    void* p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, d.handle, cudaIpcMemLazyEnablePeerAccess));
    if (g.use_pool()) {
      std::lock_guard<std::mutex> lock(g_window_mutex);
      g_ipc_cache.push_back({d.handle, s.device, p});
    } else {
      s.ipc_mapped[slot] = p;
    }
    return (char*)p;
  };
  for (const IpcDesc* d : {&dn, &up})
    if (d->win_bytes != s.win_bytes || d->off_sync != s.off_sync || d->off_gmask != s.off_gmask)
      throw CudaError{"neighbour window layout differs"};
  s.dn_win = map(dn, 0);
  s.up_win = (memcmp(&dn.handle, &up.handle, sizeof dn.handle) == 0 && dn.pid == up.pid) ? s.dn_win : map(up, 1);
  unsigned long long* dn_sync = (unsigned long long*)(s.dn_win + dn.off_sync);
  unsigned long long* up_sync = (unsigned long long*)(s.up_win + up.off_sync);
  s.dn_flag = dn_sync + kFlagFromAbove;
  s.up_flag = up_sync + kFlagFromBelow;
  s.dn_abort = dn_sync + kAbort;
  s.up_abort = up_sync + kAbort;
  s.dn_gmask = (uint32_t*)(s.dn_win + dn.off_gmask) + g.mask_pitch;
  s.up_gmask = (uint32_t*)(s.up_win + up.off_gmask);
  g.multi = true;
  g.use_flags = true;      // neighbours are other processes: device-side flags
  g.select_kernel(true, ring_k7);
  g.connected = true;
}
}  // namespace

int lbm_gpu_ipc_connect(lbm_gpu* h, const void* desc_below, const void* desc_above) {
  if (!desc_below || !desc_above) return fail("lbm_gpu_ipc_connect: NULL descriptor");
  return guarded<float>(h, "lbm_gpu_ipc_connect", [&](Grid<float>& g) {
    IpcDesc dn, up;
    memcpy(&dn, desc_below, sizeof dn);
    memcpy(&up, desc_above, sizeof up);
    ipc_connect_impl(g, dn, up, false);
  });
}

int lbm_gpu_ipc_connect_all(lbm_gpu* h, const void* descs, int n) {
  if (!descs || n < 1) return fail("lbm_gpu_ipc_connect_all: bad argument");
  return guarded<float>(h, "lbm_gpu_ipc_connect_all", [&](Grid<float>& g) {
    if (g.slabs.size() != 1) throw CudaError{"only a one-slab handle can be connected"};
    Slab<float>& s = g.slabs[0];
    std::vector<IpcDesc> all(n);
    for (int i = 0; i < n; i++) memcpy(&all[i], (const char*)descs + (size_t)i * LBM_GPU_IPC_DESC_BYTES, sizeof(IpcDesc));
    const long long ny = g.prm.ny;
    long long rows_total = 0, free_total = 0;
    int below = -1, above = -1;
    bool all_k7 = true;
    for (int i = 0; i < n; i++) {
      const IpcDesc& d = all[i];
      if (d.magic != kIpcMagic) throw CudaError{"bad descriptor in the list"};
      rows_total += d.rows;
      free_total += d.local_free_cells;
      all_k7 = all_k7 && d.tb2_ok;
      if ((d.row0 + d.rows) % ny == s.row0 % ny) below = i;
      if ((s.row0 + s.rows) % ny == d.row0 % ny) above = i;
    }
    if (rows_total != ny) throw CudaError{"the descriptors do not cover the grid's rows exactly once"};
    if (below < 0 || above < 0) throw CudaError{"no descriptor holds the rows next to this slab"};
    ipc_connect_impl(g, all[below], all[above], all_k7);
    g.global_free_cells = free_total;
  });
}

int lbm_gpu_ipc_prepare(lbm_gpu* h) {
  return guarded<float>(h, "lbm_gpu_ipc_prepare", [&](Grid<float>& g) { g.prepare(); });
}

int lbm_gpu_run(lbm_gpu* h, int n_steps, float* av_vels_out) {
  return run_impl<float>(h, n_steps, av_vels_out, nullptr, "lbm_gpu_run");
}
int lbm_gpu_run_f64(lbm_gpu* h, int n_steps, double* av_vels_out) {
  return run_impl<double>(h, n_steps, av_vels_out, nullptr, "lbm_gpu_run_f64");
}
int lbm_gpu_run_batch(lbm_gpu* const* handles, int n, int n_steps, float* av_vels_out) {
  return run_batch_impl(handles, n, n_steps, av_vels_out);
}
int lbm_gpu_run_sums(lbm_gpu* h, int n_steps, double* sums_out) {
  if (!h) return fail("lbm_gpu_run_sums: NULL handle");
  if (reinterpret_cast<GridBase*>(h)->is_f64()) return run_impl<double>(h, n_steps, nullptr, sums_out, "lbm_gpu_run_sums");
  return run_impl<float>(h, n_steps, nullptr, sums_out, "lbm_gpu_run_sums");
}

int lbm_gpu_set_global_free_cells(lbm_gpu* h, long long free_cells) {
  if (!h) return fail("lbm_gpu_set_global_free_cells: NULL handle");
  if (free_cells < 1) return fail("lbm_gpu_set_global_free_cells: count must be positive");
  GridBase* b = reinterpret_cast<GridBase*>(h);
  if (b->is_f64()) static_cast<Grid<double>*>(b)->global_free_cells = free_cells;
  else static_cast<Grid<float>*>(b)->global_free_cells = free_cells;
  return 0;
}

int lbm_gpu_download(lbm_gpu* h, float* out) {
  if (!out) return fail("lbm_gpu_download: NULL output");
  return guarded<float>(h, "lbm_gpu_download", [&](Grid<float>& g) {
    long long rows = 0;
    for (auto& s : g.slabs) rows += s.rows;
    g.download_rows(g.slabs[0].row0, rows, out);
  });
}
int lbm_gpu_download_f64(lbm_gpu* h, double* out) {
  if (!out) return fail("lbm_gpu_download_f64: NULL output");
  return guarded<double>(h, "lbm_gpu_download_f64", [&](Grid<double>& g) {
    long long rows = 0;
    for (auto& s : g.slabs) rows += s.rows;
    g.download_rows(g.slabs[0].row0, rows, out);
  });
}
int lbm_gpu_download_rows(lbm_gpu* h, long long row0, long long nrows, float* out) {
  if (!out || nrows < 0) return fail("lbm_gpu_download_rows: bad argument");
  return guarded<float>(h, "lbm_gpu_download_rows", [&](Grid<float>& g) { g.download_rows(row0, nrows, out); });
}

int lbm_gpu_final_fields(lbm_gpu* h, long long row0, long long nrows, float* ux, float* uy, float* u, float* p) {
  if (nrows < 0) return fail("lbm_gpu_final_fields: bad argument");
  return guarded<float>(h, "lbm_gpu_final_fields", [&](Grid<float>& g) { g.final_fields(row0, nrows, ux, uy, u, p); });
}
int lbm_gpu_final_fields_f64(lbm_gpu* h, long long row0, long long nrows, double* ux, double* uy, double* u, double* p) {
  if (nrows < 0) return fail("lbm_gpu_final_fields_f64: bad argument");
  return guarded<double>(h, "lbm_gpu_final_fields_f64", [&](Grid<double>& g) { g.final_fields(row0, nrows, ux, uy, u, p); });
}

int lbm_gpu_coarse_fields(lbm_gpu* h, int factor, unsigned format, long long crow0, long long ncrows,
                          void* ux, void* uy, void* u, void* p) {
  if (factor < 1 || factor > 256) return fail("lbm_gpu_coarse_fields: factor %d is not in 1..256", factor);
  if (format != LBM_GPU_FIELDS_F32 && format != LBM_GPU_FIELDS_F16)
    return fail("lbm_gpu_coarse_fields: unknown format %u", format);
  if (ncrows < 0) return fail("lbm_gpu_coarse_fields: negative ncrows");
  if (h && reinterpret_cast<GridBase*>(h)->is_f64())
    return fail("lbm_gpu_coarse_fields: double-precision handles are not served (use lbm_gpu_final_fields_f64)");
  return guarded<float>(h, "lbm_gpu_coarse_fields", [&](Grid<float>& g) {
    void* const out[4] = {ux, uy, u, p};
    g.coarse_fields(factor, format == LBM_GPU_FIELDS_F16, crow0, ncrows, out);
  });
}

int lbm_gpu_av_velocity(lbm_gpu* h, float* av_out) {
  if (!av_out) return fail("lbm_gpu_av_velocity: NULL output");
  return guarded<float>(h, "lbm_gpu_av_velocity", [&](Grid<float>& g) {
    *av_out = (float)(g.av_velocity_sum() / (double)g.divisor());
  });
}
int lbm_gpu_av_velocity_f64(lbm_gpu* h, double* av_out) {
  if (!av_out) return fail("lbm_gpu_av_velocity_f64: NULL output");
  return guarded<double>(h, "lbm_gpu_av_velocity_f64", [&](Grid<double>& g) {
    *av_out = g.av_velocity_sum() / (double)g.divisor();
  });
}

int lbm_gpu_digest(lbm_gpu* h, double* total_density, unsigned long long* checksum) {
  if (!h) return fail("lbm_gpu_digest: NULL handle");
  if (reinterpret_cast<GridBase*>(h)->is_f64())
    return guarded<double>(h, "lbm_gpu_digest", [&](Grid<double>& g) { g.digest(total_density, checksum); });
  return guarded<float>(h, "lbm_gpu_digest", [&](Grid<float>& g) { g.digest(total_density, checksum); });
}

int lbm_gpu_obstacle_force(lbm_gpu* h, int n_boxes, const int* boxes, double* force_out) {
  const char* fn = "lbm_gpu_obstacle_force";
  if (!h) return fail("%s: NULL handle", fn);
  if (n_boxes < 1 || n_boxes > lbm::kForceMaxBoxes)
    return fail("%s: n_boxes %d is not in 1..%d", fn, n_boxes, lbm::kForceMaxBoxes);
  if (!force_out) return fail("%s: NULL force_out", fn);
  if (!boxes && n_boxes != 1) return fail("%s: boxes is NULL with n_boxes %d (NULL means one box, the whole grid)", fn, n_boxes);
  auto body = [&](auto& g) {
    const int nx = g.prm.nx, ny = g.prm.ny;
    const int whole[4] = {0, 0, nx, ny};
    const int* b = boxes ? boxes : whole;
    for (int j = 0; j < n_boxes; j++) {
      const int* q = b + 4 * j;
      if (!(0 <= q[0] && q[0] <= q[2] && q[2] <= nx && 0 <= q[1] && q[1] <= q[3] && q[3] <= ny)) {
        char m[256];
        snprintf(m, sizeof m, "box %d {x0 %d, y0 %d, x1 %d, y1 %d} is not within 0 <= x0 <= x1 <= nx = %d and "
                 "0 <= y0 <= y1 <= ny = %d", j, q[0], q[1], q[2], q[3], nx, ny);
        throw CudaError{m};
      }
    }
    g.obstacle_force(n_boxes, b, force_out);
  };
  if (reinterpret_cast<GridBase*>(h)->is_f64()) return guarded<double>(h, fn, body);
  return guarded<float>(h, fn, body);
}

namespace {
// lbm_gpu_save_rows / lbm_gpu_load_rows for either precision; refused before anything is enqueued
int move_rows_impl(lbm_gpu* h, bool save, long long row0, long long nrows, void* p) {
  const char* fn = save ? "lbm_gpu_save_rows" : "lbm_gpu_load_rows";
  if (!h) return fail("%s: NULL handle", fn);
  if (nrows < 0) return fail("%s: negative nrows (%lld)", fn, nrows);
  if (!p && nrows > 0) return fail("%s: NULL %s for %lld rows", fn, save ? "output" : "input", nrows);
  auto body = [&](auto& g) {
    if (g.failed) throw CudaError{"an earlier run of this lattice was abandoned (a neighbouring slab never arrived); "
                                  "its contents are void"};
    g.move_rows(save, row0, nrows, p);
  };
  if (reinterpret_cast<GridBase*>(h)->is_f64()) return guarded<double>(h, fn, body);
  return guarded<float>(h, fn, body);
}
}  // namespace

int lbm_gpu_save_rows(lbm_gpu* h, long long row0, long long nrows, void* out) {
  return move_rows_impl(h, true, row0, nrows, out);
}
int lbm_gpu_load_rows(lbm_gpu* h, long long row0, long long nrows, const void* in) {
  return move_rows_impl(h, false, row0, nrows, const_cast<void*>(in));
}

int lbm_gpu_upload(lbm_gpu* h, const float* cells_aos) {
  if (!cells_aos) return fail("lbm_gpu_upload: NULL input");
  return guarded<float>(h, "lbm_gpu_upload", [&](Grid<float>& g) {
    const int cur = g.cur;
    const long long base = g.slabs[0].row0;
    for (auto& s : g.slabs) g.upload_cells(s, cells_aos + (size_t)(s.row0 - base) * g.prm.nx * 9, cur);
    if (!g.slab_mode || g.slabs[0].rows == g.prm.ny) g.prepare();
  });
}
int lbm_gpu_upload_f64(lbm_gpu* h, const double* cells_aos) {
  if (!cells_aos) return fail("lbm_gpu_upload_f64: NULL input");
  return guarded<double>(h, "lbm_gpu_upload_f64", [&](Grid<double>& g) {
    const int cur = g.cur;
    for (auto& s : g.slabs) g.upload_cells(s, cells_aos + (size_t)s.row0 * g.prm.nx * 9, cur);
    g.prepare();
  });
}

int lbm_gpu_get_info(lbm_gpu* h, lbm_gpu_info* info) {
  if (!h || !info) return fail("lbm_gpu_get_info: NULL argument");
  memset(info, 0, sizeof *info);
  GridBase* b = reinterpret_cast<GridBase*>(h);
  auto fill = [&](auto& g) {
    info->nx = g.prm.nx; info->ny = g.prm.ny;
    info->n_gpus = (int)g.slabs.size();
    info->is_f64 = g.is_f64();
    info->kernel = g.kernel;
    info->pitch = g.pitch;
    info->local_free_cells = g.local_free_cells();
    info->free_cells = g.divisor();
    info->local_row0 = g.slabs[0].row0;
    long long rows = 0;
    size_t bytes = 0;
    for (auto& s : g.slabs) { rows += s.rows; bytes = std::max(bytes, s.bytes + kStagingBytes); }
    info->local_rows = rows;
    info->steps_done = g.steps_done;
    info->kernel_launches = g.launches;
    info->last_run_device_ms = g.last_run_ms;
    info->last_step_kernel_ms = g.last_step_ms;
    info->device_bytes = bytes;
  };
  if (b->is_f64()) fill(*static_cast<Grid<double>*>(b));
  else fill(*static_cast<Grid<float>*>(b));
  return 0;
}

int lbm_gpu_host_alloc(size_t bytes, void** out) {
  if (!out) return fail("lbm_gpu_host_alloc: NULL argument");
  *out = nullptr;
  cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail("lbm_gpu_host_alloc: %s", cudaGetErrorString(e));
  }
  return 0;
}

void lbm_gpu_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

void lbm_gpu_destroy(lbm_gpu* h) {
  if (!h) return;
  delete reinterpret_cast<GridBase*>(h);
}

#ifdef LBM_EXPERIMENTS
// -DLBM_EXPERIMENTS builds only: K10's staging-wait and tile cycles on the current device since
// the last call (lbm::tb3_exp_cycles), then cleared
int lbm_gpu_exp_tb3_cycles(unsigned long long out[2]) {
  static const unsigned long long zero[2] = {0ULL, 0ULL};
  if (cudaDeviceSynchronize() != cudaSuccess ||
      cudaMemcpyFromSymbol(out, lbm::tb3_exp_cycles, sizeof zero) != cudaSuccess ||
      cudaMemcpyToSymbol(lbm::tb3_exp_cycles, zero, sizeof zero) != cudaSuccess)
    return fail("lbm_gpu_exp_tb3_cycles: %s", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
// ... and K10's block times since the last call (lbm::tb3_exp_blocks: earliest start, latest
// end, sum of block durations, in ns), then cleared; out[3] = resident K10 blocks of the device
int lbm_gpu_exp_tb3_blocks(unsigned long long out[4]) {
  static const unsigned long long clear[3] = {~0ULL, 0ULL, 0ULL};
  int dev = 0, sms = 0;
  if (cudaDeviceSynchronize() != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      cudaMemcpyFromSymbol(out, lbm::tb3_exp_blocks, sizeof clear) != cudaSuccess ||
      cudaMemcpyToSymbol(lbm::tb3_exp_blocks, clear, sizeof clear) != cudaSuccess)
    return fail("lbm_gpu_exp_tb3_blocks: %s", cudaGetErrorString(cudaGetLastError()));
  out[3] = (unsigned long long)LBM_TB3_MIN_BLOCKS * sms;
  return 0;
}
#endif

}  // extern "C"
