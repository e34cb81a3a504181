// helicon_b200: C-ABI host side (include/helicon_b200.h).  One translation unit.
#include "../../include/helicon_b200.h"
#include "hb2_kernels.cuh"
#include "hb2_trf.cuh"
#include "hb2_symm.cuh"
#include "hb2_tie.cuh"
#include "hb2_fwd_band.cuh"
#include "hb2_adj_tile.cuh"
#include "hb2_explicit.cuh"
#include "hb2_bilinear.cuh"

#include <cub/cub.cuh>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>

// NVTX ranges named after the reference's helicon.Timer stages (lib/logging.py:169-220; SLR:100, 131, 360 and
// pipeline.py:405), so that a timeline of the CUDA path reads like the reference's own timing log.  Header-only NVTX3: a
// no-op unless a profiler is attached.
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CK(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) {                                                                              \
      char buf_[512];                                                                                     \
      snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return fail(HB2_ERR_CUDA, buf_);                                                                    \
    }                                                                                                     \
  } while (0)
#define CKL()                                                                                             \
  do {                                                                                                    \
    cudaError_t e_ = cudaGetLastError();                                                                  \
    if (e_ != cudaSuccess) {                                                                              \
      char buf_[512];                                                                                     \
      snprintf(buf_, sizeof buf_, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
      return fail(HB2_ERR_CUDA, buf_);                                                                    \
    }                                                                                                     \
  } while (0)

static inline unsigned cdiv(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

// Opt-in dynamic shared memory limit of the current device.  Every kernel that needs more than 48 KB gets its
// cudaFuncAttributeMaxDynamicSharedMemorySize set to THIS constant (not to the size of the launch at hand): the
// attribute is per function and process-wide, so two host threads setting their own sizes would race -- the thread
// with the larger request could launch after the other thread lowered the limit ("too many resources requested").
static int hb2_max_smem() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) { cudaGetLastError(); v = 48 << 10; }
    cached = v; cached_dev = dev;
  }
  return cached;
}
// Raise the kernel's dynamic shared memory limit to everything the device allows next to the kernel's own static
// shared memory -- once per (device, kernel); the value never changes afterwards, so concurrent callers cannot race.
#include <set>
static void hb2_allow_big_smem(const void* func) {
  static std::mutex mu;
  static std::set<std::pair<int, const void*>> done;
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({dev, func})) return;
  cudaFuncAttributes fa{};
  if (cudaFuncGetAttributes(&fa, func) != cudaSuccess) { cudaGetLastError(); return; }
  const int lim = hb2_max_smem() - (int)fa.sharedSizeBytes;
  if (cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, lim) != cudaSuccess) cudaGetLastError();
  done.insert({dev, func});
}

// ---------------------------------------------------------------------------
struct hb2_problem {
  int device = 0;
  hb2_geometry g{};
  int ndisk = 0;
  float* d_pix = nullptr;          // [D2][L2]  pix[j][k] = image[j - D2//2 + ny//2, k - L2//2 + nx//2]
  int* d_rank_data = nullptr;      // [D2*D2]
  int* d_rank_sym = nullptr;       // [D3*D3]
  int* d_int2ref = nullptr;        // [ndisk] internal disk rank -> reference rank
  short2* d_yx_data = nullptr;     // [ndisk] (row y, column x) on the data grid
  short2* d_yx_sym = nullptr;      // [ndisk] on the symmetry grid, REFERENCE voxel order (row enumeration of the symmetry rows)
  std::vector<int> h_rank_data;    // reference disk rank (C-order np.nonzero) on the data grid, for exports
  std::vector<int> int2ref, ref2int;  // internal (tile-major) disk rank <-> reference rank
  std::vector<int> h_tile_begin;      // [ntile+1] first internal rank of every non-empty voxel tile
  std::vector<int> h_tilerow_begin;   // [ntilerow+1] first internal rank of every row of tiles
  int ntile = 0;
  bool tile_ok = false;               // tiles hold <= 256 voxels (k_adj_tile)
  int* d_tile_begin = nullptr;
  int* d_aslot = nullptr;             // [ndisk] tile*256 + rank inside the tile
};

// Device memory of a batch: one ARENA per (device, stream), bump-allocated.  A grid search alternates two streams
// (grid.BatchPipeline), so in steady state every batch lands in the block its stream's previous batch used and no
// allocator call happens at all -- cudaMalloc/cudaFree synchronise the device, and growing the stream-ordered pool
// (cudaMallocAsync) was measured to stall a concurrently running solve by up to 2 s (profiles/r1_summary.md section 4).
// An arena has ONE owner at a time (the batch whose pool allocated first while the arena was idle; the temporaries
// of that batch's setup / bounded branch carry the same owner token and nest like a stack).  Pools of any other
// owner that is alive at the same time -- e.g. lsq_reconstruct called from several threads of a ThreadPoolExecutor
// on the default stream (app.py:2473) -- never touch the arena: they are served by cudaMalloc, so two live batches
// can not be handed the same range and interleaved allocations can not break the stack rule.  All arena state is
// guarded by g_arena_mu.  What does not fit the arena yet is served by cudaMalloc and remembered, and the arena is
// re-sized the next time it is idle.
#include <map>
#include <mutex>
struct Arena {
  char* base = nullptr;
  size_t cap = 0, top = 0, wanted = 0, high = 0;
  int live = 0;                  // pools (of the owner) with allocations in this arena
  const void* owner = nullptr;   // owner token while live > 0
};
static std::mutex g_arena_mu;
static std::map<std::pair<int, cudaStream_t>, Arena*> g_arenas;
static Arena* arena_for_locked(cudaStream_t st) {
  int dev = 0;
  cudaGetDevice(&dev);
  Arena*& a = g_arenas[{dev, st}];
  if (!a) a = new Arena();
  return a;
}

struct DevPool {
  std::vector<void*> owned;  // overflow allocations (cudaMalloc)
  size_t bytes = 0, overflow = 0;
  cudaStream_t stream = nullptr;
  Arena* arena = nullptr;
  const void* owner = nullptr;  // owner token (the batch); null: the pool itself
  size_t first = 0, last = 0;   // arena range of this pool
  bool in_arena = false;
  template <typename T>
  cudaError_t alloc(T** p, size_t count, bool zero, cudaStream_t st) {
    const size_t nb = (std::max<size_t>(count, 1) * sizeof(T) + 255) / 256 * 256;
    stream = st;
    const void* me = owner ? owner : (const void*)this;
    cudaError_t e = cudaSuccess;
    {
      std::lock_guard<std::mutex> lk(g_arena_mu);
      if (!arena) arena = arena_for_locked(st);
      Arena& A = *arena;
      if (A.live == 0) {  // arena idle: re-size it if earlier batches did not fit, then claim it
        A.top = 0; A.owner = nullptr;
        if (A.cap == 0 && A.wanted == 0) {  // first use of this stream: start with a fifth of the free memory (<= 24 GB)
          size_t fr = 0, tot = 0;
          if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) A.wanted = std::min<size_t>(fr / 5, (size_t)24 << 30) / 9 * 8;
        }
        if (A.wanted > A.cap) {
          if (A.base) { cudaStreamSynchronize(st); cudaFree(A.base); A.base = nullptr; A.cap = 0; }
          const size_t want = A.wanted + A.wanted / 8;
          if (cudaMalloc((void**)&A.base, want) == cudaSuccess) A.cap = want;
          else cudaGetLastError();
        }
      }
      const bool mine = A.live == 0 || A.owner == me;
      if (mine && A.top + nb <= A.cap) {
        if (!in_arena) { in_arena = true; first = A.top; A.live += 1; A.owner = me; }
        *p = reinterpret_cast<T*>(A.base + A.top);
        A.top += nb; last = A.top;
        A.high = std::max(A.high, A.top);
      } else {
        e = cudaMalloc((void**)p, nb);
        if (e != cudaSuccess) return e;
        owned.push_back(*p);
        overflow += nb;
        if (mine) A.wanted = std::max(A.wanted, std::max(A.high, A.top) + overflow + nb);
      }
    }
    bytes += nb;
    if (zero) e = cudaMemsetAsync(*p, 0, nb, st);
    return e;
  }
  void release(void* p) {  // individual frees only matter for overflow blocks
    for (auto& q : owned)
      if (q == p) { cudaStreamSynchronize(stream); cudaFree(q); q = nullptr; }
  }
  void free_all() {
    if (!owned.empty()) {
      cudaStreamSynchronize(stream);
      for (void* p : owned)
        if (p) cudaFree(p);
      owned.clear();
    }
    if (in_arena) {
      std::lock_guard<std::mutex> lk(g_arena_mu);
      Arena& A = *arena;
      if (A.top == last) A.top = first;  // stack discipline inside one owner: give the range back
      A.live -= 1;
      if (A.live == 0) { A.top = 0; A.owner = nullptr; }
      in_arena = false;
    }
    bytes = 0; overflow = 0;
  }
};

struct hb2_batch {
  hb2_problem* P = nullptr;
  cudaStream_t stream = nullptr;
  DevPool pool;
  BD B{};
  bool idx16 = true;
  size_t adj_tile_smem = 0;
  int adj_chunks = 1;  // adj_tile == 2: chunks of 16 slices
  bool want_tie_info = false;
  size_t fwd_band_smem = 0, fwd_band_smem64 = 0;
  // tie views (hb2_batch_set_ties)
  int n_tie = 0, tie_TS = 0;
  std::vector<int8_t> h_tie_zlo;
  std::vector<uint8_t> h_tie_up, h_tie_rv;
  int n_tie_views = 0;
  // explicit data rows (hb2_batch_explicit_rows)
  bool explicit_rows = false;
  long long exp_nnz = 0;
  float* d_exp_b = nullptr;
  int* d_exp_pid = nullptr;
  float exp_bmax = 0.f;
  int exp_md = 0;                 // explicit data rows
  int *d_exp_ptr = nullptr, *d_exp_col = nullptr, *d_exp_erow = nullptr;
  float* d_exp_w = nullptr;
  bool exp_finished = false;
  std::vector<uint8_t> h_exp_pixmask;  // half-set mask over pixel ids k*D2 + j (empty: all rows kept)
  // trilinear symmetry rows (hb2_batch_explicit_sym_rows): 16 entries per row
  int ls_m = 0;
  int* d_ls_col = nullptr;
  float* d_ls_w = nullptr;
  uint16_t* d_amap_i = nullptr;
  // matrix-free trilinear rows (hb2_batch_bilinear_*)
  bool bilinear = false;
  int bil_nM = 0;
  std::vector<uint8_t> h_bil_rv;                 // [nM][D2]
  std::vector<int> h_bil_view_map, h_bil_colk, h_bil_cand_nview;
  std::vector<double> h_bil_ab;
  std::vector<int2*> ls_ent_c;                   // per candidate: trilinear symmetry rows, 16 entries each
  std::vector<int> ls_m_c;
  struct LsScratch {
    long long cap_rows = 0, sort_cap = 0;
    int pairs_cap = 0;
    LsymPair* pairs = nullptr;
    unsigned long long *tab_key = nullptr, *tab_seq = nullptr;
    int *tmp_a = nullptr, *tmp_b = nullptr, *flag = nullptr, *pos = nullptr, *ov = nullptr;
    void* scan_tmp = nullptr; size_t scan_bytes = 0;
    int *col = nullptr; float* w = nullptr;      // unpacked rows of the candidate being built
    int *key = nullptr, *key2 = nullptr, *id = nullptr, *id2 = nullptr, *cc = nullptr;
    void* sort_tmp = nullptr; size_t sort_bytes = 0;
  } ls_scr;
  long long extra_launches = 0;  // kernels beyond one per launch_* call (band path: projector + reduce)
  int max_views = 0;
  bool created = false;
  int nviews = 0;
  // host copies
  std::vector<hb2_candidate> cands;
  std::vector<int> h_view_count, h_view_begin, h_mdata, h_msym;
  std::vector<long long> h_uoff, h_symoff, h_symcap, h_cscoff;
  std::vector<int> tie_per_angle;
  std::vector<int> h_view_angle;
  std::vector<double> h_cs;  // (cos, sin) of every unique angle (incl. the exact per-column maps)
  std::vector<uint32_t> cand_flags;
  long long u_total = 0;
  // device (non-const views of BD members)
  double* d_cs = nullptr;
  void* d_fmap = nullptr;
  uint8_t* d_rayvalid = nullptr;
  int* d_tie = nullptr;
  uint16_t* d_amap = nullptr;
  int* d_sym_g = nullptr;                        // per symmetry row: reference index of its generating voxel
  std::vector<std::vector<int>> h_sym_round_end;  // [round][nc] rows of the candidate after that pair round
  int* d_sym_a = nullptr; int* d_sym_b = nullptr; int* d_csc_ptr = nullptr; int* d_csc_ent = nullptr; int* d_ell = nullptr;
  float* d_bmax = nullptr;
  float* d_score = nullptr;
  float* d_chain = nullptr;  // [2][nc]: sums of squares of u~ and v~ as the reference's BLAS accumulates them
  int* d_nactive = nullptr;
  int* h_nactive = nullptr;  // pinned
  double timing[16] = {0};
  std::vector<TrfState> last_trf;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<std::pair<int, int>> ev_used;  // (class, index of start event)
  size_t ev_next = 0;
  bool profiling = false;
  bool solved = false;
  // side stream of the LSMR loop: the symmetry-row forward (HBM / L2 bound) runs beside the data-row band kernel
  // (shared-memory bound; one 196 KB CTA of 768 threads per SM leaves room for two 256-thread blocks)
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

extern "C" const char* hb2_last_error(void) { return g_err.c_str(); }
extern "C" int hb2_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
extern "C" const char* hb2_build_info(void) { return "helicon_b200 sm_100a " __DATE__ " " __TIME__; }

extern "C" int hb2_stream_create(int device, void** out) {
  if (!out) return fail(HB2_ERR_ARG, "null argument");
  if (hb2_device_count() <= 0) return fail(HB2_ERR_NO_DEVICE, "no CUDA device visible; helicon_b200 has no CPU fallback");
  CK(cudaSetDevice(device));
  cudaStream_t st;
  CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  *out = (void*)st;
  return HB2_OK;
}
extern "C" int hb2_stream_destroy(int device, void* stream) {
  if (!stream) return HB2_OK;
  CK(cudaSetDevice(device));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  {  // the stream's arena goes with it
    std::lock_guard<std::mutex> lk(g_arena_mu);
    auto it = g_arenas.find({device, (cudaStream_t)stream});
    if (it != g_arenas.end() && it->second->live == 0) {
      if (it->second->base) cudaFree(it->second->base);
      delete it->second;
      g_arenas.erase(it);
    }
  }
  CK(cudaStreamDestroy((cudaStream_t)stream));
  return HB2_OK;
}
extern "C" int hb2_device_trim(int device) {
  if (hb2_device_count() <= 0) return HB2_OK;
  CK(cudaSetDevice(device));
  CK(cudaDeviceSynchronize());
  std::lock_guard<std::mutex> lk(g_arena_mu);
  for (auto& kv : g_arenas) {
    Arena* a = kv.second;
    if (kv.first.first == device && a->live == 0 && a->base) { cudaFree(a->base); a->base = nullptr; a->cap = 0; a->top = 0; }
  }
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// problem
// ---------------------------------------------------------------------------
static void disk_tables(int G, double rmin, int rmax, std::vector<int>& rank, std::vector<short2>& yx) {
  // lib/analysis.py:731-774: X*X + Y*Y < rmax*rmax, and >= rmin*rmin when 0 < rmin < rmax
  rank.assign((size_t)G * G, -1);
  yx.clear();
  int c0 = G / 2;
  for (int y = 0; y < G; ++y)
    for (int x = 0; x < G; ++x) {
      long long r2 = (long long)(x - c0) * (x - c0) + (long long)(y - c0) * (y - c0);
      bool in = r2 < (long long)rmax * rmax;
      if (in && rmin > 0 && rmin < rmax) in = (double)r2 >= rmin * rmin;
      if (in) {
        rank[(size_t)y * G + x] = (int)yx.size();
        yx.push_back(make_short2((short)y, (short)x));
      }
    }
}

// Internal voxel order ("band-column-major"): the disk is cut into BANDS of TH = 16 voxel rows (relative to the mask's
// bounding box); inside a band voxels are numbered column by column (x-major, then y).  Consequences:
//  * a band is ONE contiguous run of ranks -> one TMA bulk copy stages it in shared memory (forward band kernel), and
//    rank - band_begin is the shared-memory slot;
//  * neighbouring rows of a column are neighbouring records, and a full column is 16 records = a multiple of 8: the
//    bank group of a 16-byte chunk depends on the ROW only, so lanes that sit on adjacent rays at the same depth sample
//    (one row apart at view angles below 45 degrees) read distinct bank groups -- conflict-free 128-bit shared loads;
//  * TW = 16 consecutive columns of a band (<= 256 consecutive ranks) form a compact 16 x 16 patch: the adjoint tile,
//    whose rays are a short contiguous range in every view.
// HB2_VOXEL_ORDER=0 restores round 1's row-major 8 x 32 tiles (tile by tile).  The reference order is kept for
// everything exported and for the enumeration order of the symmetry rows.
static void tile_order(const std::vector<short2>& yx_ref, std::vector<int>& int2ref, std::vector<int>& tile_begin,
                       std::vector<int>& tilerow_begin, bool& tile_ok, int interpolation) {
  // read per problem (not latched), so that tests can compare the orders inside one process
  const char* e_o = getenv("HB2_VOXEL_ORDER"); const char* e_h = getenv("HB2_TILE_H"); const char* e_w = getenv("HB2_TILE_W");
  // Problems of trilinear searches (hb2_geometry.interpolation = 1) default to the row-major tiles: the footprint list of
  // a ray is sorted by voxel rank, and with x-contiguous ranks 10 consecutive entries touch ~half as many cache lines
  // (k_fwd_bil: 72 -> 59 us per candidate-pass at cfg2; 8 x 32, 16 x 16, 4 x 64 tiles within 2 us of each other, the
  // tile adjoint prefers the compact ones -- profiles/r2_summary.md section 8)
  const int ORDER = e_o ? atoi(e_o) : (interpolation == 1 ? 0 : 1);
  const int TH = e_h ? std::max(1, atoi(e_h)) : (ORDER ? 16 : 8);
  const int TW = e_w ? std::max(1, atoi(e_w)) : (ORDER ? 16 : 32);
  tile_ok = (long long)TH * TW <= HB2_BLOCK;
  int ymin = 1 << 30, xmin = 1 << 30;
  for (const short2& q : yx_ref) { ymin = std::min<int>(ymin, q.x); xmin = std::min<int>(xmin, q.y); }
  int2ref.resize(yx_ref.size());
  for (size_t i = 0; i < yx_ref.size(); ++i) int2ref[i] = (int)i;
  auto tkey = [&](int r) { return std::make_pair((yx_ref[r].x - ymin) / TH, (yx_ref[r].y - xmin) / TW); };
  if (ORDER) {
    std::sort(int2ref.begin(), int2ref.end(), [&](int a, int b) {
      const int ba = (yx_ref[a].x - ymin) / TH, bb = (yx_ref[b].x - ymin) / TH;
      if (ba != bb) return ba < bb;
      if (yx_ref[a].y != yx_ref[b].y) return yx_ref[a].y < yx_ref[b].y;
      return yx_ref[a].x < yx_ref[b].x;
    });
  } else {
    std::sort(int2ref.begin(), int2ref.end(), [&](int a, int b) {
      return std::make_pair(tkey(a), a) < std::make_pair(tkey(b), b);  // reference rank is row-major already
    });
  }
  tile_begin.clear();
  for (size_t i = 0; i < int2ref.size(); ++i)
    if (i == 0 || tkey(int2ref[i]) != tkey(int2ref[i - 1])) tile_begin.push_back((int)i);
  tile_begin.push_back((int)int2ref.size());
  tilerow_begin.clear();
  for (size_t i = 0; i < int2ref.size(); ++i)
    if (i == 0 || tkey(int2ref[i]).first != tkey(int2ref[i - 1]).first) tilerow_begin.push_back((int)i);
  tilerow_begin.push_back((int)int2ref.size());
}

extern "C" int hb2_problem_create(hb2_problem** out, const float* image, const hb2_geometry* g, int device, void* stream) {
  if (!out || !image || !g) return fail(HB2_ERR_ARG, "null argument");
  if (hb2_device_count() <= 0) return fail(HB2_ERR_NO_DEVICE, "no CUDA device visible; helicon_b200 has no CPU fallback");
  if (g->interpolation != 0 && g->interpolation != 1) return fail(HB2_ERR_GEOMETRY, "hb2_geometry.interpolation: 0 (nn) or 1 (linear)");
  if (g->D2 <= 0 || g->L2 <= 0 || g->D3 <= 0 || g->D2 > 32000 || g->L2 > 32000)
    return fail(HB2_ERR_ARG, "bad reconstruct sizes");
  if (g->D2 / 2 > g->ny / 2 + 0 && (g->D2 > g->ny)) return fail(HB2_ERR_ARG, "D2 larger than the image");
  if (g->L2 > g->nx) return fail(HB2_ERR_ARG, "L2 larger than the image");
  CK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  auto* P = new hb2_problem();
  P->device = device;
  P->g = *g;
  std::vector<int> rd, rs;
  std::vector<short2> yd, ys;
  disk_tables(g->D2, g->rmin, g->rmax, rd, yd);
  disk_tables(g->D3, g->rmin, g->rmax, rs, ys);
  if (yd.size() != ys.size() || yd.empty()) {
    delete P;
    return fail(HB2_ERR_GEOMETRY,
                "the cylinder mask has a different voxel count on the 2-D (D2) and 3-D (D3) grids (or is empty); "
                "the reference cannot scatter such a solution either (SLR:538)");
  }
  P->ndisk = (int)yd.size();
  P->h_rank_data = rd;
  {
    std::vector<int> i2r_sym, tb_sym, tr_sym;
    bool ok_sym;
    tile_order(yd, P->int2ref, P->h_tile_begin, P->h_tilerow_begin, P->tile_ok, g->interpolation);
    tile_order(ys, i2r_sym, tb_sym, tr_sym, ok_sym, g->interpolation);
    P->ntile = (int)P->h_tile_begin.size() - 1;
    if (i2r_sym != P->int2ref) {
      delete P;
      return fail(HB2_ERR_GEOMETRY, "the cylinder mask is not the same voxel set on the 2-D (D2) and 3-D (D3) grids");
    }
    P->ref2int.resize(P->ndisk);
    for (int i = 0; i < P->ndisk; ++i) P->ref2int[P->int2ref[i]] = i;
  }
  std::vector<short2> yd_int(yd.size());
  for (int i = 0; i < P->ndisk; ++i) yd_int[i] = yd[P->int2ref[i]];
  for (int& r : rd) if (r >= 0) r = P->ref2int[r];
  for (int& r : rs) if (r >= 0) r = P->ref2int[r];
  // crop: SLR:1706-1708
  std::vector<float> pix((size_t)g->D2 * g->L2);
  for (int j = 0; j < g->D2; ++j)
    for (int k = 0; k < g->L2; ++k) {
      int yy = j - g->D2 / 2 + g->ny / 2, xx = k - g->L2 / 2 + g->nx / 2;
      // numpy fancy indexing wraps negative indices (odd sizes can reach -1)
      if (yy < 0) yy += g->ny;
      if (xx < 0) xx += g->nx;
      pix[(size_t)j * g->L2 + k] = image[(size_t)yy * g->nx + xx];
    }
  CK(cudaMalloc(&P->d_pix, pix.size() * sizeof(float)));
  CK(cudaMalloc(&P->d_rank_data, rd.size() * sizeof(int)));
  CK(cudaMalloc(&P->d_rank_sym, rs.size() * sizeof(int)));
  CK(cudaMalloc(&P->d_yx_data, yd.size() * sizeof(short2)));
  CK(cudaMalloc(&P->d_yx_sym, ys.size() * sizeof(short2)));
  std::vector<int> aslot(P->ndisk);
  for (int t = 0; t < P->ntile; ++t)
    for (int i = P->h_tile_begin[t]; i < P->h_tile_begin[t + 1]; ++i) aslot[i] = t * HB2_BLOCK + (i - P->h_tile_begin[t]);
  CK(cudaMalloc(&P->d_int2ref, P->int2ref.size() * sizeof(int)));
  CK(cudaMemcpyAsync(P->d_int2ref, P->int2ref.data(), P->int2ref.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMalloc(&P->d_tile_begin, P->h_tile_begin.size() * sizeof(int)));
  CK(cudaMalloc(&P->d_aslot, aslot.size() * sizeof(int)));
  CK(cudaMemcpyAsync(P->d_tile_begin, P->h_tile_begin.data(), P->h_tile_begin.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_aslot, aslot.data(), aslot.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_pix, pix.data(), pix.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_rank_data, rd.data(), rd.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_rank_sym, rs.data(), rs.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_yx_data, yd_int.data(), yd_int.size() * sizeof(short2), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(P->d_yx_sym, ys.data(), ys.size() * sizeof(short2), cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));  // host vectors go out of scope
  *out = P;
  return HB2_OK;
}

extern "C" void hb2_problem_destroy(hb2_problem* P) {
  if (!P) return;
  cudaSetDevice(P->device);
  cudaFree(P->d_tile_begin); cudaFree(P->d_aslot); cudaFree(P->d_int2ref);
  cudaFree(P->d_pix); cudaFree(P->d_rank_data); cudaFree(P->d_rank_sym); cudaFree(P->d_yx_data); cudaFree(P->d_yx_sym);
  delete P;
}
extern "C" int hb2_problem_ndisk(const hb2_problem* P) { return P ? P->ndisk : 0; }
extern "C" int hb2_problem_rank_table(const hb2_problem* P, int32_t* out) {
  if (!P || !out) return fail(HB2_ERR_ARG, "null argument");
  memcpy(out, P->h_rank_data.data(), P->h_rank_data.size() * sizeof(int));
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// batch step 1: in-plane maps
// ---------------------------------------------------------------------------
extern "C" int hb2_batch_begin(hb2_batch** out, hb2_problem* P, int32_t L3, int32_t MC, int32_t nA, const double* cos_sin,
                               int32_t* nvalid_rays, int32_t* tie_samples, void* stream) {
  if (!out || !P || !cos_sin || nA <= 0 || L3 <= 0 || MC <= 0) return fail(HB2_ERR_ARG, "bad argument");
  NvtxRange nvtx_("build_A_data_matrix - nn: in-plane maps");
  if ((long long)L3 * MC > HB2_MAX_ZMC) return fail(HB2_ERR_GEOMETRY, "L3*MC exceeds HB2_MAX_ZMC");
  if ((long long)(L3 + 3) * P->ndisk >= (1ll << 31)) return fail(HB2_ERR_GEOMETRY, "too many unknowns");
  CK(cudaSetDevice(P->device));
  auto* b = new hb2_batch();
  b->pool.owner = b;
  b->P = P;
  b->stream = (cudaStream_t)stream;
  cudaStream_t st = b->stream;
  BD& B = b->B;
  const hb2_geometry& g = P->g;
  B.D2 = g.D2; B.L2 = g.L2; B.D3 = g.D3; B.ndisk = P->ndisk; B.L3 = L3; B.MC = MC; B.ZMC = L3 * MC;
  B.L3P = (L3 + 3) / 4 * 4; B.ZMP = (B.ZMC + 3) / 4 * 4;
  B.n = L3 * P->ndisk; B.nrp = (B.n + 31) / 32 * 32; B.npad = B.L3P * P->ndisk; B.rows_per_view = B.ZMP * g.D2;
  B.nA = nA; B.s = g.scale2d_to_3d; B.only_cand = -1;
  b->idx16 = P->ndisk < 65535;
  size_t ns = (size_t)nA * g.D2 * g.D2;
#define BEGIN_FAIL(e) do { b->pool.free_all(); delete b; return (e); } while (0)
#define CKB(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { std::string m_ = std::string(#call) + ": " + cudaGetErrorString(e_); b->pool.free_all(); delete b; return fail(HB2_ERR_CUDA, m_); } } while (0)
  CKB(b->pool.alloc(&b->d_cs, (size_t)2 * nA, false, st));
  CKB(cudaMemcpyAsync(b->d_cs, cos_sin, sizeof(double) * 2 * nA, cudaMemcpyHostToDevice, st));
  b->h_cs.assign(cos_sin, cos_sin + 2 * (size_t)nA);
  if (b->idx16) { uint16_t* p; CKB(b->pool.alloc(&p, ns, false, st)); b->d_fmap = p; }
  else { uint32_t* p; CKB(b->pool.alloc(&p, ns, false, st)); b->d_fmap = p; }
  CKB(b->pool.alloc(&b->d_rayvalid, (size_t)nA * g.D2, true, st));
  CKB(b->pool.alloc(&b->d_tie, (size_t)nA, true, st));
  if (b->idx16)
    k_build_fmap<uint16_t><<<cdiv(ns, 256), 256, 0, st>>>(nA, g.D2, g.scale2d_to_3d, b->d_cs, P->d_rank_data, (uint16_t*)b->d_fmap, b->d_rayvalid, b->d_tie);
  else
    k_build_fmap<uint32_t><<<cdiv(ns, 256), 256, 0, st>>>(nA, g.D2, g.scale2d_to_3d, b->d_cs, P->d_rank_data, (uint32_t*)b->d_fmap, b->d_rayvalid, b->d_tie);
  CKB(cudaGetLastError());
  std::vector<uint8_t> rv((size_t)nA * g.D2);
  b->tie_per_angle.resize(nA);
  CKB(cudaMemcpyAsync(rv.data(), b->d_rayvalid, rv.size(), cudaMemcpyDeviceToHost, st));
  CKB(cudaMemcpyAsync(b->tie_per_angle.data(), b->d_tie, sizeof(int) * nA, cudaMemcpyDeviceToHost, st));
  CKB(cudaStreamSynchronize(st));
  for (int a = 0; a < nA; ++a) {
    int cnt = 0;
    for (int j = 0; j < g.D2; ++j) cnt += rv[(size_t)a * g.D2 + j];
    if (nvalid_rays) nvalid_rays[a] = cnt;
    if (tie_samples) tie_samples[a] = b->tie_per_angle[a];
  }
  B.fmap = b->d_fmap; B.rayvalid = b->d_rayvalid;
  *out = b;
  return HB2_OK;
}

// Exact per-column maps for in-plane tie views: appended to the batch's angle table as extra "angles".
extern "C" int hb2_batch_add_exact_maps(hb2_batch* b, int32_t nE, const double* cos_sin, const double* x0rows,
                                        int32_t* nvalid_rays) {
  if (!b || nE <= 0 || !cos_sin || !x0rows) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "hb2_batch_add_exact_maps must precede hb2_batch_create");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  const int D2 = B.D2, nA = B.nA, nT = nA + nE;
  const size_t per = (size_t)D2 * D2, esz = b->idx16 ? 2 : 4;
  double* cs2; void* fm2; uint8_t* rv2; int* tie2; double* d_x0;
  CK(b->pool.alloc(&cs2, (size_t)2 * nT, false, st));
  { uint8_t* p; CK(b->pool.alloc(&p, (size_t)nT * per * esz, false, st)); fm2 = p; }
  CK(b->pool.alloc(&rv2, (size_t)nT * D2, true, st));
  CK(b->pool.alloc(&tie2, (size_t)nT, true, st));
  CK(b->pool.alloc(&d_x0, (size_t)nE * D2, false, st));
  CK(cudaMemcpyAsync(cs2, b->d_cs, sizeof(double) * 2 * nA, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(cs2 + 2 * nA, cos_sin, sizeof(double) * 2 * nE, cudaMemcpyHostToDevice, st));
  b->h_cs.insert(b->h_cs.end(), cos_sin, cos_sin + 2 * (size_t)nE);
  CK(cudaMemcpyAsync(fm2, b->d_fmap, (size_t)nA * per * esz, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(rv2, b->d_rayvalid, (size_t)nA * D2, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(tie2, b->d_tie, sizeof(int) * nA, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(d_x0, x0rows, sizeof(double) * nE * D2, cudaMemcpyHostToDevice, st));
  const long long ns = (long long)nE * per;
  if (b->idx16)
    k_build_fmap_exact<uint16_t><<<cdiv(ns, 256), 256, 0, st>>>(nE, D2, B.s, cs2 + 2 * nA, d_x0, P->d_rank_data,
                                                                  (uint16_t*)fm2 + (size_t)nA * per, rv2 + (size_t)nA * D2);
  else
    k_build_fmap_exact<uint32_t><<<cdiv(ns, 256), 256, 0, st>>>(nE, D2, B.s, cs2 + 2 * nA, d_x0, P->d_rank_data,
                                                                  (uint32_t*)fm2 + (size_t)nA * per, rv2 + (size_t)nA * D2);
  CKL();
  std::vector<uint8_t> rv((size_t)nE * D2);
  CK(cudaMemcpyAsync(rv.data(), rv2 + (size_t)nA * D2, rv.size(), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int a = 0; a < nE; ++a) {
    int cnt = 0;
    for (int j = 0; j < D2; ++j) cnt += rv[(size_t)a * D2 + j];
    if (nvalid_rays) nvalid_rays[a] = cnt;
  }
  b->d_cs = cs2; b->d_fmap = fm2; b->d_rayvalid = rv2; b->d_tie = tie2;
  b->tie_per_angle.resize(nT, 0);
  B.nA = nT; B.fmap = fm2; B.rayvalid = rv2;
  return HB2_OK;
}

// Half-set mask for explicit rows (fsc_test): rows whose pixel id is not set are dropped AFTER the early stop
// (the reference splits the finished matrix, SLR:441-444).  Call before hb2_batch_explicit_rows.
extern "C" int hb2_batch_explicit_pixel_mask(hb2_batch* b, const uint8_t* mask) {
  if (!b) return fail(HB2_ERR_ARG, "null argument");
  if (b->explicit_rows) return fail(HB2_ERR_STATE, "hb2_batch_explicit_pixel_mask must precede hb2_batch_explicit_rows");
  if (mask) b->h_exp_pixmask.assign(mask, mask + (size_t)b->B.L2 * b->B.D2);
  else b->h_exp_pixmask.clear();
  return HB2_OK;
}

// Explicit data rows (general orientation and/or trilinear interpolation): built on the GPU, see hb2_explicit.cuh.
extern "C" int hb2_batch_explicit_rows(hb2_batch* b, const hb2_explicit_geometry* eg, int32_t ncopies, const double* copy_mats,
                                       const double* zshift, const double* xtab, const double* ztab,
                                       int64_t min_projection_lines, int32_t* copies_used, int32_t* rows_per_copy,
                                       int64_t* n_rows, int64_t* nnz_out) {
  NvtxRange nvtx_("build csr matrix (explicit rows: linear / tilted)");
  if (!b || !eg || ncopies <= 0 || !copy_mats || !zshift || !xtab || !ztab) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "hb2_batch_explicit_rows must precede hb2_batch_create");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  ExpGeo G{};
  G.D2 = B.D2; G.L2 = B.L2; G.L3 = B.L3; G.L3P = B.L3P; G.linear = eg->interpolation == 1 ? 1 : 0;
  G.s = B.s; G.dy = eg->dy_pixel;
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) G.Ayx[r * 3 + c] = eg->rot_yx[c * 3 + r];  // transpose: apply(inverse=True)
  std::vector<ExpCopy> hc(ncopies);
  for (int q = 0; q < ncopies; ++q) {
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) hc[q].A[r * 3 + c] = copy_mats[(size_t)q * 9 + c * 3 + r];
    hc[q].zshift = zshift[q];
  }
  const long long R = (long long)B.L2 * B.D2, NT = (long long)ncopies * R;
  if (NT >= (1ll << 31)) return fail(HB2_ERR_CAPACITY, "too many potential rows");
  ExpCopy* d_cp; double *d_xt, *d_zt; int *d_cnt, *d_flag, *d_off, *d_ridx;
  CK(b->pool.alloc(&d_cp, (size_t)ncopies, false, st));
  CK(b->pool.alloc(&d_xt, (size_t)R, false, st));
  CK(b->pool.alloc(&d_zt, (size_t)R, false, st));
  CK(b->pool.alloc(&d_cnt, (size_t)NT + 1, true, st));
  CK(b->pool.alloc(&d_flag, (size_t)NT + 1, true, st));
  CK(b->pool.alloc(&d_off, (size_t)NT + 1, false, st));
  CK(b->pool.alloc(&d_ridx, (size_t)NT + 1, false, st));
  CK(cudaMemcpyAsync(d_cp, hc.data(), sizeof(ExpCopy) * ncopies, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_xt, xtab, sizeof(double) * R, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_zt, ztab, sizeof(double) * R, cudaMemcpyHostToDevice, st));
  k_exp_rows<0><<<cdiv(NT, 128), 128, 0, st>>>(G, ncopies, d_cp, d_xt, d_zt, P->d_rank_data, P->d_pix, d_cnt, nullptr, nullptr,
                                                nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  k_exp_flags<<<cdiv(NT, 256), 256, 0, st>>>(NT, d_cnt, d_flag);
  CKL();
  // row index of every potential row (exclusive scan of the flags; NT + 1 entries so the total is the last one)
  size_t sb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, sb, d_flag, d_ridx, (int)(NT + 1), st);
  void* d_tmp; { uint8_t* p; CK(b->pool.alloc(&p, sb, false, st)); d_tmp = p; }
  CK(cub::DeviceScan::ExclusiveSum(d_tmp, sb, d_flag, d_ridx, (int)(NT + 1), st));
  std::vector<int> bound(ncopies + 1);
  CK(cudaMemcpy2DAsync(bound.data(), sizeof(int), d_ridx, sizeof(int) * R, sizeof(int), ncopies + 1, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  // SLR:1640-1647: copies are appended until the row count exceeds min_projection_lines
  int used = ncopies;
  for (int q = 0; q < ncopies; ++q) {
    if (rows_per_copy) rows_per_copy[q] = bound[q + 1] - bound[q];
    if (min_projection_lines > 0 && bound[q + 1] > min_projection_lines) { used = q + 1; break; }
  }
  if (rows_per_copy) for (int q = used; q < ncopies; ++q) rows_per_copy[q] = bound[q + 1] - bound[q];
  const long long NU = (long long)used * R;
  int m = bound[used];
  if (!b->h_exp_pixmask.empty()) {  // half set: drop the other half's rows, keep the order
    uint8_t* d_pm;
    CK(b->pool.alloc(&d_pm, (size_t)R, false, st));
    CK(cudaMemcpyAsync(d_pm, b->h_exp_pixmask.data(), (size_t)R, cudaMemcpyHostToDevice, st));
    k_exp_maskrows<<<cdiv(NU, 256), 256, 0, st>>>(NU, R, B.D2, d_pm, d_cnt);
    k_exp_flags<<<cdiv(NT, 256), 256, 0, st>>>(NT, d_cnt, d_flag);
    CKL();
    CK(cub::DeviceScan::ExclusiveSum(d_tmp, sb, d_flag, d_ridx, (int)(NT + 1), st));
    CK(cudaMemcpyAsync(&m, d_ridx + NU, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  // entry offsets over the used copies: the count pass may exceed 2^31 entries in total, so check with a 64-bit sum
  {
    std::vector<int> hcnt((size_t)NU);
    CK(cudaMemcpyAsync(hcnt.data(), d_cnt, sizeof(int) * NU, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    long long tot = 0;
    for (long long t = 0; t < NU; ++t) tot += hcnt[t];
    if (tot >= (1ll << 31) - 64) return fail(HB2_ERR_CAPACITY, "explicit rows exceed 2^31 matrix entries");
    b->exp_nnz = tot;
  }
  CK(cudaMemsetAsync(d_cnt + NU, 0, sizeof(int), st));
  CK(cub::DeviceScan::ExclusiveSum(d_tmp, sb, d_cnt, d_off, (int)(NU + 1), st));
  const long long nnz = b->exp_nnz;
  int *d_ptr, *d_col, *d_erow, *d_pid; float *d_w, *d_rb;
  CK(b->pool.alloc(&d_ptr, (size_t)m + 1, false, st));
  CK(b->pool.alloc(&d_col, (size_t)nnz, false, st));
  CK(b->pool.alloc(&d_w, (size_t)nnz, false, st));
  CK(b->pool.alloc(&d_erow, (size_t)nnz, false, st));
  CK(b->pool.alloc(&d_rb, (size_t)m, false, st));
  CK(b->pool.alloc(&d_pid, (size_t)m, false, st));
  if (m > 0) {
    k_exp_rows<1><<<cdiv(NU, 128), 128, 0, st>>>(G, used, d_cp, d_xt, d_zt, P->d_rank_data, P->d_pix, d_cnt, d_off, d_ridx, d_col,
                                                  d_w, d_erow, d_ptr, d_rb, d_pid);
    CKL();
  }
  {
    const int nnz_i = (int)nnz;
    CK(cudaMemcpyAsync(d_ptr + m, &nnz_i, sizeof(int), cudaMemcpyHostToDevice, st));
  }
  // trilinear rows: merge the duplicate entries of every row (k_exp_merge); rows of at most 8*D2 entries fit shared memory
  static const bool no_merge = getenv("HB2_NO_MERGE") && atoi(getenv("HB2_NO_MERGE"));
  int maxe = 1;
  while (maxe < 8 * B.D2) maxe <<= 1;  // a row has at most 8*D2 entries; the sort works on the next power of two
  const size_t msm = (size_t)maxe * (sizeof(unsigned long long) + sizeof(float));
  if (G.linear && m > 0 && nnz > 0 && !no_merge && msm <= 160 * 1024) {
    int *d_ucnt, *d_nptr;
    CK(b->pool.alloc(&d_ucnt, (size_t)m + 1, true, st));
    CK(b->pool.alloc(&d_nptr, (size_t)m + 1, false, st));
    hb2_allow_big_smem((const void*)k_exp_merge<0>);
    k_exp_merge<0><<<m, HB2_MERGE_THREADS, msm, st>>>(m, maxe, d_ptr, d_col, d_w, d_ucnt, nullptr, nullptr, nullptr, nullptr);
    CKL();
    size_t sb6 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, sb6, d_ucnt, d_nptr, m + 1, st);
    void* d_t6; { uint8_t* p; CK(b->pool.alloc(&p, sb6, false, st)); d_t6 = p; }
    CK(cub::DeviceScan::ExclusiveSum(d_t6, sb6, d_ucnt, d_nptr, m + 1, st));
    int nnz_m = 0;
    CK(cudaMemcpyAsync(&nnz_m, d_nptr + m, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int *d_ncol, *d_nerow; float* d_nw;
    CK(b->pool.alloc(&d_ncol, (size_t)std::max(nnz_m, 1), false, st));
    CK(b->pool.alloc(&d_nw, (size_t)std::max(nnz_m, 1), false, st));
    CK(b->pool.alloc(&d_nerow, (size_t)std::max(nnz_m, 1), false, st));
    k_exp_merge<1><<<m, HB2_MERGE_THREADS, 0, st>>>(m, maxe, d_ptr, d_col, d_w, nullptr, d_nptr, d_ncol, d_nw, d_nerow);
    CKL();
    d_ptr = d_nptr; d_col = d_ncol; d_w = d_nw; d_erow = d_nerow;
    b->exp_nnz = nnz_m;
  }
  // max(b) over the rows: upper bound of the positive constraint (SLR:248)
  std::vector<float> hb((size_t)std::max(m, 1), 0.f);
  if (m > 0) CK(cudaMemcpyAsync(hb.data(), d_rb, sizeof(float) * m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  float bm = m > 0 ? hb[0] : 0.f;
  for (int r = 1; r < m; ++r) bm = std::max(bm, hb[r]);
  b->exp_bmax = bm;
  b->explicit_rows = true;
  b->d_exp_b = d_rb; b->d_exp_pid = d_pid;
  b->exp_md = m; b->d_exp_ptr = d_ptr; b->d_exp_col = d_col; b->d_exp_w = d_w; b->d_exp_erow = d_erow;
  B.exp_m = m; B.exp_m_data = m; B.exp_ptr = d_ptr; B.exp_col = d_col; B.exp_w = d_w;
  if (copies_used) *copies_used = used;
  if (n_rows) *n_rows = m;
  if (nnz_out) *nnz_out = b->exp_nnz;
  return HB2_OK;
}

// Trilinear symmetry rows, see hb2_explicit.cuh.  pair_mats[p*12 ..] = M00, M01, M10, M11, M22, rise*h of member i,
// then of member j (scipy's as_matrix entries).  One round per pair; stops when the row count reaches min_sym_pairs.
extern "C" int hb2_batch_explicit_sym_rows(hb2_batch* b, int32_t npairs, const double* pair_mats, int64_t min_sym_pairs,
                                           int64_t* n_rows) {
  if (!b || npairs < 0 || (npairs > 0 && !pair_mats)) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "hb2_batch_explicit_sym_rows must precede hb2_batch_create");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  b->ls_m = 0;
  if (n_rows) *n_rows = 0;
  if (npairs == 0 || min_sym_pairs < 0) return HB2_OK;
  static_assert(sizeof(LsymPair) == 12 * sizeof(double), "LsymPair layout");
  const long long cap_rows = std::min<long long>(min_sym_pairs + B.n, (long long)npairs * B.n);
  if (cap_rows * 16 >= (1ll << 31)) return fail(HB2_ERR_CAPACITY, "too many trilinear symmetry rows");
  LsymSetup Q{};
  Q.n = B.n; Q.ndisk = B.ndisk; Q.D3 = B.D3; Q.L3 = B.L3; Q.L3P = B.L3P;
  Q.rank_sym = P->d_rank_sym; Q.disk_yx_sym = P->d_yx_sym;
  Q.tab_cap = (unsigned long long)(2 * cap_rows + 17);
  LsymPair* d_pairs; int* d_ov;
  CK(b->pool.alloc(&d_pairs, (size_t)npairs, false, st));
  CK(cudaMemcpyAsync(d_pairs, pair_mats, sizeof(LsymPair) * npairs, cudaMemcpyHostToDevice, st));
  CK(b->pool.alloc(&Q.tab_key, (size_t)Q.tab_cap, false, st));
  CK(b->pool.alloc(&Q.tab_seq, (size_t)Q.tab_cap, false, st));
  CK(cudaMemsetAsync(Q.tab_key, 0xFF, sizeof(unsigned long long) * Q.tab_cap, st));
  CK(cudaMemsetAsync(Q.tab_seq, 0xFF, sizeof(unsigned long long) * Q.tab_cap, st));
  CK(b->pool.alloc(&Q.tmp_a, (size_t)B.n + 1, false, st));
  CK(b->pool.alloc(&Q.tmp_b, (size_t)B.n + 1, false, st));
  CK(b->pool.alloc(&Q.flag, (size_t)B.n + 1, true, st));
  CK(b->pool.alloc(&Q.pos, (size_t)B.n + 1, true, st));
  CK(b->pool.alloc(&d_ov, 1, true, st));
  Q.overflow = d_ov;
  CK(b->pool.alloc(&b->d_ls_col, (size_t)cap_rows * 16, false, st));
  CK(b->pool.alloc(&b->d_ls_w, (size_t)cap_rows * 16, false, st));
  size_t sb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, sb, Q.flag, Q.pos, B.n + 1, st);
  void* d_tmp; { uint8_t* p; CK(b->pool.alloc(&p, sb, false, st)); d_tmp = p; }
  long long rows = 0;
  const unsigned gn = cdiv((long long)B.n + 1, 256);
  for (int rnd = 0; rnd < npairs; ++rnd) {
    k_lsym_insert<<<gn, 256, 0, st>>>(Q, d_pairs, rnd);
    k_lsym_check<<<gn, 256, 0, st>>>(Q, rnd);
    CK(cub::DeviceScan::ExclusiveSum(d_tmp, sb, Q.flag, Q.pos, B.n + 1, st));
    k_lsym_emit<<<gn, 256, 0, st>>>(Q, d_pairs, rnd, (int)rows, (int)cap_rows, b->d_ls_col, b->d_ls_w);
    CKL();
    int h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], Q.pos + B.n, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[1], d_ov, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (h[1]) return fail(HB2_ERR_CAPACITY, "trilinear symmetry rows: table overflow");
    rows += h[0];
    if (rows >= min_sym_pairs) break;  // SLR:1286
  }
  b->ls_m = (int)rows;
  if (n_rows) *n_rows = rows;
  return HB2_OK;
}

extern "C" int hb2_batch_explicit_sym_export(hb2_batch* b, int32_t* cols, float* w) {
  if (!b) return fail(HB2_ERR_ARG, "null argument");
  CK(cudaSetDevice(b->P->device));
  const size_t ne = (size_t)b->ls_m * 16;
  if (ne == 0) return HB2_OK;
  if (cols) CK(cudaMemcpyAsync(cols, b->d_ls_col, sizeof(int) * ne, cudaMemcpyDeviceToHost, b->stream));
  if (w) CK(cudaMemcpyAsync(w, b->d_ls_w, sizeof(float) * ne, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  if (cols) {
    const int L3P = b->B.L3P, nd = b->B.ndisk;
    const std::vector<int>& i2r = b->P->int2ref;
    for (size_t e = 0; e < ne; ++e) cols[e] = (cols[e] % L3P) * nd + i2r[cols[e] / L3P];
  }
  return HB2_OK;
}

// Appends the trilinear symmetry rows (b = 0) to the explicit rows and builds the transpose (stable sort of the entries
// by voxel -> deterministic adjoint order; column pointers from a histogram).  Called by hb2_batch_create.
static int exp_finish(hb2_batch* b) {
  if (b->exp_finished) return HB2_OK;
  cudaStream_t st = b->stream;
  BD& B = b->B;
  const int md = b->exp_md, ms = b->ls_m, m = md + ms;
  const long long nnz_d = b->exp_nnz, nnz = nnz_d + 16ll * ms;
  if (nnz >= (1ll << 31) - 64) return fail(HB2_ERR_CAPACITY, "explicit rows exceed 2^31 matrix entries");
  if (ms > 0) {
    int *ptr, *col, *erow; float *w, *rb;
    CK(b->pool.alloc(&ptr, (size_t)m + 1, false, st));
    CK(b->pool.alloc(&col, (size_t)nnz, false, st));
    CK(b->pool.alloc(&w, (size_t)nnz, false, st));
    CK(b->pool.alloc(&erow, (size_t)nnz, false, st));
    CK(b->pool.alloc(&rb, (size_t)m, true, st));
    CK(cudaMemcpyAsync(ptr, b->d_exp_ptr, sizeof(int) * (md + 1), cudaMemcpyDeviceToDevice, st));
    if (nnz_d) {
      CK(cudaMemcpyAsync(col, b->d_exp_col, sizeof(int) * nnz_d, cudaMemcpyDeviceToDevice, st));
      CK(cudaMemcpyAsync(w, b->d_exp_w, sizeof(float) * nnz_d, cudaMemcpyDeviceToDevice, st));
      CK(cudaMemcpyAsync(erow, b->d_exp_erow, sizeof(int) * nnz_d, cudaMemcpyDeviceToDevice, st));
    }
    if (md) CK(cudaMemcpyAsync(rb, b->d_exp_b, sizeof(float) * md, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(col + nnz_d, b->d_ls_col, sizeof(int) * 16 * ms, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(w + nnz_d, b->d_ls_w, sizeof(float) * 16 * ms, cudaMemcpyDeviceToDevice, st));
    k_lsym_ptr<<<cdiv(16ll * ms + 1, 256), 256, 0, st>>>(md, (int)nnz_d, ms, ptr, erow);
    CKL();
    b->d_exp_ptr = ptr; b->d_exp_col = col; b->d_exp_w = w; b->d_exp_erow = erow; b->d_exp_b = rb;
  }
  int *d_cptr, *d_crow; float* d_cw;
  CK(b->pool.alloc(&d_cptr, (size_t)B.npad + 2, true, st));
  CK(b->pool.alloc(&d_crow, (size_t)std::max<long long>(nnz, 1), false, st));
  CK(b->pool.alloc(&d_cw, (size_t)std::max<long long>(nnz, 1), false, st));
  if (nnz > 0) {
    const int nnz_i = (int)nnz;
    int *d_keys2, *d_id, *d_id2, *d_cc;
    CK(b->pool.alloc(&d_keys2, (size_t)nnz, false, st));
    CK(b->pool.alloc(&d_id, (size_t)nnz, false, st));
    CK(b->pool.alloc(&d_id2, (size_t)nnz, false, st));
    CK(b->pool.alloc(&d_cc, (size_t)B.npad + 2, true, st));
    k_iota<<<cdiv(nnz, 256), 256, 0, st>>>(nnz_i, d_id);
    int bits = 1;
    while ((1ll << bits) < (long long)B.npad) ++bits;
    size_t sb3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sb3, b->d_exp_col, d_keys2, d_id, d_id2, nnz_i, 0, bits, st);
    void* d_t3; { uint8_t* p; CK(b->pool.alloc(&p, sb3, false, st)); d_t3 = p; }
    CK(cub::DeviceRadixSort::SortPairs(d_t3, sb3, b->d_exp_col, d_keys2, d_id, d_id2, nnz_i, 0, bits, st));
    k_exp_gather<<<cdiv(nnz, 256), 256, 0, st>>>(nnz_i, d_id2, b->d_exp_erow, b->d_exp_w, d_crow, d_cw);
    k_exp_colcount<<<cdiv(nnz, 256), 256, 0, st>>>(nnz_i, b->d_exp_col, d_cc);
    CKL();
    size_t sb4 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, sb4, d_cc, d_cptr, B.npad + 1, st);
    void* d_t4; { uint8_t* p; CK(b->pool.alloc(&p, sb4, false, st)); d_t4 = p; }
    CK(cub::DeviceScan::ExclusiveSum(d_t4, sb4, d_cc, d_cptr, B.npad + 1, st));
  }
  B.exp_m = m; B.exp_m_data = md;
  B.exp_ptr = b->d_exp_ptr; B.exp_col = b->d_exp_col; B.exp_w = b->d_exp_w;
  B.exp_cptr = d_cptr; B.exp_crow = d_crow; B.exp_cw = d_cw;
  b->exp_finished = true;
  return HB2_OK;
}

extern "C" int hb2_batch_explicit_export(hb2_batch* b, int64_t* indptr, int32_t* indices, float* data, float* b_out, int32_t* pid_out) {
  if (!b || !b->explicit_rows) return fail(HB2_ERR_STATE, "no explicit rows in this batch");
  CK(cudaSetDevice(b->P->device));
  cudaStream_t st = b->stream;
  const BD& B = b->B;
  const int m = b->exp_md;  // the data rows (trilinear symmetry rows: hb2_batch_explicit_sym_export)
  const long long nnz = b->exp_nnz;
  std::vector<int> ptr((size_t)m + 1);
  CK(cudaMemcpyAsync(ptr.data(), b->d_exp_ptr, sizeof(int) * (m + 1), cudaMemcpyDeviceToHost, st));
  if (indices && nnz) CK(cudaMemcpyAsync(indices, b->d_exp_col, sizeof(int) * nnz, cudaMemcpyDeviceToHost, st));
  if (data && nnz) CK(cudaMemcpyAsync(data, b->d_exp_w, sizeof(float) * nnz, cudaMemcpyDeviceToHost, st));
  if (b_out && m) CK(cudaMemcpyAsync(b_out, b->d_exp_b, sizeof(float) * m, cudaMemcpyDeviceToHost, st));
  if (pid_out && m) CK(cudaMemcpyAsync(pid_out, b->d_exp_pid, sizeof(int) * m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (indptr) for (int r = 0; r <= m; ++r) indptr[r] = ptr[r];
  if (indices) {  // internal p*L3P + z -> reference z*ndisk + rank
    const int L3P = B.L3P, nd = B.ndisk;
    const std::vector<int>& i2r = b->P->int2ref;
    for (long long e = 0; e < nnz; ++e) indices[e] = (indices[e] % L3P) * nd + i2r[indices[e] / L3P];
  }
  return HB2_OK;
}

extern "C" int hb2_batch_ray_valid(hb2_batch* b, uint8_t* out) {
  if (!b || !out) return fail(HB2_ERR_ARG, "null argument");
  CK(cudaSetDevice(b->P->device));
  CK(cudaMemcpyAsync(out, b->d_rayvalid, (size_t)b->B.nA * b->B.D2, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return HB2_OK;
}

extern "C" int hb2_batch_angle_map(hb2_batch* b, int32_t angle, int32_t* out) {
  if (!b || !out || angle < 0 || angle >= b->B.nA) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  size_t n = (size_t)b->B.D2 * b->B.D2;
  if (b->idx16) {
    std::vector<uint16_t> t(n);
    CK(cudaMemcpyAsync(t.data(), (uint16_t*)b->d_fmap + n * angle, n * 2, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    for (size_t i = 0; i < n; ++i) out[i] = t[i] == 0xFFFFu ? -1 : b->P->int2ref[t[i]];
  } else {
    std::vector<uint32_t> t(n);
    CK(cudaMemcpyAsync(t.data(), (uint32_t*)b->d_fmap + n * angle, n * 4, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    for (size_t i = 0; i < n; ++i) out[i] = t[i] == 0xFFFFFFFFu ? -1 : b->P->int2ref[t[i]];
  }
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// batch step 2: candidates
// ---------------------------------------------------------------------------
template <typename T>
static cudaError_t upload(DevPool& pool, const T** dst, const std::vector<T>& src, cudaStream_t st) {
  T* p = nullptr;
  cudaError_t e = pool.alloc(&p, src.size(), false, st);
  if (e != cudaSuccess) return e;
  if (!src.empty()) e = cudaMemcpyAsync(p, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, st);
  *dst = p;
  return e;
}

// ---------------------------------------------------------------------------
// Matrix-free trilinear rows (hb2_bilinear.cuh)
// ---------------------------------------------------------------------------
// In-plane bilinear footprint maps.  build_tables = 0: only ray validity and tie counts (the host decides from them which
// views need exact per-column maps); 1: also the transposed maps and the forward lists the kernels use (call once, with
// ALL maps of the batch).  xrows / zrows [n_tab_rows][D2]: rows of the reference's coordinate tables (SLR:1712-1719)
// that maps[].xrow / zrow index.
extern "C" int hb2_batch_bilinear_maps(hb2_batch* b, int32_t nM, const hb2_bilinear_map* maps, int32_t n_tab_rows,
                                       const double* xrows, const double* zrows, int32_t build_tables,
                                       int32_t* nvalid_rays, int32_t* tie_samples, uint64_t* content_hash) {
  if (!b || nM <= 0 || !maps || n_tab_rows < 0 || (n_tab_rows > 0 && (!xrows || !zrows))) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "hb2_batch_bilinear_maps must precede hb2_batch_create");
  static_assert(sizeof(BilMap) == sizeof(hb2_bilinear_map), "hb2_bilinear_map layout");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  NvtxRange nvtx_("build_A_data_matrix - linear: in-plane bilinear maps");
  if (B.s != 1.0 || B.MC != 1) return fail(HB2_ERR_GEOMETRY, "matrix-free trilinear rows need scale2d_to_3d == 1");
  if (B.L3P > 16) return fail(HB2_ERR_GEOMETRY, "matrix-free trilinear rows need L3 <= 16");
  if (!P->tile_ok) return fail(HB2_ERR_GEOMETRY, "HB2_TILE_H*HB2_TILE_W must be <= 256");
  const int D2 = B.D2;
  for (int m = 0; m < nM; ++m)
    if (maps[m].xrow >= n_tab_rows || maps[m].zrow >= n_tab_rows) return fail(HB2_ERR_ARG, "bad table row index");
  DevPool tmp;
  tmp.owner = b;
  DevPool& keep = build_tables ? b->pool : tmp;  // probe calls keep nothing
#define CKM(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { tmp.free_all(); return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
  BilMap* d_maps; double *d_x = nullptr, *d_z = nullptr; uint8_t* d_rv; int* d_tie;
  CKM(keep.alloc(&d_maps, (size_t)nM, false, st));
  CKM(cudaMemcpyAsync(d_maps, maps, sizeof(BilMap) * nM, cudaMemcpyHostToDevice, st));
  CKM(keep.alloc(&d_x, (size_t)std::max(n_tab_rows, 1) * D2, false, st));
  CKM(keep.alloc(&d_z, (size_t)std::max(n_tab_rows, 1) * D2, false, st));
  if (n_tab_rows > 0) {
    CKM(cudaMemcpyAsync(d_x, xrows, sizeof(double) * n_tab_rows * D2, cudaMemcpyHostToDevice, st));
    CKM(cudaMemcpyAsync(d_z, zrows, sizeof(double) * n_tab_rows * D2, cudaMemcpyHostToDevice, st));
  }
  CKM(keep.alloc(&d_rv, (size_t)nM * D2, true, st));
  CKM(keep.alloc(&d_tie, (size_t)nM, true, st));
  k_bil_rayvalid<<<cdiv((long long)nM * D2 * D2, 256), 256, 0, st>>>(nM, D2, B.L3, d_maps, d_x, d_z, P->d_rank_data, d_rv, d_tie);
  CKM(cudaGetLastError());
  std::vector<uint8_t> rv((size_t)nM * D2);
  std::vector<int> tie(nM);
  CKM(cudaMemcpyAsync(rv.data(), d_rv, rv.size(), cudaMemcpyDeviceToHost, st));
  CKM(cudaMemcpyAsync(tie.data(), d_tie, sizeof(int) * nM, cudaMemcpyDeviceToHost, st));
  CKM(cudaStreamSynchronize(st));
  for (int m = 0; m < nM; ++m) {
    int cnt = 0;
    for (int j = 0; j < D2; ++j) cnt += rv[(size_t)m * D2 + j];
    if (nvalid_rays) nvalid_rays[m] = cnt;
    if (tie_samples) tie_samples[m] = tie[m];
  }
  if (!build_tables) { tmp.free_all(); return HB2_OK; }
  b->h_bil_rv = rv;
  // transposed maps (voxel-driven): count pass, then fill
  const int apitch = P->ntile * HB2_BLOCK;
  // (everything the batch keeps is allocated before the big sort temporaries, so that those nest like a stack in the arena)
  int *d_kmax, *d_fcount, *d_fptr, *d_cursor;
  const int NP = (D2 + 1) / 2;  // forward lists are kept per pair of adjacent rays
  CKM(b->pool.alloc(&d_kmax, 1, true, st));
  CKM(b->pool.alloc(&d_fcount, (size_t)nM * NP + 1, true, st));
  const long long nmp = (long long)nM * P->ndisk;
  k_bil_T<0><<<cdiv(nmp, 128), 128, 0, st>>>(nM, D2, B.L3, P->ndisk, apitch, 0, d_maps, d_x, d_z, P->d_rank_data, P->d_yx_data,
                                             P->d_aslot, nullptr, nullptr, d_kmax, d_fcount);
  CKM(cudaGetLastError());
  int KB = 0;
  CKM(cudaMemcpyAsync(&KB, d_kmax, sizeof(int), cudaMemcpyDeviceToHost, st));
  CKM(cudaStreamSynchronize(st));
  KB = std::max(KB, 1);
  if (KB > 4) { tmp.free_all(); return fail(HB2_ERR_CAPACITY, "more than 4 rays of one view touch one voxel (internal error)"); }
  CKM(b->pool.alloc(&d_fptr, (size_t)nM * NP + 1, false, st));
  uint16_t* d_Tj; float* d_Tw;
  CKM(b->pool.alloc(&d_Tj, (size_t)nM * KB * apitch, false, st));
  CKM(b->pool.alloc(&d_Tw, (size_t)nM * KB * apitch, true, st));
  CKM(cudaMemsetAsync(d_Tj, 0xFF, sizeof(uint16_t) * (size_t)nM * KB * apitch, st));
  size_t sb = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, sb, d_fcount, d_fptr, nM * NP + 1, st);
  void* d_scan; { uint8_t* p; CKM(b->pool.alloc(&p, sb, false, st)); d_scan = p; }
  CKM(cub::DeviceScan::ExclusiveSum(d_scan, sb, d_fcount, d_fptr, nM * NP + 1, st));
  int nent = 0;
  CKM(cudaMemcpyAsync(&nent, d_fptr + (size_t)nM * NP, sizeof(int), cudaMemcpyDeviceToHost, st));
  k_bil_T<1><<<cdiv(nmp, 128), 128, 0, st>>>(nM, D2, B.L3, P->ndisk, apitch, KB, d_maps, d_x, d_z, P->d_rank_data, P->d_yx_data,
                                             P->d_aslot, d_Tj, d_Tw, d_kmax, nullptr);
  CKM(cudaGetLastError());
  CKM(cudaStreamSynchronize(st));
  if (nent < 0) { tmp.free_all(); return fail(HB2_ERR_CAPACITY, "bilinear maps exceed 2^31 entries"); }
  if (content_hash) {
    unsigned long long* d_hash;
    CKM(b->pool.alloc(&d_hash, (size_t)nM, true, st));
    k_bil_hash<<<dim3(cdiv(std::max<long long>((long long)KB * apitch, D2), 256), nM), 256, 0, st>>>(nM, D2, apitch, KB, d_Tj, d_Tw, d_rv, d_hash);
    CKM(cudaGetLastError());
    CKM(cudaMemcpyAsync(content_hash, d_hash, sizeof(unsigned long long) * nM, cudaMemcpyDeviceToHost, st));
    CKM(cudaStreamSynchronize(st));
  }
  // forward lists = the transpose, every ray sorted by voxel rank (deterministic summation order)
  float2* d_Fw; void* d_Fp;
  CKM(b->pool.alloc(&d_Fw, (size_t)std::max(nent, 1), false, st));
  { uint8_t* p; CKM(b->pool.alloc(&p, (size_t)std::max(nent, 1) * (b->idx16 ? 2 : 4), false, st)); d_Fp = p; }
  if (nent > 0) {
    unsigned *d_key, *d_key2; float2* d_val;
    CKM(tmp.alloc(&d_cursor, (size_t)nM * NP, true, st));
    CKM(tmp.alloc(&d_key, (size_t)nent, false, st));
    CKM(tmp.alloc(&d_key2, (size_t)nent, false, st));
    CKM(tmp.alloc(&d_val, (size_t)nent, false, st));
    k_bil_F_fill<<<cdiv(nmp, 128), 128, 0, st>>>(nM, D2, P->ndisk, apitch, KB, P->d_aslot, d_Tj, d_Tw, d_fptr, d_cursor, d_key, d_val);
    CKM(cudaGetLastError());
    size_t sb2 = 0;
    cub::DeviceSegmentedSort::SortPairs(nullptr, sb2, d_key, d_key2, d_val, d_Fw, nent, nM * NP, d_fptr, d_fptr + 1, st);
    void* d_s2; { uint8_t* p; CKM(tmp.alloc(&p, sb2, false, st)); d_s2 = p; }
    CKM(cub::DeviceSegmentedSort::SortPairs(d_s2, sb2, d_key, d_key2, d_val, d_Fw, nent, nM * NP, d_fptr, d_fptr + 1, st));
    if (b->idx16) k_bil_pack<uint16_t><<<cdiv(nent, 256), 256, 0, st>>>(nent, d_key2, (uint16_t*)d_Fp);
    else k_bil_pack<uint32_t><<<cdiv(nent, 256), 256, 0, st>>>(nent, d_key2, (uint32_t*)d_Fp);
    CKM(cudaGetLastError());
  }
  {  // ray window of every (map, voxel tile) for the tile adjoint
    uint16_t *d_jlo, *d_nr; int* d_rmax;
    CKM(b->pool.alloc(&d_jlo, (size_t)nM * P->ntile, false, st));
    CKM(b->pool.alloc(&d_nr, (size_t)nM * P->ntile, false, st));
    CKM(b->pool.alloc(&d_rmax, 1, true, st));
    k_tile_rays<<<dim3(P->ntile, nM), HB2_BLOCK, 0, st>>>(KB, apitch, P->ntile, d_Tj, d_jlo, d_nr, d_rmax);
    CKM(cudaGetLastError());
    int rmax = 0;
    CKM(cudaMemcpyAsync(&rmax, d_rmax, sizeof(int), cudaMemcpyDeviceToHost, st));
    CKM(cudaStreamSynchronize(st));
    B.bil_tile_jlo = d_jlo; B.bil_tile_nr = d_nr; B.bil_rmax = std::max(rmax, 1);
  }
  CKM(cudaStreamSynchronize(st));
  tmp.free_all();
#undef CKM
  b->bilinear = true;
  b->bil_nM = nM;
  B.bil = 1; B.bil_KB = KB;
  B.bilF_p = d_Fp; B.bilF_w = d_Fw; B.bilF_ptr = d_fptr;
  B.bilT_j = d_Tj; B.bilT_w = d_Tw; B.bil_rayvalid = d_rv;
  return HB2_OK;
}

/* ray validity of every bilinear map, out[n_maps*D2] */
extern "C" int hb2_batch_bilinear_ray_valid(hb2_batch* b, uint8_t* out) {
  if (!b || !out || !b->bilinear) return fail(HB2_ERR_ARG, "bad argument or no bilinear maps");
  memcpy(out, b->h_bil_rv.data(), b->h_bil_rv.size());
  return HB2_OK;
}

// Views of a matrix-free trilinear batch, indexed like the views of hb2_batch_create: view_map[v] >= 0 (bilinear view
// of that map) or -1 (pseudo view of the candidate's trilinear symmetry rows); colk[v*ZMP + t], ab[(v*ZMP + t)*2 ..].
extern "C" int hb2_batch_bilinear_views(hb2_batch* b, int32_t nviews, const int32_t* view_map, const int32_t* colk,
                                        const double* ab, int32_t nc, const int32_t* cand_nview) {
  if (!b || nviews <= 0 || !view_map || !colk || !ab || nc <= 0 || !cand_nview) return fail(HB2_ERR_ARG, "bad argument");
  if (!b->bilinear || b->created) return fail(HB2_ERR_STATE, "hb2_batch_bilinear_views: after hb2_batch_bilinear_maps, before hb2_batch_create");
  const int ZMP = b->B.ZMP;
  for (int v = 0; v < nviews; ++v) {
    if (view_map[v] >= b->bil_nM) return fail(HB2_ERR_ARG, "bad map index");
    for (int t = 0; t < ZMP; ++t)
      if (colk[(size_t)v * ZMP + t] >= b->B.L2 || (t >= b->B.L3 && colk[(size_t)v * ZMP + t] >= 0)) return fail(HB2_ERR_ARG, "bad column slot");
  }
  b->h_bil_view_map.assign(view_map, view_map + nviews);
  b->h_bil_colk.assign(colk, colk + (size_t)nviews * ZMP);
  b->h_bil_ab.assign(ab, ab + (size_t)nviews * ZMP * 2);
  b->h_bil_cand_nview.assign(cand_nview, cand_nview + nc);
  return HB2_OK;
}

// Trilinear symmetry rows of candidate c of a matrix-free trilinear batch (same rows as hb2_batch_explicit_sym_rows; call
// for c = 0, 1, ... in order, before hb2_batch_create).  Two passes over the pair rounds: count (insert / check / scan),
// then emit into an exactly sized array; the scratch is shared by the candidates of the batch.
extern "C" int hb2_batch_bilinear_sym_rows(hb2_batch* b, int32_t c, int32_t npairs, const double* pair_mats,
                                           int64_t min_sym_pairs, int64_t* n_rows) {
  if (!b || c < 0 || npairs < 0 || (npairs > 0 && !pair_mats)) return fail(HB2_ERR_ARG, "bad argument");
  if (!b->bilinear || b->created) return fail(HB2_ERR_STATE, "hb2_batch_bilinear_sym_rows: after hb2_batch_bilinear_maps, before hb2_batch_create");
  if (c != (int)b->ls_ent_c.size()) return fail(HB2_ERR_ARG, "candidates must be given in order");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  NvtxRange nvtx_("build_A_helical_sym_matrix - linear");
  if (n_rows) *n_rows = 0;
  b->ls_ent_c.push_back(nullptr);
  b->ls_m_c.push_back(0);
  if (npairs == 0 || min_sym_pairs < 0) return HB2_OK;
  const long long cap_rows = std::min<long long>(min_sym_pairs + B.n, (long long)npairs * B.n);
  if (cap_rows * 16 >= (1ll << 31)) return fail(HB2_ERR_CAPACITY, "too many trilinear symmetry rows");
  hb2_batch::LsScratch& S = b->ls_scr;
  if (cap_rows > S.cap_rows) {  // grow the scratch (the old one stays in the batch's arena until it is destroyed)
    const unsigned long long tc = (unsigned long long)(2 * cap_rows + 17);
    CK(b->pool.alloc(&S.tab_key, (size_t)tc, false, st));
    CK(b->pool.alloc(&S.tab_seq, (size_t)tc, false, st));
    CK(b->pool.alloc(&S.col, (size_t)cap_rows * 16, false, st));
    CK(b->pool.alloc(&S.w, (size_t)cap_rows * 16, false, st));
    S.cap_rows = cap_rows;
    if (!S.tmp_a) {
      CK(b->pool.alloc(&S.tmp_a, (size_t)B.n + 1, false, st));
      CK(b->pool.alloc(&S.tmp_b, (size_t)B.n + 1, false, st));
      CK(b->pool.alloc(&S.flag, (size_t)B.n + 1, true, st));
      CK(b->pool.alloc(&S.pos, (size_t)B.n + 1, true, st));
      CK(b->pool.alloc(&S.ov, 1, true, st));
      cub::DeviceScan::ExclusiveSum(nullptr, S.scan_bytes, S.flag, S.pos, B.n + 1, st);
      { uint8_t* p; CK(b->pool.alloc(&p, S.scan_bytes, false, st)); S.scan_tmp = p; }
      CK(b->pool.alloc(&S.cc, (size_t)B.npad + 2, false, st));
    }
  }
  if (npairs > S.pairs_cap) { CK(b->pool.alloc(&S.pairs, (size_t)npairs, false, st)); S.pairs_cap = npairs; }
  CK(cudaMemcpyAsync(S.pairs, pair_mats, sizeof(LsymPair) * npairs, cudaMemcpyHostToDevice, st));
  LsymSetup Q{};
  Q.n = B.n; Q.ndisk = B.ndisk; Q.D3 = B.D3; Q.L3 = B.L3; Q.L3P = B.L3P;
  Q.rank_sym = P->d_rank_sym; Q.disk_yx_sym = P->d_yx_sym;
  Q.tab_cap = (unsigned long long)(2 * cap_rows + 17);
  Q.tab_key = S.tab_key; Q.tab_seq = S.tab_seq; Q.tmp_a = S.tmp_a; Q.tmp_b = S.tmp_b; Q.flag = S.flag; Q.pos = S.pos;
  Q.overflow = S.ov;
  CK(cudaMemsetAsync(Q.tab_key, 0xFF, sizeof(unsigned long long) * Q.tab_cap, st));
  CK(cudaMemsetAsync(Q.tab_seq, 0xFF, sizeof(unsigned long long) * Q.tab_cap, st));
  CK(cudaMemsetAsync(S.ov, 0, sizeof(int), st));
  long long rows = 0;
  const unsigned gn = cdiv((long long)B.n + 1, 256);
  for (int rnd = 0; rnd < npairs; ++rnd) {
    k_lsym_insert<<<gn, 256, 0, st>>>(Q, S.pairs, rnd);
    k_lsym_check<<<gn, 256, 0, st>>>(Q, rnd);
    CK(cub::DeviceScan::ExclusiveSum(S.scan_tmp, S.scan_bytes, Q.flag, Q.pos, B.n + 1, st));
    k_lsym_emit<<<gn, 256, 0, st>>>(Q, S.pairs, rnd, (int)rows, (int)cap_rows, S.col, S.w);
    CKL();
    int h[2] = {0, 0};
    CK(cudaMemcpyAsync(&h[0], Q.pos + B.n, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h[1], S.ov, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (h[1]) return fail(HB2_ERR_CAPACITY, "trilinear symmetry rows: table overflow");
    rows += h[0];
    if (rows >= min_sym_pairs) break;  // SLR:1286
  }
  if (rows > 0) {
    int2* ent;
    CK(b->pool.alloc(&ent, (size_t)rows * 16, false, st));
    k_ls_pack<<<cdiv(rows * 16, 256), 256, 0, st>>>(rows * 16, S.col, S.w, ent);
    CKL();
    b->ls_ent_c.back() = ent;
  }
  b->ls_m_c.back() = (int)rows;
  if (n_rows) *n_rows = rows;
  return HB2_OK;
}

/* the trilinear symmetry rows of candidate c as 16 (column, weight) entries each, columns in the reference's voxel order */
extern "C" int hb2_batch_bilinear_sym_export(hb2_batch* b, int32_t c, int32_t* cols, float* w) {
  if (!b || !b->bilinear || c < 0 || c >= (int)b->ls_ent_c.size()) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  const size_t ne = (size_t)b->ls_m_c[c] * 16;
  if (ne == 0) return HB2_OK;
  std::vector<int2> ent(ne);
  CK(cudaMemcpyAsync(ent.data(), b->ls_ent_c[c], sizeof(int2) * ne, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  const int L3P = b->B.L3P, nd = b->B.ndisk;
  const std::vector<int>& i2r = b->P->int2ref;
  for (size_t e = 0; e < ne; ++e) {
    if (cols) cols[e] = (ent[e].x % L3P) * nd + i2r[ent[e].x / L3P];
    if (w) memcpy(&w[e], &ent[e].y, 4);
  }
  return HB2_OK;
}

// Called by hb2_batch_create for a matrix-free trilinear batch: uploads the view tables, right-hand side, transpose
// lists of the trilinear symmetry rows.
static int bil_finish(hb2_batch* b, int nviews) {
  hb2_problem* P = b->P;
  cudaStream_t st = b->stream;
  BD& B = b->B;
  const int nc = B.nc;
  if ((int)b->h_bil_view_map.size() != nviews || (int)b->h_bil_cand_nview.size() != nc)
    return fail(HB2_ERR_ARG, "hb2_batch_bilinear_views does not match the views of hb2_batch_create");
  while ((int)b->ls_ent_c.size() < nc) { b->ls_ent_c.push_back(nullptr); b->ls_m_c.push_back(0); }
  for (int c = 0; c < nc; ++c) {
    const int nvw = b->h_bil_cand_nview[c], vc = b->h_view_count[c];
    const long long need = ((long long)b->ls_m_c[c] + B.rows_per_view - 1) / B.rows_per_view;
    if (nvw < 0 || nvw > vc || vc - nvw < need) return fail(HB2_ERR_ARG, "not enough pseudo views for the trilinear symmetry rows");
    for (int v = 0; v < vc; ++v)
      if ((b->h_bil_view_map[b->h_view_begin[c] + v] >= 0) != (v < nvw)) return fail(HB2_ERR_ARG, "bilinear views must come first");
  }
  CK(upload(b->pool, &B.bil_view_map, b->h_bil_view_map, st));
  CK(upload(b->pool, &B.bil_colk, b->h_bil_colk, st));
  CK(upload(b->pool, &B.bil_ab, b->h_bil_ab, st));
  CK(upload(b->pool, &B.bil_cand_nview, b->h_bil_cand_nview, st));
  CK(b->pool.alloc(&B.bil_ub, (size_t)b->u_total, true, st));
  {
    int max_nv = 0;
    for (int c = 0; c < nc; ++c) max_nv = std::max(max_nv, b->h_bil_cand_nview[c]);
    const bool no_tile = getenv("HB2_NO_BIL_TILE") && atoi(getenv("HB2_NO_BIL_TILE"));  // tests compare the tile adjoint with the gather kernel
    B.bil_adj_tile = (!no_tile && max_nv <= HB2_BILT_MAXV) ? 1 : 0;
  }
  k_bil_rhs<<<cdiv((long long)nviews * B.rows_per_view, 256), 256, 0, st>>>(B, P->d_pix, nviews, b->d_bmax);
  CKL();
  // transpose lists of the trilinear symmetry rows, candidate by candidate (stable radix sort of the entries by voxel)
  std::vector<long long> eoff(nc, 0), ceoff(nc, 0);
  std::vector<int2*> cent(nc, nullptr);
  int* d_cptr;
  CK(b->pool.alloc(&d_cptr, (size_t)nc * (B.npad + 1), true, st));
  hb2_batch::LsScratch& S = b->ls_scr;
  long long max_ne = 0;
  for (int c = 0; c < nc; ++c) max_ne = std::max<long long>(max_ne, 16ll * b->ls_m_c[c]);
  if (max_ne > 0) {
    int bits = 1;
    while ((1ll << bits) < (long long)B.npad) ++bits;
    for (int c = 0; c < nc; ++c) CK(b->pool.alloc(&cent[c], (size_t)std::max(16ll * b->ls_m_c[c], 1ll), false, st));
    CK(b->pool.alloc(&S.key, (size_t)max_ne, false, st));
    CK(b->pool.alloc(&S.key2, (size_t)max_ne, false, st));
    CK(b->pool.alloc(&S.id, (size_t)max_ne, false, st));
    CK(b->pool.alloc(&S.id2, (size_t)max_ne, false, st));
    cub::DeviceRadixSort::SortPairs(nullptr, S.sort_bytes, S.key, S.key2, S.id, S.id2, (int)max_ne, 0, bits, st);
    { uint8_t* p; CK(b->pool.alloc(&p, S.sort_bytes, false, st)); S.sort_tmp = p; }
    size_t sbc = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, sbc, S.cc, d_cptr, B.npad + 1, st);
    void* d_sc; { uint8_t* p; CK(b->pool.alloc(&p, sbc, false, st)); d_sc = p; }
    for (int c = 0; c < nc; ++c) {
      const long long ne = 16ll * b->ls_m_c[c];
      if (ne == 0) continue;
      CK(cudaMemsetAsync(S.cc, 0, sizeof(int) * ((size_t)B.npad + 2), st));
      k_ls_keys<<<cdiv(ne, 256), 256, 0, st>>>(ne, b->ls_ent_c[c], S.key, S.id, S.cc);
      size_t sbytes = S.sort_bytes;
      CK(cub::DeviceRadixSort::SortPairs(S.sort_tmp, sbytes, S.key, S.key2, S.id, S.id2, (int)ne, 0, bits, st));
      k_ls_gather<<<cdiv(ne, 256), 256, 0, st>>>(ne, S.id2, b->ls_ent_c[c], cent[c]);
      CK(cub::DeviceScan::ExclusiveSum(d_sc, sbc, S.cc, d_cptr + (size_t)c * (B.npad + 1), B.npad + 1, st));
      CKL();
    }
  }
  const int2* base_e = nullptr; const int2* base_c = nullptr;
  for (int c = 0; c < nc; ++c) {
    if (b->ls_m_c[c] == 0) continue;
    if (!base_e) { base_e = b->ls_ent_c[c]; base_c = cent[c]; }
    eoff[c] = ((intptr_t)b->ls_ent_c[c] - (intptr_t)base_e) / (intptr_t)sizeof(int2);
    ceoff[c] = ((intptr_t)cent[c] - (intptr_t)base_c) / (intptr_t)sizeof(int2);
  }
  B.ls_ent = base_e; B.ls_cent = base_c; B.ls_cptr = d_cptr;
  CK(upload(b->pool, &B.ls_eoff, eoff, st));
  CK(upload(b->pool, &B.ls_ceoff, ceoff, st));
  CK(upload(b->pool, &B.ls_m, b->ls_m_c, st));
  CK(cudaStreamSynchronize(st));
  return HB2_OK;
}

extern "C" int hb2_batch_set_ties(hb2_batch* b, int32_t n_tie, int32_t TS, const int8_t* zlo, const uint8_t* up,
                                  const uint8_t* rowvalid) {
  if (!b || n_tie < 0 || (n_tie > 0 && (!zlo || !up || !rowvalid || TS <= 0))) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "hb2_batch_set_ties must precede hb2_batch_create");
  const int D2 = b->B.D2;
  b->n_tie = n_tie; b->tie_TS = TS;
  b->h_tie_zlo.assign(zlo, zlo + (size_t)n_tie * TS);
  b->h_tie_up.assign(up, up + (size_t)n_tie * TS * D2);
  b->h_tie_rv.assign(rowvalid, rowvalid + (size_t)n_tie * TS * D2);
  return HB2_OK;
}

// Band tables of the forward band path for one element size (hb2_fwd_band.cuh).  Bands = contiguous runs of the
// band-column-major voxel order: whole 16-row bands of the disk merged while they fit ~200 KB of shared memory, a band
// that does not fit is cut at column boundaries (multiples of 16 ranks).  Partial rows are compact: view_poff[view] +
// band_off[angle][band] + (j - jlo).  On any limit (too many bands) the table stays empty and the gather kernel runs.
static int build_band_tab(hb2_batch* b, size_t elem, BandTab& out, size_t& smem_out) {
  BD& B = b->B;
  hb2_problem* P = b->P;
  cudaStream_t st = b->stream;
  const int D2 = B.D2;
  out = BandTab{};
  const long long cap = (long long)(200 * 1024) / (B.L3P * (long long)elem);
  const long long cap16 = cap / 16 * 16;
  if (cap16 < 16) return HB2_OK;
  std::vector<int> bands{0};
  const std::vector<int>& tr = P->h_tilerow_begin;
  for (size_t r = 0; r + 1 < tr.size(); ++r) {
    const int lo = tr[r], hi = tr[r + 1];
    if (hi - bands.back() <= cap) continue;            // the 16-row band joins the open band
    if (lo > bands.back()) bands.push_back(lo);        // close the open band in front of it
    while (hi - bands.back() > cap) bands.push_back(bands.back() + (int)cap16);  // cut at column boundaries
  }
  bands.push_back(B.ndisk);
  const int NB = (int)bands.size() - 1;
  if (NB > HB2_MAX_BANDS) return HB2_OK;
  int max_bn = 0;
  for (int q = 0; q < NB; ++q) max_bn = std::max(max_bn, bands[q + 1] - bands[q]);
  smem_out = (size_t)max_bn * B.L3P * elem;
#define CKB2(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)
  CKB2(upload(b->pool, &out.band_begin, bands, st));
  ushort2 *d_seg, *d_rng;
  CKB2(b->pool.alloc(&d_seg, (size_t)B.nA * NB * D2, false, st));
  CKB2(b->pool.alloc(&d_rng, (size_t)B.nA * NB, false, st));
  const long long nt = (long long)B.nA * NB * D2;
  k_band_segs<uint16_t><<<cdiv(nt, 256), 256, 0, st>>>(B.nA, NB, D2, out.band_begin, (const uint16_t*)b->d_fmap, d_seg);
  k_band_rng<<<dim3(NB, B.nA), HB2_BLOCK, 0, st>>>(NB, D2, d_seg, d_rng);
  CKB2(cudaGetLastError());
  std::vector<ushort2> h_rng((size_t)B.nA * NB);
  CKB2(cudaMemcpyAsync(h_rng.data(), d_rng, sizeof(ushort2) * h_rng.size(), cudaMemcpyDeviceToHost, st));
  CKB2(cudaStreamSynchronize(st));
  std::vector<int> band_off((size_t)B.nA * NB), rows_of_angle(B.nA, 0);
  for (int a = 0; a < B.nA; ++a) {
    int acc = 0;
    for (int q = 0; q < NB; ++q) {
      band_off[(size_t)a * NB + q] = acc;
      acc += (int)h_rng[(size_t)a * NB + q].y - (int)h_rng[(size_t)a * NB + q].x;
    }
    rows_of_angle[a] = acc;
  }
  const int nviews = (int)b->h_view_angle.size();
  std::vector<long long> view_poff(std::max(nviews, 1), 0);
  long long total = 0;
  for (int v = 0; v < nviews; ++v) { view_poff[v] = total; total += rows_of_angle[b->h_view_angle[v]]; }
  CKB2(upload(b->pool, &out.band_off, band_off, st));
  CKB2(upload(b->pool, &out.view_poff, view_poff, st));
  uint8_t* part;
  CKB2(b->pool.alloc(&part, (size_t)std::max<long long>(total, 1) * B.L3P * elem, false, st));
#undef CKB2
  out.part = part; out.seg = d_seg; out.rng = d_rng; out.nband = NB;
  return HB2_OK;
}

extern "C" int hb2_batch_create(hb2_batch* b, int32_t nc, const hb2_candidate* cands, int32_t nviews, const hb2_view* views,
                                int32_t ncolk, const int32_t* colk, int32_t npairs, const hb2_pair* pairs) {
  if (!b || !cands || nc <= 0 || !views || nviews <= 0 || !colk) return fail(HB2_ERR_ARG, "bad argument");
  if (b->created) return fail(HB2_ERR_STATE, "batch already created");
  if (nc > 65535) return fail(HB2_ERR_ARG, "at most 65535 candidates per batch");
  NvtxRange nvtx_("build_A_data_matrix + build_A_helical_sym_matrix (batch)");
  hb2_problem* P = b->P;
  CK(cudaSetDevice(P->device));
  cudaStream_t st = b->stream;
  BD& B = b->B;
  B.nc = nc;
  b->nviews = nviews;
  b->cands.assign(cands, cands + nc);
  const int D2 = B.D2, ntiles = (D2 + HB2_TILE_RAYS - 1) / HB2_TILE_RAYS;
  // ---- host tables ---------------------------------------------------------
  std::vector<int> view_cand(nviews, -1), view_angle(nviews), view_colbegin(nviews), view_tie(nviews, -1), view_tie_slot0(nviews, 0);
  std::vector<int> tie_views, cand_tie_begin(nc, 0), cand_tie_count(nc, 0);
  std::vector<int> view_dupof(nviews, -1), view_mult(nviews, 1), view_dups((size_t)nviews * HB2_MAXDUP, -1);
  std::vector<long long> view_uoff(nviews);
  b->h_view_begin.resize(nc); b->h_view_count.resize(nc); b->h_mdata.resize(nc); b->h_msym.assign(nc, 0);
  b->h_uoff.resize(nc); b->h_symoff.resize(nc); b->h_symcap.resize(nc); b->h_cscoff.resize(nc);
  b->cand_flags.assign(nc, 0);
  std::vector<int> pair_begin(nc), pair_count(nc);
  std::vector<long long> min_pairs(nc), tab_off(nc), tab_cap(nc);
  long long uo = 0, so = 0, to = 0;
  int expect_view = 0;
  for (int c = 0; c < nc; ++c) {
    const hb2_candidate& q = cands[c];
    if (q.view_begin != expect_view || q.view_count < 0 || q.view_begin + q.view_count > nviews)
      return fail(HB2_ERR_ARG, "candidate views must tile the view array in order");
    expect_view += q.view_count;
    if (q.pair_count < 0 || q.pair_begin < 0 || q.pair_begin + q.pair_count > npairs) return fail(HB2_ERR_ARG, "bad pair range");
    b->h_view_begin[c] = q.view_begin; b->h_view_count[c] = q.view_count;
    long long md = (long long)q.view_count * B.rows_per_view;
    if (md >= (1ll << 31)) return fail(HB2_ERR_GEOMETRY, "too many data rows in one candidate");
    b->h_mdata[c] = (int)md;
    long long cap = std::min<long long>(q.min_sym_pairs + B.n, (long long)q.pair_count * B.n);
    if (q.pair_count == 0 || q.min_sym_pairs < 0) cap = 0;
    cap = (cap + 3) / 4 * 4;  // keeps every candidate's rows 16-byte aligned
    if (cap >= (1ll << 31) - 1) return fail(HB2_ERR_GEOMETRY, "too many symmetry rows in one candidate");
    b->h_symcap[c] = cap;
    b->h_uoff[c] = uo; b->h_symoff[c] = so; b->h_cscoff[c] = 2 * so;
    for (int v = 0; v < q.view_count; ++v) {
      int vi = q.view_begin + v;
      const hb2_view& w = views[vi];
      if (w.angle < 0 || w.angle >= B.nA || w.col_begin < 0 || w.col_begin + B.ZMC > ncolk) return fail(HB2_ERR_ARG, "bad view");
      view_cand[vi] = c; view_angle[vi] = w.angle; view_colbegin[vi] = w.col_begin;
      static const bool no_dedupe = getenv("HB2_NO_DEDUPE") && atoi(getenv("HB2_NO_DEDUPE"));
      if (w.dup_of >= 0 && (w.tie < 0 || b->bilinear) && !no_dedupe) {  // duplicate of an earlier regular view of the same candidate
        const int prim = q.view_begin + w.dup_of;
        if (w.dup_of >= v || views[prim].angle != w.angle || (views[prim].tie >= 0 && !b->bilinear) || views[prim].dup_of >= 0)
          return fail(HB2_ERR_ARG, "bad duplicate view");
        int slot = 0;
        while (slot < HB2_MAXDUP && view_dups[(size_t)prim * HB2_MAXDUP + slot] >= 0) ++slot;
        if (slot < HB2_MAXDUP) {  // more than HB2_MAXDUP duplicates: the extra ones are computed on their own
          view_dups[(size_t)prim * HB2_MAXDUP + slot] = vi;
          view_dupof[vi] = prim; view_mult[vi] = 0; view_mult[prim] += 1;
        }
      }
      if ((b->explicit_rows || b->bilinear) && w.tie < 0) return fail(HB2_ERR_ARG, "a batch with explicit / trilinear rows takes pseudo views only");
      if (w.tie >= 0) {
        if (!b->explicit_rows && !b->bilinear) {
          if (w.tie >= b->n_tie || w.tie_slot0 < 0 || w.tie_slot0 + B.ZMC > b->tie_TS) return fail(HB2_ERR_ARG, "bad tie view");
          if (B.ZMC > HB2_TIE_MAXZMC) return fail(HB2_ERR_GEOMETRY, "tie views need L3*MC <= 16");
        }
        view_tie[vi] = w.tie; view_tie_slot0[vi] = w.tie_slot0;
        if (cand_tie_count[c] == 0) cand_tie_begin[c] = (int)tie_views.size();
        tie_views.push_back(vi);
        cand_tie_count[c] += 1;
      }
      view_uoff[vi] = uo + (long long)v * B.rows_per_view;
      if (b->tie_per_angle[w.angle] > 0 && !b->explicit_rows && !b->bilinear) b->cand_flags[c] |= HB2_FLAG_TIE_XY;
    }
    b->cand_flags[c] |= q.flags_in;
    if (q.view_count == 0) b->cand_flags[c] |= HB2_FLAG_NO_ROWS;
    uo += md + cap; so += cap;
    pair_begin[c] = q.pair_begin; pair_count[c] = q.pair_count; min_pairs[c] = q.min_sym_pairs;
    tab_off[c] = to; tab_cap[c] = 2 * cap + 17; to += tab_cap[c];
  }
  if (expect_view != nviews) return fail(HB2_ERR_ARG, "views not fully assigned to candidates");
  if (2 * so >= (1ll << 31)) return fail(HB2_ERR_CAPACITY, "batch too large: symmetry-row lists exceed 2^31 entries; use smaller batches");
  if ((long long)nc * (B.npad + 1) >= (1ll << 31) || (long long)nc * B.nrp >= (1ll << 31))
    return fail(HB2_ERR_CAPACITY, "batch too large: nc*n exceeds 2^31; use smaller batches");
  b->u_total = uo;
  b->h_view_angle = view_angle;
  for (int e = 0; e < ncolk; ++e)
    if (colk[e] >= B.L2) return fail(HB2_ERR_ARG, "column index out of range");
#define CKC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
  // ---- device tables -------------------------------------------------------
  CKC(upload(b->pool, &B.view_cand, view_cand, st));
  CKC(upload(b->pool, &B.view_angle, view_angle, st));
  CKC(upload(b->pool, &B.view_colbegin, view_colbegin, st));
  CKC(upload(b->pool, &B.view_dupof, view_dupof, st));
  CKC(upload(b->pool, &B.view_mult, view_mult, st));
  CKC(upload(b->pool, &B.view_dups, view_dups, st));
  b->n_tie_views = (int)tie_views.size();
  B.n_tie_views = b->n_tie_views; B.tie_TS = b->tie_TS;
  CKC(upload(b->pool, &B.cand_tie_begin, cand_tie_begin, st));
  CKC(upload(b->pool, &B.cand_tie_count, cand_tie_count, st));
  if (b->n_tie_views > 0) {
    CKC(upload(b->pool, &B.view_tie, view_tie, st));
    CKC(upload(b->pool, &B.view_tie_slot0, view_tie_slot0, st));
    CKC(upload(b->pool, &B.tie_views, tie_views, st));
    CKC(upload(b->pool, (const int8_t**)&B.tie_zlo, b->h_tie_zlo, st));
    CKC(upload(b->pool, &B.tie_up, b->h_tie_up, st));
    B.tie_upmask = nullptr;
    if (!b->explicit_rows && b->n_tie > 0 && b->tie_TS % B.ZMC == 0 && B.ZMC <= 16) {
      uint16_t* d_mask;
      const long long nm = (long long)b->n_tie * (b->tie_TS / B.ZMC) * D2;
      CKC(b->pool.alloc(&d_mask, (size_t)nm, false, st));
      k_tie_pack<<<cdiv(nm, 256), 256, 0, st>>>(b->n_tie, b->tie_TS, B.ZMC, D2, B.tie_up, d_mask);
      B.tie_upmask = d_mask;
      b->want_tie_info = true;  // filled once colk is on the device (below)
    }
    CKC(upload(b->pool, &B.tie_rowvalid, b->h_tie_rv, st));
  }
  CKC(upload(b->pool, &B.view_uoff, view_uoff, st));
  std::vector<int> colk_v(colk, colk + ncolk);
  CKC(upload(b->pool, &B.colk, colk_v, st));
  B.tie_info = nullptr;
  if (b->want_tie_info && b->n_tie_views > 0) {
    int* d_info;
    CKC(b->pool.alloc(&d_info, (size_t)nviews, true, st));
    k_tie_info<<<cdiv(b->n_tie_views, 128), 128, 0, st>>>(b->n_tie_views, B.tie_views, B.ZMC, b->tie_TS, B.view_tie, B.view_tie_slot0,
                                                        B.view_colbegin, B.colk, B.tie_zlo, d_info);
    B.tie_info = d_info;
  }
  CKC(upload(b->pool, &B.cand_view_begin, b->h_view_begin, st));
  CKC(upload(b->pool, &B.cand_view_count, b->h_view_count, st));
  CKC(upload(b->pool, &B.cand_uoff, b->h_uoff, st));
  CKC(upload(b->pool, &B.cand_mdata, b->h_mdata, st));
  CKC(upload(b->pool, &B.cand_symoff, b->h_symoff, st));
  CKC(upload(b->pool, &B.cand_cscoff, b->h_cscoff, st));
  CKC(b->pool.alloc(&B.cand_msym, nc, true, st));
  {  // depth-sample range of every ray (all maps incl. the exact per-column ones are final here)
    ushort2* rr;
    CKC(b->pool.alloc(&rr, (size_t)B.nA * B.D2, false, st));
    const unsigned gr = cdiv((long long)B.nA * B.D2 * 32, HB2_BLOCK);
    if (b->idx16) k_ray_range<uint16_t><<<gr, HB2_BLOCK, 0, st>>>(B.nA, B.D2, (const uint16_t*)B.fmap, rr);
    else k_ray_range<uint32_t><<<gr, HB2_BLOCK, 0, st>>>(B.nA, B.D2, (const uint32_t*)B.fmap, rr);
    B.rayrange = rr;
  }
  // ---- adjoint maps --------------------------------------------------------
  {
    int* d_kmax; unsigned long long *d_h1, *d_h2;
    CKC(b->pool.alloc(&d_kmax, 1, true, st));
    CKC(b->pool.alloc(&d_h1, B.nA, true, st));
    CKC(b->pool.alloc(&d_h2, B.nA, true, st));
    B.apitch = P->tile_ok ? P->ntile * HB2_BLOCK : 0;
    B.aslot = P->d_aslot; B.tile_begin = P->d_tile_begin; B.ntile = P->ntile;
    if (!P->tile_ok) return fail(HB2_ERR_GEOMETRY, "HB2_TILE_H*HB2_TILE_W must be <= 256");
    long long na = (long long)B.nA * B.ndisk;
    if (b->idx16) k_build_amap<uint16_t><<<cdiv(na, 256), 256, 0, st>>>(B.nA, D2, B.ndisk, B.apitch, B.s, 0, 0, b->d_cs, P->d_yx_data, P->d_aslot, (const uint16_t*)b->d_fmap, nullptr, d_kmax, nullptr);
    else k_build_amap<uint32_t><<<cdiv(na, 256), 256, 0, st>>>(B.nA, D2, B.ndisk, B.apitch, B.s, 0, 0, b->d_cs, P->d_yx_data, P->d_aslot, (const uint32_t*)b->d_fmap, nullptr, d_kmax, nullptr);
    CKL();
    int K = 0;
    CKC(cudaMemcpyAsync(&K, d_kmax, sizeof(int), cudaMemcpyDeviceToHost, st));
    CKC(cudaStreamSynchronize(st));
    if (K < 1) K = 1;
    if (K > 64) return fail(HB2_ERR_CAPACITY, "more than 64 samples of one view land in one voxel (scale2d_to_3d too small)");
    B.K = K;
    CKC(b->pool.alloc(&b->d_amap, (size_t)B.nA * K * B.apitch, false, st));
    CKC(cudaMemsetAsync(b->d_amap, 0xFF, (size_t)B.nA * K * B.apitch * sizeof(uint16_t), st));
    if (b->n_tie_views > 0) {  // the tie adjoint needs the depth sample of every map entry
      CKC(b->pool.alloc(&b->d_amap_i, (size_t)B.nA * K * B.apitch, false, st));
      CKC(cudaMemsetAsync(b->d_amap_i, 0, (size_t)B.nA * K * B.apitch * sizeof(uint16_t), st));
      B.amap_i = b->d_amap_i;
    }
    if (b->idx16) k_build_amap<uint16_t><<<cdiv(na, 256), 256, 0, st>>>(B.nA, D2, B.ndisk, B.apitch, B.s, K, 1, b->d_cs, P->d_yx_data, P->d_aslot, (const uint16_t*)b->d_fmap, b->d_amap, d_kmax, b->d_amap_i);
    else k_build_amap<uint32_t><<<cdiv(na, 256), 256, 0, st>>>(B.nA, D2, B.ndisk, B.apitch, B.s, K, 1, b->d_cs, P->d_yx_data, P->d_aslot, (const uint32_t*)b->d_fmap, b->d_amap, d_kmax, b->d_amap_i);
    CKL();
    // consistency: every hit of the forward map must appear in the adjoint map
    if (b->idx16) k_count_hits<uint16_t><<<dim3(cdiv((long long)D2 * D2, 256), B.nA), 256, 0, st>>>(B.nA, D2, (const uint16_t*)b->d_fmap, d_h1);
    else k_count_hits<uint32_t><<<dim3(cdiv((long long)D2 * D2, 256), B.nA), 256, 0, st>>>(B.nA, D2, (const uint32_t*)b->d_fmap, d_h1);
    k_count_amap<<<dim3(cdiv((long long)K * B.apitch, 256), B.nA), 256, 0, st>>>(B.nA, K, B.apitch, b->d_amap, d_h2);
    CKL();
    std::vector<unsigned long long> h1(B.nA), h2(B.nA);
    CKC(cudaMemcpyAsync(h1.data(), d_h1, 8 * B.nA, cudaMemcpyDeviceToHost, st));
    CKC(cudaMemcpyAsync(h2.data(), d_h2, 8 * B.nA, cudaMemcpyDeviceToHost, st));
    CKC(cudaStreamSynchronize(st));
    for (int a = 0; a < B.nA; ++a)
      if (h1[a] != h2[a]) return fail(HB2_ERR_CAPACITY, "adjoint map does not cover the forward map (internal error)");
    B.amap = b->d_amap;
    {  // ray window of every (angle, tile) for the tile adjoint
      uint16_t *d_jlo, *d_nr; int* d_rmax;
      CKC(b->pool.alloc(&d_jlo, (size_t)B.nA * B.ntile, false, st));
      CKC(b->pool.alloc(&d_nr, (size_t)B.nA * B.ntile, false, st));
      CKC(b->pool.alloc(&d_rmax, 1, true, st));
      k_tile_rays<<<dim3(B.ntile, B.nA), HB2_BLOCK, 0, st>>>(K, B.apitch, B.ntile, b->d_amap, d_jlo, d_nr, d_rmax);
      CKL();
      int rmax = 0;
      CKC(cudaMemcpyAsync(&rmax, d_rmax, sizeof(int), cudaMemcpyDeviceToHost, st));
      CKC(cudaStreamSynchronize(st));
      B.tile_jlo = d_jlo; B.tile_nr = d_nr; B.rmax = std::max(rmax, 1);
      b->pool.release(d_rmax);
    }
    b->pool.release(d_kmax); b->pool.release(d_h1); b->pool.release(d_h2);
  }
  // ---- vectors -----------------------------------------------------------------
  size_t nv = (size_t)nc * B.npad;
  CKC(b->pool.alloc(&B.u, (size_t)uo, true, st));
  CKC(b->pool.alloc(&B.b, (size_t)uo, true, st));
  CKC(b->pool.alloc(&B.v, nv, true, st));
  CKC(b->pool.alloc(&B.h, nv, true, st));
  CKC(b->pool.alloc(&B.xs, nv, true, st));
  CKC(b->pool.alloc(&B.x, nv, true, st));
  CKC(b->pool.alloc(&B.hbar, nv, true, st));
  if (b->n_tie_views > 0) CKC(b->pool.alloc(&B.vtie, nv, true, st));
  CKC(b->pool.alloc(&B.st, nc, true, st));
  CKC(b->pool.alloc(&b->d_bmax, nc, false, st));
  CKC(b->pool.alloc(&b->d_score, nc, true, st));
  CKC(b->pool.alloc(&b->d_chain, (size_t)2 * nc, true, st));
  CKC(b->pool.alloc(&b->d_nactive, 1, true, st));
  CKC(cudaMallocHost(&b->h_nactive, sizeof(int)));
  {
    std::vector<int> neg(nc, (int)0x80000000);  // ordered-int encoding of -inf-ish
    CKC(cudaMemcpyAsync(b->d_bmax, neg.data(), sizeof(int) * nc, cudaMemcpyHostToDevice, st));
    CKC(cudaStreamSynchronize(st));
  }
  // partial-sum buffers
  B.part_u_n = nviews * ntiles;
  int max_symcap = 0;
  for (int c = 0; c < nc; ++c) max_symcap = std::max<long long>(max_symcap, b->h_symcap[c]);
  B.part_us_per_cand = std::max(1u, cdiv(max_symcap, HB2_BLOCK * 4));
  {
    long long max_md = 0;
    for (int c = 0; c < nc; ++c) max_md = std::max<long long>(max_md, b->h_mdata[c]);
    B.adj_fast = (B.MC == 1 && B.K <= 2 && max_md + (long long)B.ZMP * B.D2 < (1ll << 32)) ? 1 : 0;
    int max_views = 0;
    for (int c = 0; c < nc; ++c) max_views = std::max(max_views, b->h_view_count[c]);
    b->adj_tile_smem = (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.K * HB2_BLOCK * sizeof(uint16_t) +
                       (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.rmax * B.L3P * sizeof(float);
    const char* no_tile = getenv("HB2_NO_ADJ_TILE");
    B.adj_tile = (B.adj_fast && B.L3P <= 16 && max_views <= HB2_ADJT_MAXV && b->adj_tile_smem <= 96 * 1024 &&
                  !(no_tile && atoi(no_tile))) ? 1 : 0;
    b->adj_chunks = 1;
    // More than 16 slices: the tile adjoint in chunks of 16 slices (grid.z), one 64-byte piece per ray row.  Measured
    // (profiles/r1_summary.md section 7) 35 % SLOWER than the (voxel, quad) fallback at L3 = 44...104 -- ~40 small bulk
    // copies per view and chunk instead of one -- so it is opt-in (HB2_ADJ_CHUNKED=1).
    static const bool use_chunked = getenv("HB2_ADJ_CHUNKED") && atoi(getenv("HB2_ADJ_CHUNKED"));
    if (use_chunked && !B.adj_tile && B.adj_fast && B.L3P > 16 && max_views <= HB2_ADJT_MAXV) {
      const size_t sm = (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.K * HB2_BLOCK * sizeof(uint16_t) +
                        (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.rmax * 16 * sizeof(float);
      if (sm <= 160 * 1024) { B.adj_tile = 2; b->adj_tile_smem = sm; b->adj_chunks = (B.L3P + 15) / 16; }
    }
    B.part_v_per_cand = B.adj_tile ? B.ntile * b->adj_chunks : cdiv((long long)B.ndisk * (B.L3P / 4), HB2_BLOCK);
  }
  B.part_x_per_cand = cdiv(B.npad, HB2_BLOCK * 4);
  // ---- forward band path: bands that fit shared memory, ray segments per (angle, band), compact partial rows -------
  B.fwd_band = 0; B.fwd_ppv = ntiles; B.bt32 = BandTab{}; B.bt64 = BandTab{};
  {
    int max_views = 0;
    for (int c = 0; c < nc; ++c) max_views = std::max(max_views, b->h_view_count[c]);
    b->max_views = max_views;
    // Default whenever it applies (one column slot per slice, <= 16 slices, 16-bit maps); HB2_FWD_BAND=0 forces the
    // gather kernels (tests compare the two), HB2_FWD_BAND=1 keeps the float64 operator of the bounded branch on them.
    const char* use_band = getenv("HB2_FWD_BAND");
    const int band_mode = use_band ? atoi(use_band) : 2;
    const bool ok = B.MC == 1 && B.L3P <= 16 && max_views <= HB2_FWDB_MAXV && band_mode > 0 && b->idx16 && D2 % 8 == 0 &&
                    !b->explicit_rows && !b->bilinear;
    bool any_positive = false;
    for (int c = 0; c < nc; ++c) any_positive = any_positive || cands[c].positive != 0;
    if (ok) {
      int rc = build_band_tab(b, sizeof(float), B.bt32, b->fwd_band_smem);
      if (rc != HB2_OK) { b->pool.free_all(); return rc; }
      if (B.bt32.nband > 0) { B.fwd_band = 1; B.fwd_ppv = 1; }
      if (B.fwd_band && band_mode > 1 && any_positive) {
        rc = build_band_tab(b, sizeof(double), B.bt64, b->fwd_band_smem64);
        if (rc != HB2_OK) { b->pool.free_all(); return rc; }
      }
    }
  }
  CKC(b->pool.alloc(&B.part_u, (size_t)B.part_u_n, true, st));
  CKC(b->pool.alloc(&B.part_us, (size_t)nc * B.part_us_per_cand, true, st));
  CKC(b->pool.alloc(&B.part_v, (size_t)nc * B.part_v_per_cand, true, st));
  CKC(b->pool.alloc(&B.part_x, (size_t)nc * B.part_x_per_cand, true, st));
  CKC(b->pool.alloc(&B.part_s, (size_t)3 * B.part_u_n, true, st));
  // ---- right-hand side ---------------------------------------------------------
  k_build_rhs<<<cdiv((long long)nviews * B.rows_per_view, 256), 256, 0, st>>>(B, P->d_pix, nviews, b->d_bmax);
  CKL();
  if (b->explicit_rows) {  // the explicit rows bring their own right-hand side (pseudo views have no columns)
    { int rc_ = exp_finish(b); if (rc_ != HB2_OK) return rc_; }
    if (nc != 1) return fail(HB2_ERR_ARG, "a batch with explicit rows holds one candidate");
    if ((long long)B.exp_m > b->h_mdata[0]) return fail(HB2_ERR_ARG, "not enough pseudo views for the explicit rows");
    CKC(cudaMemcpyAsync(B.b + b->h_uoff[0], b->d_exp_b, sizeof(float) * B.exp_m, cudaMemcpyDeviceToDevice, st));
    int iv;
    memcpy(&iv, &b->exp_bmax, sizeof(int));
    iv = iv >= 0 ? iv : iv ^ 0x7fffffff;
    CKC(cudaMemcpyAsync(b->d_bmax, &iv, sizeof(int), cudaMemcpyHostToDevice, st));
    CKC(cudaStreamSynchronize(st));
  }
  if (b->bilinear) {  // matrix-free trilinear rows: view tables, right-hand side, symmetry-row transposes
    int rc_ = bil_finish(b, nviews);
    if (rc_ != HB2_OK) return rc_;
  }
  // ---- symmetry rows -----------------------------------------------------------
  NvtxRange nvtx_sym_("build_A_helical_sym_matrix - nn");
  CKC(b->pool.alloc(&b->d_sym_a, (size_t)so, false, st));
  CKC(b->pool.alloc(&b->d_sym_b, (size_t)so, false, st));
  CKC(b->pool.alloc(&b->d_sym_g, (size_t)so, false, st));
  B.sym_a = b->d_sym_a; B.sym_b = b->d_sym_b;
  CKC(b->pool.alloc(&b->d_csc_ptr, (size_t)nc * (B.npad + 1), true, st));
  CKC(b->pool.alloc(&b->d_csc_ent, (size_t)2 * so, false, st));
  B.csc_ptr = b->d_csc_ptr; B.csc_ent = b->d_csc_ent;
  int max_rounds = 0;
  for (int c = 0; c < nc; ++c) if (b->h_symcap[c] > 0) max_rounds = std::max(max_rounds, pair_count[c]);
  if (max_rounds > 0 && so > 0) {
    SymSetup Q{};
    std::vector<double> pr((size_t)npairs * 6);
    for (int i = 0; i < npairs; ++i) {
      pr[6 * i] = pairs[i].ci; pr[6 * i + 1] = pairs[i].si; pr[6 * i + 2] = pairs[i].zi;
      pr[6 * i + 3] = pairs[i].cj; pr[6 * i + 4] = pairs[i].sj; pr[6 * i + 5] = pairs[i].zj;
    }
    DevPool tmp;
    tmp.owner = b;
#define CKT(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { tmp.free_all(); return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
    CKT(upload(tmp, &Q.pairs, pr, st));
    CKT(upload(tmp, &Q.pair_begin, pair_begin, st));
    CKT(upload(tmp, &Q.pair_count, pair_count, st));
    CKT(upload(tmp, &Q.min_pairs, min_pairs, st));
    CKT(upload(tmp, &Q.tab_off, tab_off, st));
    CKT(upload(tmp, &Q.tab_cap, tab_cap, st));
    CKT(upload(tmp, &Q.symcap, b->h_symcap, st));
    CKT(tmp.alloc(&Q.tab_key, (size_t)to, false, st));
    CKT(tmp.alloc(&Q.tab_seq, (size_t)to, false, st));
    CKT(cudaMemsetAsync(Q.tab_key, 0xFF, (size_t)to * 8, st));
    CKT(cudaMemsetAsync(Q.tab_seq, 0xFF, (size_t)to * 8, st));
    const size_t nr = (size_t)nc * B.nrp;
    CKT(tmp.alloc(&Q.tmp_a, nr, false, st));
    CKT(tmp.alloc(&Q.tmp_b, nr, false, st));
    CKT(tmp.alloc(&Q.flag, nr, true, st));
    CKT(tmp.alloc(&Q.pos, nr, true, st));
    CKT(tmp.alloc(&Q.done, nc, false, st));
    CKT(tmp.alloc(&Q.ndone, 1, true, st));
    CKT(tmp.alloc(&Q.overflow, 1, true, st));
    {
      std::vector<int> done0(nc);
      int nd0 = 0;
      for (int c = 0; c < nc; ++c) { done0[c] = b->h_symcap[c] == 0; nd0 += done0[c]; }
      CKT(cudaMemcpyAsync(Q.done, done0.data(), sizeof(int) * nc, cudaMemcpyHostToDevice, st));
      CKT(cudaMemcpyAsync(Q.ndone, &nd0, sizeof(int), cudaMemcpyHostToDevice, st));
      CKT(cudaStreamSynchronize(st));
    }
    Q.sym_a_w = b->d_sym_a; Q.sym_b_w = b->d_sym_b; Q.sym_g_w = b->d_sym_g;
    Q.rank_sym = P->d_rank_sym; Q.disk_yx_sym = P->d_yx_sym; Q.int2ref = P->d_int2ref;
    b->h_sym_round_end.clear();
    void* d_scan_tmp = nullptr; size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, Q.flag, Q.pos, (int)nr, st);
    { char* p; CKT(tmp.alloc(&p, scan_bytes, false, st)); d_scan_tmp = p; }
    dim3 gn(cdiv(B.n, 256), nc), gp(cdiv(B.nrp, 256), nc);
    for (int rnd = 0; rnd < max_rounds; ++rnd) {
      k_sym_insert<<<gn, 256, 0, st>>>(B, Q, rnd);
      k_sym_check<<<gp, 256, 0, st>>>(B, Q, rnd);
      CKT(cub::DeviceScan::ExclusiveSum(d_scan_tmp, scan_bytes, Q.flag, Q.pos, (int)nr, st));
      k_sym_compact<<<gn, 256, 0, st>>>(B, Q);
      k_sym_finalize<<<cdiv(nc, 128), 128, 0, st>>>(B, Q, rnd);
      CKT(cudaGetLastError());
      int nd = 0, ovf = 0;
      CKT(cudaMemcpyAsync(&nd, Q.ndone, sizeof(int), cudaMemcpyDeviceToHost, st));
      CKT(cudaMemcpyAsync(&ovf, Q.overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
      b->h_sym_round_end.emplace_back(nc);
      CKT(cudaMemcpyAsync(b->h_sym_round_end.back().data(), B.cand_msym, sizeof(int) * nc, cudaMemcpyDeviceToHost, st));
      CKT(cudaStreamSynchronize(st));
      if (ovf) { tmp.free_all(); return fail(HB2_ERR_CAPACITY, "symmetry-row table overflow (internal error)"); }
      if (nd >= nc) break;
    }
    CKT(cudaMemcpyAsync(b->h_msym.data(), B.cand_msym, sizeof(int) * nc, cudaMemcpyDeviceToHost, st));
    CKT(cudaStreamSynchronize(st));
    // transpose lists
    int max_m = 0;
    for (int c = 0; c < nc; ++c) max_m = std::max(max_m, b->h_msym[c]);
    if (max_m > 0) {
      size_t np1 = (size_t)nc * (B.npad + 1);
      int *d_cnt, *d_scan;
      CKT(tmp.alloc(&d_cnt, np1, true, st));
      CKT(tmp.alloc(&d_scan, np1, false, st));
      dim3 gr(cdiv(max_m, 256), nc), gq(cdiv(B.npad + 1, 256), nc), gs(cdiv(B.npad, 256), nc);
      k_csc_count<<<gr, 256, 0, st>>>(B, d_cnt);
      size_t sb2 = 0; void* d_t2 = nullptr;
      cub::DeviceScan::ExclusiveSum(nullptr, sb2, d_cnt, d_scan, (int)np1, st);
      { char* p; CKT(tmp.alloc(&p, sb2, false, st)); d_t2 = p; }
      CKT(cub::DeviceScan::ExclusiveSum(d_t2, sb2, d_cnt, d_scan, (int)np1, st));
      k_csc_rebase2<<<gq, 256, 0, st>>>(B, d_scan, b->d_csc_ptr);
      CKT(cudaMemsetAsync(d_cnt, 0, np1 * sizeof(int), st));
      k_csc_fill<<<gr, 256, 0, st>>>(B, d_cnt, b->d_csc_ent);
      k_csc_sort<<<gs, 256, 0, st>>>(B, b->d_csc_ent);
      CKT(cudaGetLastError());
    }
    CKT(cudaStreamSynchronize(st));
    tmp.free_all();
  }
  // fixed-width copy of the transpose lists for the fast adjoint
  CKC(b->pool.alloc(&b->d_ell, (size_t)nc * HB2_ELL_W * B.npad, false, st));
  k_ell_fill<<<dim3(cdiv(B.npad, 256), nc), 256, 0, st>>>(B, b->d_ell);
  CKL();
  B.ell = b->d_ell;
  CKC(cudaStreamSynchronize(st));
  b->created = true;
  return HB2_OK;
}

// Half-set masks (fsc_test): upload, then rebuild the right-hand side and max(b) with the masks applied.
extern "C" int hb2_batch_set_pixel_masks(hb2_batch* b, int32_t n_masks, const uint8_t* masks, const int32_t* cand_mask) {
  if (!b || n_masks < 0 || (n_masks > 0 && !masks) || !cand_mask) return fail(HB2_ERR_ARG, "bad argument");
  if (!b->created) return fail(HB2_ERR_STATE, "hb2_batch_set_pixel_masks must follow hb2_batch_create");
  BD& B = b->B;
  CK(cudaSetDevice(b->P->device));
  cudaStream_t st = b->stream;
  const int nc = B.nc;
  const size_t npx = (size_t)B.L2 * B.D2;
  for (int c = 0; c < nc; ++c)
    if (cand_mask[c] >= n_masks) return fail(HB2_ERR_ARG, "cand_mask entry out of range");
  std::vector<uint8_t> hm(masks, masks + (size_t)n_masks * npx);
  std::vector<int> cm(cand_mask, cand_mask + nc);
  CK(upload(b->pool, &B.pixmask, hm, st));
  CK(upload(b->pool, &B.cand_pixmask, cm, st));
  if (n_masks == 0) B.pixmask = nullptr;
  std::vector<int> neg(nc, (int)0x80000000);
  CK(cudaMemcpyAsync(b->d_bmax, neg.data(), sizeof(int) * nc, cudaMemcpyHostToDevice, st));
  k_build_rhs<<<cdiv((long long)b->nviews * B.rows_per_view, 256), 256, 0, st>>>(B, b->P->d_pix, b->nviews, b->d_bmax);
  if (b->bilinear) k_bil_rhs<<<cdiv((long long)b->nviews * B.rows_per_view, 256), 256, 0, st>>>(B, b->P->d_pix, b->nviews, b->d_bmax);
  CKL();
  CK(cudaStreamSynchronize(st));
  return HB2_OK;
}

extern "C" void hb2_batch_destroy(hb2_batch* b) {
  if (!b) return;
  cudaSetDevice(b->P->device);
  cudaStreamSynchronize(b->stream);
  b->pool.free_all();
  for (cudaEvent_t e : b->ev_pool) cudaEventDestroy(e);
  if (b->side) { cudaStreamSynchronize(b->side); cudaStreamDestroy(b->side); }
  if (b->ev_fork) cudaEventDestroy(b->ev_fork);
  if (b->ev_join) cudaEventDestroy(b->ev_join);
  if (b->h_nactive) cudaFreeHost(b->h_nactive);
  delete b;
}

// Stored position of every symmetry row in the reference's order.  The rows of one pair round are stored in internal
// voxel order (k_sym_insert); the reference enumerates them in mask order (SLR:1197-1202): ord[r] = stored index of the
// reference's r-th row, recovered per round from the generating voxel's reference index.
static int sym_ref_order(hb2_batch* b, int c, std::vector<int>& ord) {
  const int m = b->h_msym[c];
  ord.resize(m);
  for (int r = 0; r < m; ++r) ord[r] = r;
  if (m == 0 || !b->d_sym_g) return HB2_OK;
  std::vector<int> gref(m);
  CK(cudaMemcpyAsync(gref.data(), b->d_sym_g + b->h_symoff[c], sizeof(int) * m, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  int start = 0;
  for (size_t rd = 0; rd < b->h_sym_round_end.size() && start < m; ++rd) {
    const int end = std::min(m, b->h_sym_round_end[rd][c]);
    if (end > start) std::sort(ord.begin() + start, ord.begin() + end, [&](int x, int y) { return gref[x] < gref[y]; });
    start = std::max(start, end);
  }
  return HB2_OK;
}

extern "C" int hb2_batch_sym_order(hb2_batch* b, int32_t c, int32_t* ord_host, int64_t capacity) {
  if (!b || !b->created || !ord_host || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  if (capacity < b->h_msym[c]) return fail(HB2_ERR_ARG, "capacity too small");
  CK(cudaSetDevice(b->P->device));
  std::vector<int> ord;
  if (int e = sym_ref_order(b, c, ord)) return e;
  memcpy(ord_host, ord.data(), sizeof(int) * ord.size());
  return HB2_OK;
}

extern "C" int hb2_batch_sym_rows(hb2_batch* b, int32_t c, int32_t* n_rows, int32_t* a_host, int32_t* b_host, int64_t capacity) {
  if (!b || !b->created || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  int m = b->h_msym[c];
  if (n_rows) *n_rows = m;
  if (a_host && b_host) {
    if (capacity < m) return fail(HB2_ERR_ARG, "capacity too small");
    CK(cudaMemcpyAsync(a_host, b->d_sym_a + b->h_symoff[c], sizeof(int) * m, cudaMemcpyDeviceToHost, b->stream));
    CK(cudaMemcpyAsync(b_host, b->d_sym_b + b->h_symoff[c], sizeof(int) * m, cudaMemcpyDeviceToHost, b->stream));
    const int L3P = b->B.L3P, nd = b->B.ndisk;
    const std::vector<int>& i2r = b->P->int2ref;
    std::vector<int> ord;
    if (int e = sym_ref_order(b, c, ord)) return e;
    std::vector<int> ta(a_host, a_host + m), tb(b_host, b_host + m);
    for (int r = 0; r < m; ++r) {  // internal p*L3P+z -> reference z*ndisk+rank
      a_host[r] = (ta[ord[r]] % L3P) * nd + i2r[ta[ord[r]] / L3P];
      b_host[r] = (tb[ord[r]] % L3P) * nd + i2r[tb[ord[r]] / L3P];
    }
  }
  return HB2_OK;
}

extern "C" int64_t hb2_batch_rows_padded(hb2_batch* b, int32_t c, int64_t* n_data_padded) {
  if (!b || !b->created || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  if (n_data_padded) *n_data_padded = b->h_mdata[c];
  return (int64_t)b->h_mdata[c] + b->h_msym[c];
}

extern "C" int hb2_batch_rhs(hb2_batch* b, int32_t c, float* out) {
  if (!b || !b->created || !out || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  CK(cudaMemcpyAsync(out, b->B.b + b->h_uoff[c], sizeof(float) * b->h_mdata[c], cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// optional per-launch profiling with CUDA events on the launching stream
// ---------------------------------------------------------------------------
enum { KC_FWD_DATA = 0, KC_FWD_SYM = 1, KC_ADJ = 2, KC_UPDATE = 3, KC_SCALAR = 4, KC_NORM = 5, KC_N = 6 };
struct ProfScope {
  hb2_batch* b;
  cudaStream_t s;
  int first = 0;
  ProfScope(hb2_batch* b_, int cls, cudaStream_t s_ = nullptr) : b(b_), s(s_ ? s_ : b_->stream) {
    if (!b->profiling) return;
    while (b->ev_pool.size() < b->ev_next + 2) { cudaEvent_t e; cudaEventCreate(&e); b->ev_pool.push_back(e); }
    first = (int)b->ev_next;
    b->ev_used.push_back({cls, first});
    cudaEventRecord(b->ev_pool[first], s);
    b->ev_next += 2;
  }
  ~ProfScope() {
    if (!b->profiling) return;
    cudaEventRecord(b->ev_pool[first + 1], s);
  }
};

// ---------------------------------------------------------------------------
// kernel dispatch
// ---------------------------------------------------------------------------
static void launch_fwd_data(hb2_batch* b, int mode) {
  ProfScope ps(b, KC_FWD_DATA);
  const BD& B = b->B;
  cudaStream_t st = b->stream;
  if (b->nviews == 0) return;
  if (b->n_tie_views > 0) {  // exact rows of the tie views (the projector kernels below skip them)
    const float* src = mode == MODE_LSMR ? B.v : B.xs;
    if (b->bilinear) {
      const dim3 gv(b->n_tie_views, B.fwd_ppv);
#define FBIL(I, Q) k_fwd_bil<I, Q, float, false><<<gv, HB2_BLOCK, 0, st>>>(B, TD{}, src, B.u, mode)
#define FBILQ(I) do { if (B.L3P == 4) FBIL(I, 1); else if (B.L3P == 8) FBIL(I, 2); else if (B.L3P == 12) FBIL(I, 3); else FBIL(I, 4); } while (0)
      if (b->idx16) FBILQ(uint16_t); else FBILQ(uint32_t);
#undef FBILQ
#undef FBIL
      k_fwd_lsym<float, false><<<gv, HB2_BLOCK, 0, st>>>(B, TD{}, src, B.u, mode);
      b->extra_launches += 1;
    } else if (b->explicit_rows) k_fwd_csr<float, false><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, TD{}, src, B.u, mode);
    else if (b->idx16) k_fwd_tie<uint16_t, float, false><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, TD{}, src, B.u, mode);
    else k_fwd_tie<uint32_t, float, false><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, TD{}, src, B.u, mode);
    b->extra_launches += 1;
  }
  if (B.fwd_band) {
    const size_t sm = b->fwd_band_smem;
    const dim3 gb(B.bt32.nband, B.nc), gr(b->max_views, B.nc);
#define FWB(Q)                                                                                            \
  do {                                                                                                    \
    hb2_allow_big_smem((const void*)k_fwd_band<Q, float, false>);                                         \
    k_fwd_band<Q, float, false><<<gb, HB2_FWDB_THREADS, sm, st>>>(B, TD{}, nullptr, mode);                \
    k_fwd_band_reduce<Q, float, false><<<gr, HB2_BLOCK, 0, st>>>(B, TD{}, nullptr, mode);                 \
  } while (0)
    if (B.L3P == 4) FWB(1); else if (B.L3P == 8) FWB(2); else if (B.L3P == 12) FWB(3); else FWB(4);
    b->extra_launches += 1;
#undef FWB
    return;
  }
  const int ntiles = (B.D2 + HB2_TILE_RAYS - 1) / HB2_TILE_RAYS;
  unsigned grid = (unsigned)b->nviews * ntiles;
#define FWD(T)                                                                              \
  do {                                                                                      \
    if (B.L3P == 4) k_fwd_data<T, 1><<<grid, HB2_BLOCK, 0, st>>>(B, mode);                  \
    else if (B.L3P == 8) k_fwd_data<T, 2><<<grid, HB2_BLOCK, 0, st>>>(B, mode);             \
    else if (B.L3P == 12) k_fwd_data<T, 3><<<grid, HB2_BLOCK, 0, st>>>(B, mode);            \
    else k_fwd_data<T, 4><<<grid, HB2_BLOCK, 0, st>>>(B, mode);                             \
  } while (0)
  if (b->idx16) FWD(uint16_t); else FWD(uint32_t);
#undef FWD
}
static void launch_fwd_sym(hb2_batch* b, int mode, cudaStream_t on = nullptr) {
  ProfScope ps(b, KC_FWD_SYM, on);
  const BD& B = b->B;
  dim3 g(B.part_us_per_cand, B.nc);
  k_fwd_sym<<<g, HB2_BLOCK, 0, on ? on : b->stream>>>(B, mode);
}
static void launch_adj(hb2_batch* b, int mode) {
  ProfScope ps(b, KC_ADJ);
  const BD& B = b->B;
  dim3 g(B.part_v_per_cand, B.nc);
  cudaStream_t st = b->stream;
  if (b->n_tie_views > 0) {  // contribution of the tie views, added by the adjoint kernels below
    if (b->bilinear) {
      const dim3 ga(cdiv(B.ndisk, (HB2_BLOCK / 32) * (32 / (B.L3P / 4))), B.nc);  // (voxel, quad) lanes
      const size_t smt = (size_t)HB2_BILT_NS * HB2_BILT_SV * ((size_t)B.bil_KB * HB2_BLOCK * 6 + (size_t)B.bil_rmax * B.L3P * sizeof(float));
      const bool use_tile = B.bil_adj_tile && smt <= 200 * 1024;
#define ABIL(Q)                                                                                      \
  do {                                                                                               \
    k_bil_unblend<Q, float, false><<<b->n_tie_views, HB2_BLOCK, 0, st>>>(B, TD{}, B.u, B.bil_ub, mode); \
    if (use_tile && B.bil_KB == 3) {                                                                 \
      hb2_allow_big_smem((const void*)k_adj_bil_tile<Q, 3, float, false>);                           \
      k_adj_bil_tile<Q, 3, float, false><<<dim3(B.ntile, B.nc), HB2_BILT_THREADS, smt, st>>>(B, TD{}, B.bil_ub, B.vtie, mode); \
    } else if (use_tile) {                                                                           \
      hb2_allow_big_smem((const void*)k_adj_bil_tile<Q, 0, float, false>);                           \
      k_adj_bil_tile<Q, 0, float, false><<<dim3(B.ntile, B.nc), HB2_BILT_THREADS, smt, st>>>(B, TD{}, B.bil_ub, B.vtie, mode); \
    } else k_adj_bil<Q, float, false><<<ga, HB2_BLOCK, 0, st>>>(B, TD{}, B.bil_ub, B.vtie, mode);   \
  } while (0)
      if (B.L3P == 4) ABIL(1); else if (B.L3P == 8) ABIL(2); else if (B.L3P == 12) ABIL(3); else ABIL(4);
#undef ABIL
      k_adj_lsym<float, false><<<dim3(cdiv(B.npad, HB2_BLOCK), B.nc), HB2_BLOCK, 0, st>>>(B, TD{}, B.u, B.vtie, mode);
      b->extra_launches += 2;
    } else if (b->explicit_rows) k_adj_csc<float, false><<<dim3(cdiv(B.npad, HB2_BLOCK / 32), B.nc), HB2_BLOCK, 0, st>>>(B, TD{}, B.u, B.vtie, mode);
    else k_adj_tie<float, false><<<dim3(cdiv(B.ndisk, HB2_BLOCK), B.nc), HB2_BLOCK, 0, st>>>(B, TD{}, B.u, B.vtie, mode);
    b->extra_launches += 1;
  }
  if (B.adj_tile == 2) {
    const size_t sm = b->adj_tile_smem;
    const dim3 gc(B.ntile, B.nc, b->adj_chunks);
#define ADJTC(K)                                                                                                        \
  do {                                                                                                                  \
    hb2_allow_big_smem((const void*)k_adj_tile<4, K, float, false, true>);   \
    k_adj_tile<4, K, float, false, true><<<gc, HB2_ADJT_THREADS, sm, st>>>(B, TD{}, B.u, nullptr, mode);                \
  } while (0)
    if (B.K == 1) ADJTC(1); else ADJTC(2);
#undef ADJTC
    return;
  }
  if (B.adj_tile) {
    const size_t sm = b->adj_tile_smem;
#define ADJT(Q, K)                                                                                                   \
  do {                                                                                                               \
    hb2_allow_big_smem((const void*)k_adj_tile<Q, K, float, false>);      \
    k_adj_tile<Q, K, float, false><<<g, HB2_ADJT_THREADS, sm, st>>>(B, TD{}, B.u, nullptr, mode);                    \
  } while (0)
#define ADJTQ(K) do { if (B.L3P == 4) ADJT(1, K); else if (B.L3P == 8) ADJT(2, K); else if (B.L3P == 12) ADJT(3, K); else ADJT(4, K); } while (0)
    if (B.K == 1) ADJTQ(1); else ADJTQ(2);
#undef ADJTQ
#undef ADJT
    return;
  }
  if (B.adj_fast) {
    if (B.K == 1) k_adj_pq<1><<<g, HB2_BLOCK, 0, st>>>(B, mode);
    else k_adj_pq<2><<<g, HB2_BLOCK, 0, st>>>(B, mode);
    return;
  }
#define ADJ(K, M) k_adj<K, M><<<g, HB2_BLOCK, 0, st>>>(B, mode)
  if (B.MC == 1) ADJ(0, 1);
  else ADJ(0, 0);
#undef ADJ
}
static void launch_update(hb2_batch* b, int mode) {
  ProfScope ps(b, KC_UPDATE);
  const BD& B = b->B;
  dim3 g(B.part_x_per_cand, B.nc);
  k_update<<<g, HB2_BLOCK, 0, b->stream>>>(B, mode);
}

extern "C" int hb2_batch_apply_forward(hb2_batch* b, int32_t c, const float* x_host, float* y_host) {
  if (!b || !b->created || !x_host || !y_host || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  BD& B = b->B;
  cudaStream_t st = b->stream;
  long long m = (long long)b->h_mdata[c] + b->h_msym[c];
  std::vector<float> xi((size_t)B.npad, 0.f);  // reference order z*ndisk+p -> internal p*L3P+z
  for (int z = 0; z < B.L3; ++z)
    for (int pp = 0; pp < B.ndisk; ++pp) xi[(size_t)pp * B.L3P + z] = x_host[(size_t)z * B.ndisk + b->P->int2ref[pp]];
  CK(cudaMemcpyAsync(B.xs + (size_t)c * B.npad, xi.data(), sizeof(float) * B.npad, cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(B.u + b->h_uoff[c], 0, sizeof(float) * m, st));
  B.only_cand = c;
  launch_fwd_data(b, MODE_PLAIN);
  launch_fwd_sym(b, MODE_PLAIN);
  B.only_cand = -1;
  CKL();
  CK(cudaMemcpyAsync(y_host, B.u + b->h_uoff[c], sizeof(float) * m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  b->solved = false;
  return HB2_OK;
}

extern "C" int hb2_batch_apply_adjoint(hb2_batch* b, int32_t c, const float* y_host, float* x_host) {
  if (!b || !b->created || !x_host || !y_host || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  BD& B = b->B;
  cudaStream_t st = b->stream;
  long long m = (long long)b->h_mdata[c] + b->h_msym[c];
  CK(cudaMemcpyAsync(B.u + b->h_uoff[c], y_host, sizeof(float) * m, cudaMemcpyHostToDevice, st));
  B.only_cand = c;
  launch_adj(b, MODE_PLAIN);
  B.only_cand = -1;
  CKL();
  std::vector<float> xi((size_t)B.npad);
  CK(cudaMemcpyAsync(xi.data(), B.xs + (size_t)c * B.npad, sizeof(float) * B.npad, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int z = 0; z < B.L3; ++z)
    for (int pp = 0; pp < B.ndisk; ++pp) x_host[(size_t)z * B.ndisk + b->P->int2ref[pp]] = xi[(size_t)pp * B.L3P + z];
  b->solved = false;
  return HB2_OK;
}


// ---------------------------------------------------------------------------
// bounded branch driver (hb2_trf.cuh): scipy trf_linear as a batched state machine
// ---------------------------------------------------------------------------
static int run_trf(hb2_batch* b, const hb2_solve_options* opt, std::vector<TrfState>& out, long long& launches, int& outer_iters) {
  BD& B = b->B;
  cudaStream_t st = b->stream;
  const int nc = B.nc;
  bool any = false;
  for (int c = 0; c < nc; ++c) any = any || b->cands[c].positive;
  out.assign(nc, TrfState{});
  if (!any) return HB2_OK;
  DevPool tmp;
  tmp.owner = b;
  TD T{};
#define CKT2(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { tmp.free_all(); return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
  const size_t nv = (size_t)nc * B.npad, nu = (size_t)b->u_total;
  double** nvecs[] = {&T.G, &T.D, &T.DH, &T.PH, &T.RH, &T.V, &T.H, &T.HBAR, &T.XIN, &T.W, &T.UN};
  for (double** p : nvecs) CKT2(tmp.alloc(p, nv, true, st));
  T.W2 = T.HBAR; T.AG = T.H;  // see TD
  B.vtie64 = nullptr;
  if (b->n_tie_views > 0) CKT2(tmp.alloc(&B.vtie64, nv, true, st));
  B.bil_ub64 = nullptr;
  if (b->bilinear) CKT2(tmp.alloc(&B.bil_ub64, nu, true, st));
  double** mvecs[] = {&T.R, &T.UM, &T.Y, &T.YP, &T.YAG};
  for (double** p : mvecs) CKT2(tmp.alloc(p, nu, true, st));
  long long max_m = 0;
  for (int c = 0; c < nc; ++c) max_m = std::max<long long>(max_m, (long long)b->h_mdata[c] + b->h_msym[c]);
  const unsigned gn = cdiv(B.npad, TRF_SPAN), gm = std::max(1u, cdiv(max_m, TRF_SPAN));
  T.gn = (int)gn; T.gm = (int)gm;
  T.red_slots = (int)(gn + gm);
  CKT2(tmp.alloc(&T.red, (size_t)nc * T.red_slots * TRF_NRED, true, st));
  CKT2(tmp.alloc(&T.st, nc, true, st));
  CKT2(tmp.alloc(&T.nactive, 1, true, st));
  CKT2(tmp.alloc(&T.ninner, 1, true, st));
  {
    std::vector<float> bmax(nc);
    CKT2(cudaMemcpyAsync(bmax.data(), b->d_bmax, sizeof(float) * nc, cudaMemcpyDeviceToHost, st));
    CKT2(cudaStreamSynchronize(st));
    std::vector<TrfState> hs(nc, TrfState{});
    for (int c = 0; c < nc; ++c) {
      int iv;
      memcpy(&iv, &bmax[c], 4);
      iv = iv >= 0 ? iv : iv ^ 0x7fffffff;  // undo the ordered-int encoding of k_build_rhs
      float ub;
      memcpy(&ub, &iv, 4);
      hs[c].needed = b->cands[c].positive ? 1 : 0;
      hs[c].lb = 0.0; hs[c].ub = (double)ub;  // SLR:247-248
      hs[c].tol = opt->trf_tol > 0 ? opt->trf_tol : 1e-2;
      if (!(hs[c].ub > hs[c].lb)) hs[c].needed = 0;  // scipy would raise "lb >= ub"
    }
    CKT2(cudaMemcpyAsync(T.st, hs.data(), sizeof(TrfState) * nc, cudaMemcpyHostToDevice, st));
    CKT2(cudaStreamSynchronize(st));
  }
  const double EPS = 2.220446049250313e-16;
  const int lsmr_maxiter = opt->max_iter > 0 ? opt->max_iter : 1000;
  const int max_iter = opt->trf_max_iter > 0 ? opt->trf_max_iter : 200;
  const dim3 g_sym(std::max(1, B.part_us_per_cand), nc);
  const dim3 g_adj(cdiv((long long)B.ndisk * (B.L3P / 4), HB2_BLOCK), nc);
  const size_t sm64 = (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.K * HB2_BLOCK * sizeof(uint16_t) +
                      (size_t)HB2_ADJT_NS * HB2_ADJT_SV * B.rmax * B.L3P * sizeof(double);
  const unsigned g_fwd = (unsigned)b->nviews * ((B.D2 + HB2_TILE_RAYS - 1) / HB2_TILE_RAYS);
  // pass<OP>() runs an element-wise pass; red(OP, SC) combines its partials and takes the scalar decision SC
  auto pass = [&](auto op) {
    constexpr int OP = decltype(op)::value;
    k_trf_pass<OP><<<dim3(trf_blocks(OP, gn, gm), nc), HB2_BLOCK, 0, st>>>(B, T);
    ++launches;
  };
  auto red = [&](auto op, int sc) {
    constexpr int OP = decltype(op)::value;
    k_trf_reduce<<<nc, HB2_BLOCK, 0, st>>>(B, T, (int)trf_blocks(OP, gn, gm), trf_mask(OP), sc, EPS, lsmr_maxiter, max_iter);
    ++launches;
  };
  auto pr = [&](auto op, int sc) { pass(op); red(op, sc); };
  using std::integral_constant;
#define OPC(X) integral_constant<int, X>{}
  auto fwd = [&](const double* src, double* dst, int gate) {
    if (B.bt64.nband > 0) {  // float64 instantiation of the band path (bands of half the voxels)
      const dim3 gb(B.bt64.nband, nc), gr(b->max_views, nc);
#define FWB64(Q)                                                                                          \
  do {                                                                                                    \
    hb2_allow_big_smem((const void*)k_fwd_band<Q, double, true>);                                         \
    k_fwd_band<Q, double, true><<<gb, HB2_FWDB_THREADS, b->fwd_band_smem64, st>>>(B, T, src, gate);       \
    k_fwd_band_reduce<Q, double, true><<<gr, HB2_BLOCK, 0, st>>>(B, T, dst, gate);                        \
  } while (0)
      if (B.L3P == 4) FWB64(2); else if (B.L3P == 8) FWB64(4); else if (B.L3P == 12) FWB64(6); else FWB64(8);
#undef FWB64
      ++launches;
    } else if (b->idx16) k_fwd64_data<uint16_t><<<g_fwd, HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
    else k_fwd64_data<uint32_t><<<g_fwd, HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
    k_fwd64_sym<<<g_sym, HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
    launches += 2;
    if (b->n_tie_views > 0) {
      if (b->bilinear) {
        const dim3 gv(b->n_tie_views, B.fwd_ppv);
#define FBIL(I, Q) k_fwd_bil<I, Q, double, true><<<gv, HB2_BLOCK, 0, st>>>(B, T, src, dst, gate)
#define FBILQ(I) do { if (B.L3P == 4) FBIL(I, 1); else if (B.L3P == 8) FBIL(I, 2); else if (B.L3P == 12) FBIL(I, 3); else FBIL(I, 4); } while (0)
        if (b->idx16) FBILQ(uint16_t); else FBILQ(uint32_t);
#undef FBILQ
#undef FBIL
        k_fwd_lsym<double, true><<<gv, HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
        ++launches;
      } else if (b->explicit_rows) k_fwd_csr<double, true><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
      else if (b->idx16) k_fwd_tie<uint16_t, double, true><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
      else k_fwd_tie<uint32_t, double, true><<<dim3(b->n_tie_views, B.fwd_ppv), HB2_BLOCK, 0, st>>>(B, T, src, dst, gate);
      ++launches;
    }
  };
  auto adj = [&](const double* rows, double* dst, int gate) {
    if (b->n_tie_views > 0) {
      if (b->bilinear) {
        const dim3 ga(cdiv(B.ndisk, (HB2_BLOCK / 32) * (32 / (B.L3P / 4))), nc);
        const size_t smt = (size_t)HB2_BILT_NS * HB2_BILT_SV * ((size_t)B.bil_KB * HB2_BLOCK * 6 + (size_t)B.bil_rmax * B.L3P * sizeof(double));
        const bool use_tile = B.bil_adj_tile && smt <= 200 * 1024;
#define ABIL(Q)                                                                                        \
  do {                                                                                                 \
    k_bil_unblend<Q, double, true><<<b->n_tie_views, HB2_BLOCK, 0, st>>>(B, T, rows, B.bil_ub64, gate); \
    if (use_tile) {                                                                                    \
      hb2_allow_big_smem((const void*)k_adj_bil_tile<Q, 0, double, true>);                             \
      k_adj_bil_tile<Q, 0, double, true><<<dim3(B.ntile, nc), HB2_BILT_THREADS, smt, st>>>(B, T, B.bil_ub64, B.vtie64, gate); \
    } else k_adj_bil<Q, double, true><<<ga, HB2_BLOCK, 0, st>>>(B, T, B.bil_ub64, B.vtie64, gate);    \
  } while (0)
        if (B.L3P == 4) ABIL(1); else if (B.L3P == 8) ABIL(2); else if (B.L3P == 12) ABIL(3); else ABIL(4);
#undef ABIL
        k_adj_lsym<double, true><<<dim3(cdiv(B.npad, HB2_BLOCK), nc), HB2_BLOCK, 0, st>>>(B, T, rows, B.vtie64, gate);
        launches += 2;
      } else if (b->explicit_rows) k_adj_csc<double, true><<<dim3(cdiv(B.npad, HB2_BLOCK / 32), nc), HB2_BLOCK, 0, st>>>(B, T, rows, B.vtie64, gate);
      else k_adj_tie<double, true><<<dim3(cdiv(B.ndisk, HB2_BLOCK), nc), HB2_BLOCK, 0, st>>>(B, T, rows, B.vtie64, gate);
      ++launches;
    }
    if (B.adj_tile == 1 && sm64 <= 200 * 1024) {  // float64 instantiation of the TMA-staged tile adjoint
      const dim3 gt(B.ntile, nc);
#define ADJT64(Q, K)                                                                                                 \
  do {                                                                                                               \
    hb2_allow_big_smem((const void*)k_adj_tile<Q, K, double, true>);    \
    k_adj_tile<Q, K, double, true><<<gt, HB2_ADJT_THREADS, sm64, st>>>(B, T, rows, dst, gate);                       \
  } while (0)
#define ADJT64Q(K) do { if (B.L3P == 4) ADJT64(1, K); else if (B.L3P == 8) ADJT64(2, K); else if (B.L3P == 12) ADJT64(3, K); else ADJT64(4, K); } while (0)
      if (B.K == 1) ADJT64Q(1); else ADJT64Q(2);
#undef ADJT64Q
#undef ADJT64
    } else {
      k_adj64<<<g_adj, HB2_BLOCK, 0, st>>>(B, T, rows, dst, gate);
    }
    ++launches;
  };
  auto read_counter = [&](int* dptr, int& v) -> cudaError_t {
    cudaError_t e = cudaMemcpyAsync(b->h_nactive, dptr, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(st);
    v = *b->h_nactive;
    return e;
  };
  // is the unconstrained solution feasible? (lsq_linear.py:328)
  pr(OPC(EW_START), SC_START);
  int nact = 0;
  CKT2(read_counter(T.nactive, nact));
  outer_iters = 0;
  if (nact > 0) {
    pass(OPC(EW_START_APPLY));
    fwd(T.W, T.Y, 0); pr(OPC(MW_RESID), SC_RESID0);
    adj(T.R, T.G, 0);
    for (int it = 0; it <= max_iter && nact > 0; ++it) {
      // scaling, the inner solve's first vector D*(A^T r) (A^T r = G: no adjoint) and the anti-gradient's n-space terms
      CKT2(cudaMemsetAsync(T.ninner, 0, sizeof(int), st));
      pr(OPC(EW_PREP), SC_PREP);
      CKT2(read_counter(T.nactive, nact));
      if (nact == 0) break;
      ++outer_iters;
      // inner LSMR on [A D; sqrt(diag_h)] p_h = -[r; 0]   (trf_linear.py:209-216)
      pass(OPC(EW_INNER_UPD));  // itn == 0: normalise v, h = v, hbar = x = 0, W = D v
      int ninner = 1;
      for (int k = 0; k < lsmr_maxiter && ninner > 0; ++k) {
        fwd(T.W, T.Y, 1); pr(OPC(NM_INNER_U), SC_INNER_BETA);
        adj(T.UM, T.W, 1); pr(OPC(EW_INNER_V), SC_INNER_ROT);
        pr(OPC(EW_INNER_UPD), SC_INNER_TEST);
        if (k % 2 == 1 || k + 1 == lsmr_maxiter) CKT2(read_counter(T.ninner, ninner));
      }
      // select_step (trf_linear.py:91-144): A*(D*RH), A*(D*PH) (full steps too), A*(-D*D*G)
      pr(OPC(EW_STEP1), SC_STEP1);
      pr(OPC(EW_STEP2), SC_STEP2);
      fwd(T.W, T.Y, 2); fwd(T.W2, T.YP, 0); fwd(T.AG, T.YAG, 2);
      pr(OPC(MW_DOTS), SC_SELECT);
      // predicted cost change from the three products, new point, residual, gradient (trf_linear.py:219-243)
      pr(OPC(NM_STEP), SC_CC);
      pass(OPC(EW_XUPD));
      fwd(T.W, T.Y, 0); pr(OPC(MW_RESID), SC_RESID);
      adj(T.R, T.G, 0);
      CKT2(cudaGetLastError());
    }
  }
  pass(OPC(EW_FINAL));
#undef OPC
  CKT2(cudaGetLastError());
  CKT2(cudaMemcpyAsync(out.data(), T.st, sizeof(TrfState) * nc, cudaMemcpyDeviceToHost, st));
  CKT2(cudaStreamSynchronize(st));
  tmp.free_all();
  B.vtie64 = nullptr;
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// solve + score
// ---------------------------------------------------------------------------
extern "C" int hb2_batch_solve(hb2_batch* b, const hb2_solve_options* opt, hb2_result* res) {
  if (!b || !b->created || !opt || !res) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(b->P->device));
  NvtxRange nvtx_("solve_equations + score (batch)");
  nvtxRangePushA("solve_equations: LSMR");
  struct PopGuard { int n = 1; ~PopGuard() { while (n-- > 0) nvtxRangePop(); } } nvtx_stage_;  // closes the open stage on every return
  BD& B = b->B;
  cudaStream_t st = b->stream;
  const int nc = B.nc;
  const int maxit = opt->max_iter > 0 ? opt->max_iter : 1000;
  const int check = opt->check_every > 0 ? opt->check_every : 8;
  B.clip_pred = opt->clip_pred;
  B.only_cand = -1;
  b->profiling = opt->profile != 0;
  b->ev_used.clear();
  b->ev_next = 0;
  cudaEvent_t e0, e1, e2;
  CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreate(&e2));
  CK(cudaEventRecord(e0, st));
  size_t nv = (size_t)nc * B.npad;
  CK(cudaMemsetAsync(B.x, 0, nv * sizeof(double), st));
  CK(cudaMemsetAsync(B.hbar, 0, nv * sizeof(double), st));
  CK(cudaMemsetAsync(B.h, 0, nv * sizeof(float), st));
  CK(cudaMemsetAsync(B.v, 0, nv * sizeof(float), st));
  CK(cudaMemcpyAsync(B.u, B.b, sizeof(float) * (size_t)b->u_total, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemsetAsync(b->d_nactive, 0, sizeof(int), st));
  long long launches = 0;
  b->extra_launches = 0;
  // norm_mode 1 (default): ||u||, ||v|| as numpy/OpenBLAS compute them for the reference (k_chain_sumsq); 0: exactly
  // rounded norms from the kernels' partial sums.  HB2_NORM_MODE overrides (experiments).
  static const int env_norm = [] { const char* e = getenv("HB2_NORM_MODE"); return e ? atoi(e) : -1; }();
  const bool chain = (env_norm >= 0 ? env_norm : opt->norm_mode) != 0;
  if (chain) {
    hb2_allow_big_smem((const void*)k_chain_sumsq<CHAIN_U>);
    hb2_allow_big_smem((const void*)k_chain_sumsq<CHAIN_V>);
    hb2_allow_big_smem((const void*)k_chain_sumsq<CHAIN_B>);
  }
  float* ch_u = chain ? b->d_chain : nullptr;
  float* ch_v = chain ? b->d_chain + nc : nullptr;
  if (chain) { k_chain_sumsq<CHAIN_B><<<nc, 64, HB2_CHAIN_SMEM, st>>>(B, ch_u, MODE_INIT); ++launches; }
  k_scal_normb<<<nc, HB2_BLOCK, 0, st>>>(B, ch_u);
  launch_adj(b, MODE_INIT);
  if (chain) { k_chain_sumsq<CHAIN_V><<<nc, 64, HB2_CHAIN_SMEM, st>>>(B, ch_v, MODE_INIT); ++launches; }
  k_scal_init<<<nc, HB2_BLOCK, 0, st>>>(B, b->d_nactive, ch_v);
  launch_update(b, MODE_INIT);
  launches += 4;
  CKL();
  int it = 0;
  // The symmetry-row forward runs on a side stream beside the band kernel unless per-launch profiling is on (the
  // per-class event times would overlap) or HB2_OVERLAP=0.  Measured at cfg2, 100 candidates: 37.53 -> 36.70 us per
  // candidate-iteration, identical scores -- both kernels load the LSU pipe, so only ~1 of the 4.3 us hides.
  static const int env_overlap = [] { const char* e = getenv("HB2_OVERLAP"); return e ? atoi(e) : 1; }();
  const bool overlap = env_overlap != 0 && !b->profiling;
  if (overlap && !b->side) {
    CK(cudaStreamCreateWithFlags(&b->side, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming));
  }
  *b->h_nactive = 1;
  CK(cudaMemcpyAsync(b->h_nactive, b->d_nactive, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  while (*b->h_nactive > 0 && it < maxit) {
    int burst = std::min(check, maxit - it);
    for (int q = 0; q < burst; ++q) {
      if (overlap) {  // fork: v and the scalars of this iteration are ready at this point of the main stream
        cudaEventRecord(b->ev_fork, st);
        launch_fwd_data(b, MODE_LSMR);
        cudaStreamWaitEvent(b->side, b->ev_fork, 0);
        launch_fwd_sym(b, MODE_LSMR, b->side);  // disjoint rows of u~ and its own partial sums
        cudaEventRecord(b->ev_join, b->side);
        cudaStreamWaitEvent(st, b->ev_join, 0);  // join before the norm of u~
      } else {
        launch_fwd_data(b, MODE_LSMR);
        launch_fwd_sym(b, MODE_LSMR);
      }
      if (chain) { ProfScope ps(b, KC_NORM); k_chain_sumsq<CHAIN_U><<<nc, 64, HB2_CHAIN_SMEM, st>>>(B, ch_u, MODE_LSMR); ++launches; }
      { ProfScope ps(b, KC_SCALAR); k_scal_beta<<<nc, HB2_BLOCK, 0, st>>>(B, ch_u); }
      launch_adj(b, MODE_LSMR);
      if (chain) { ProfScope ps(b, KC_NORM); k_chain_sumsq<CHAIN_V><<<nc, 64, HB2_CHAIN_SMEM, st>>>(B, ch_v, MODE_LSMR); ++launches; }
      { ProfScope ps(b, KC_SCALAR); k_scal_rot<<<nc, HB2_BLOCK, 0, st>>>(B, ch_v); }
      launch_update(b, MODE_LSMR);
      { ProfScope ps(b, KC_SCALAR); k_scal_test<<<nc, HB2_BLOCK, 0, st>>>(B, opt->atol, opt->btol, opt->conlim, maxit, opt->fixed_iters, b->d_nactive); }
      launches += 7;
    }
    it += burst;
    CKL();
    CK(cudaMemcpyAsync(b->h_nactive, b->d_nactive, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  CK(cudaEventRecord(e1, st));
  std::vector<TrfState> trf;
  int trf_outer = 0;
  cudaEvent_t e1b;
  CK(cudaEventCreate(&e1b));
  {
    dim3 g(cdiv(B.npad, 256), nc);
    k_x_to_f32<<<g, 256, 0, st>>>(B);
    ++launches;
  }
  nvtxRangePop(); nvtxRangePushA("solve_equations: bounded TRF");
  if (opt->fixed_iters <= 0) {  // bounded branch for candidates with the positive constraint (SLR:246-270)
    int rc = run_trf(b, opt, trf, launches, trf_outer);
    if (rc != HB2_OK) return rc;
  } else trf.assign(nc, TrfState{});
  CK(cudaEventRecord(e1b, st));
  nvtxRangePop(); nvtxRangePushA("cosine_similarity (reprojection + score)");
  // score: reprojection of float32(x) + cosine similarity
  {
    launch_fwd_data(b, MODE_SCORE);
    k_scal_score<<<nc, HB2_BLOCK, 0, st>>>(B, b->d_score);
    launches += 2;
    CKL();
  }
  CK(cudaEventRecord(e2, st));
  std::vector<LsmrState> hs(nc);
  std::vector<float> sc(nc);
  CK(cudaMemcpyAsync(hs.data(), B.st, sizeof(LsmrState) * nc, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(sc.data(), b->d_score, sizeof(float) * nc, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  float ms_l = 0, ms_s = 0, ms_t = 0;
  cudaEventElapsedTime(&ms_l, e0, e1); cudaEventElapsedTime(&ms_t, e1, e1b); cudaEventElapsedTime(&ms_s, e1b, e2);
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e1b); cudaEventDestroy(e2);
  for (double& t : b->timing) t = 0;
  b->timing[0] = ms_l; b->timing[1] = ms_t; b->timing[2] = ms_s; b->timing[13] = trf_outer; b->timing[3] = (double)(launches + b->extra_launches); b->timing[4] = it;
  if (b->profiling) {
    for (auto& pr : b->ev_used) {
      float ms = 0;
      cudaEventElapsedTime(&ms, b->ev_pool[pr.second], b->ev_pool[pr.second + 1]);
      if (pr.first == KC_NORM) b->timing[14] += ms;
      else b->timing[5 + pr.first] += ms;
      if (pr.first == KC_FWD_DATA) b->timing[10] += 1;
      if (pr.first == KC_ADJ) b->timing[11] += 1;
      if (pr.first == KC_UPDATE) b->timing[12] += 1;
    }
    b->profiling = false;
  }
  for (int c = 0; c < nc; ++c) {
    hb2_result& r = res[c];
    r.score = sc[c]; r.itn = hs[c].itn; r.istop = hs[c].istop; r.trf_nit = trf[c].status == 3 ? 0 : trf[c].nit;
    r.flags = b->cand_flags[c] | ((trf[c].needed && trf[c].status != 3) ? HB2_FLAG_BOUNDED : 0u);
    r.n_data_rows = 0; r.n_sym_rows = b->h_msym[c];
    r.normr = (float)hs[c].normr; r.normar = hs[c].normar; r.normA = (float)hs[c].normA; r.normx = (float)hs[c].normx;
  }
  b->solved = true;
  b->last_trf = trf;
  return HB2_OK;
}

extern "C" int hb2_batch_trf_trace(hb2_batch* b, int32_t c, double* out, int32_t max_rows) {
  if (!b || !out || c < 0 || c >= (int)b->last_trf.size()) return fail(HB2_ERR_ARG, "bad argument or no solve yet");
  const TrfState& S = b->last_trf[c];
  int n = std::min(std::min(S.nit, 24), (int)max_rows);
  for (int i = 0; i < n; ++i)
    for (int k = 0; k < 8; ++k) out[i * 8 + k] = S.trace[i][k];
  return S.nit * 16 + (S.status + 1);  // nit and status packed
}

extern "C" int hb2_batch_get_x(hb2_batch* b, int32_t c, float* x_host) {
  if (!b || !b->solved || !x_host || c < 0 || c >= b->B.nc) return fail(HB2_ERR_ARG, "bad argument or batch not solved");
  CK(cudaSetDevice(b->P->device));
  const BD& B = b->B;
  std::vector<float> xi((size_t)B.npad);
  CK(cudaMemcpyAsync(xi.data(), B.xs + (size_t)c * B.npad, sizeof(float) * B.npad, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  for (int z = 0; z < B.L3; ++z)
    for (int pp = 0; pp < B.ndisk; ++pp) x_host[(size_t)z * B.ndisk + b->P->int2ref[pp]] = xi[(size_t)pp * B.L3P + z];
  return HB2_OK;
}

extern "C" int hb2_batch_timing(hb2_batch* b, double* out16) {
  if (!b || !out16) return fail(HB2_ERR_ARG, "null argument");
  memcpy(out16, b->timing, sizeof(b->timing));
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// host test hook for the scalar recurrences
// ---------------------------------------------------------------------------
extern "C" int hb2_lsmr_scalar_step(double* state64, int phase, float alpha, float beta, double normx, double atol,
                                    double btol, double conlim, int maxiter, float* coef_hbar, float* coef_x,
                                    float* coef_h, double* trace8) {
  static_assert(sizeof(LsmrState) <= 64 * sizeof(double), "state scratch too small");
  LsmrState S;
  memcpy(&S, state64, sizeof(S));
  int ret = 0;
  if (phase == 0) lsmr_init_(S, alpha, beta);
  else if (phase == 1) lsmr_rotate_(S, alpha, beta);
  else ret = lsmr_test_(S, normx, atol, btol, conlim, maxiter);
  memcpy(state64, &S, sizeof(S));
  if (coef_hbar) *coef_hbar = S.cf_hbar;
  if (coef_x) *coef_x = S.cf_x;
  if (coef_h) *coef_h = S.cf_h;
  if (trace8) {
    trace8[0] = S.rho; trace8[1] = S.rhobar; trace8[2] = S.zeta; trace8[3] = S.normr; trace8[4] = S.normA;
    trace8[5] = S.test1; trace8[6] = S.test2; trace8[7] = S.active;
  }
  return ret;
}

// ---------------------------------------------------------------------------
// post-solve display products (hb2_symm.cuh)
// ---------------------------------------------------------------------------
extern "C" int hb2_helical_symmetrize(const float* data_host, const hb2_symm_params* p, const int64_t* k_begin,
                                      const int32_t* ent_h, const int32_t* ent_floor, const int32_t* ent_ceil,
                                      const double* ent_wk, const double* mats, int32_t n_mats, float* vol_out_host,
                                      float* xsum_out, float* ysum_out, float* zsum_out, int device, void* stream) {
  NvtxRange nvtx_("apply_helical_symmetry");
  if (!data_host || !p || !k_begin || !mats) return fail(HB2_ERR_ARG, "null argument");
  if (hb2_device_count() <= 0) return fail(HB2_ERR_NO_DEVICE, "no CUDA device visible; helicon_b200 has no CPU fallback");
  if (p->nz1 <= 0 || p->ny1 <= 0 || p->nx1 <= 0 || p->csym <= 0 || p->n_ent < 0) return fail(HB2_ERR_ARG, "bad sizes");
  if (p->zs0 < 0 || p->zs1 > p->nz1) return fail(HB2_ERR_ARG, "z-section slab outside the output");
  CK(cudaSetDevice(device));
  cudaStream_t st = (cudaStream_t)stream;
  SymmP P{};
  P.nz0 = p->nz0; P.ny0 = p->ny0; P.nx0 = p->nx0; P.nz = p->nz; P.ny = p->ny; P.nx = p->nx;
  P.oz = p->oz; P.oy = p->oy; P.ox = p->ox; P.nz1 = p->nz1; P.ny1 = p->ny1; P.nx1 = p->nx1;
  P.apix = p->apix; P.new_apix = p->new_apix; P.csym = p->csym; P.zs0 = p->zs0; P.zs1 = p->zs1;
  for (int e = 0; e < p->n_ent; ++e)
    if (ent_floor[e] < 0 || ent_ceil[e] >= p->nz0 || ent_h[e] < 0 || (long long)(ent_h[e] + 1) * p->csym > n_mats)
      return fail(HB2_ERR_ARG, "entry table out of range");
  DevPool pool;
  const size_t nd = (size_t)p->nz0 * p->ny0 * p->nx0, nv = (size_t)p->nz1 * p->ny1 * p->nx1;
  float *d_data, *d_vol, *d_x, *d_y, *d_z;
  long long* d_kb; int *d_h, *d_f, *d_c; double *d_w, *d_m;
#define CKS(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { pool.free_all(); return fail(HB2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } } while (0)
  CKS(pool.alloc(&d_data, nd, false, st)); CKS(pool.alloc(&d_vol, nv, false, st));
  CKS(pool.alloc(&d_x, (size_t)p->nz1 * p->ny1, false, st)); CKS(pool.alloc(&d_y, (size_t)p->nz1 * p->nx1, false, st));
  CKS(pool.alloc(&d_z, (size_t)p->ny1 * p->nx1, false, st));
  CKS(pool.alloc(&d_kb, (size_t)p->nz1 + 1, false, st)); CKS(pool.alloc(&d_h, (size_t)p->n_ent, false, st));
  CKS(pool.alloc(&d_f, (size_t)p->n_ent, false, st)); CKS(pool.alloc(&d_c, (size_t)p->n_ent, false, st));
  CKS(pool.alloc(&d_w, (size_t)p->n_ent, false, st)); CKS(pool.alloc(&d_m, (size_t)n_mats * 4, false, st));
  CKS(cudaMemcpyAsync(d_data, data_host, nd * sizeof(float), cudaMemcpyHostToDevice, st));
  CKS(cudaMemcpyAsync(d_kb, k_begin, ((size_t)p->nz1 + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
  if (p->n_ent) {
    CKS(cudaMemcpyAsync(d_h, ent_h, (size_t)p->n_ent * sizeof(int), cudaMemcpyHostToDevice, st));
    CKS(cudaMemcpyAsync(d_f, ent_floor, (size_t)p->n_ent * sizeof(int), cudaMemcpyHostToDevice, st));
    CKS(cudaMemcpyAsync(d_c, ent_ceil, (size_t)p->n_ent * sizeof(int), cudaMemcpyHostToDevice, st));
    CKS(cudaMemcpyAsync(d_w, ent_wk, (size_t)p->n_ent * sizeof(double), cudaMemcpyHostToDevice, st));
  }
  CKS(cudaMemcpyAsync(d_m, mats, (size_t)n_mats * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
  k_symm_volume<<<cdiv((long long)nv, 256), 256, 0, st>>>(P, d_data, d_kb, d_h, d_f, d_c, d_w, d_m, d_vol);
  const long long nproj = (long long)p->nz1 * p->ny1 + (long long)p->nz1 * p->nx1 + (long long)p->ny1 * p->nx1;
  k_symm_project<<<cdiv(nproj, 128), 128, 0, st>>>(P, d_vol, d_x, d_y, d_z);
  CKS(cudaGetLastError());
  if (vol_out_host) CKS(cudaMemcpyAsync(vol_out_host, d_vol, nv * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (xsum_out) CKS(cudaMemcpyAsync(xsum_out, d_x, (size_t)p->nz1 * p->ny1 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (ysum_out) CKS(cudaMemcpyAsync(ysum_out, d_y, (size_t)p->nz1 * p->nx1 * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (zsum_out) CKS(cudaMemcpyAsync(zsum_out, d_z, (size_t)p->ny1 * p->nx1 * sizeof(float), cudaMemcpyDeviceToHost, st));
  CKS(cudaStreamSynchronize(st));
  pool.free_all();
#undef CKS
  return HB2_OK;
}

// ---------------------------------------------------------------------------
// device-resident score map + top-K of a search (include/helicon_b200.h)
// ---------------------------------------------------------------------------
struct hb2_scoremap {
  int device = 0;
  long long n = 0;
  float* d_score = nullptr;  // [n] float32 scores, then [n] int32 iterations, then [n] uint32 flags
  int* d_itn = nullptr;
  unsigned* d_flags = nullptr;
  long long* d_idx = nullptr;  // staging of a batch's task indices (+ flags behind them)
  size_t idx_cap = 0;
  float* d_top = nullptr;      // [k] scores + [k] indices (as long long)
  long long* d_topi = nullptr;
  int top_cap = 0;
};

__global__ void k_scoremap_fill(float* __restrict__ sc, int* __restrict__ it, unsigned* __restrict__ fl, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { sc[i] = __int_as_float(0x7fc00000); it[i] = 0; fl[i] = 0u; }
}
__global__ void k_scoremap_scatter(const float* __restrict__ score, const LsmrState* __restrict__ st,
                                   const long long* __restrict__ idx, int nc, long long n, float* __restrict__ sc,
                                   int* __restrict__ it, unsigned* __restrict__ fl) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const long long t = idx[c];
  if (t < 0 || t >= n) return;
  sc[t] = score[c];
  it[t] = st[c].itn;
  fl[t] = (unsigned)idx[nc + c];
}
// other ranks' maps (an all-gathered buffer of n_maps x [scores | iterations]): a task is owned by at most one rank
__global__ void k_scoremap_merge(float* __restrict__ sc, int* __restrict__ it, unsigned* __restrict__ fl,
                                 const float* __restrict__ g, int n_maps, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = sc[i];
  int q = it[i];
  unsigned f = fl[i];
  for (int r = 0; r < n_maps; ++r) {
    const float v = g[(size_t)r * 3 * n + i];
    if (v == v && !(s == s)) {
      s = v;
      q = reinterpret_cast<const int*>(g)[(size_t)r * 3 * n + n + i];
      f = reinterpret_cast<const unsigned*>(g)[(size_t)r * 3 * n + 2 * n + i];
    }
  }
  sc[i] = s; it[i] = q; fl[i] = f;
}
// K rounds of a CTA-wide arg-max (score descending, lower index wins ties, NaN skipped); entries already selected are
// excluded by comparing with the previous winner in (score, index) order, so the map itself stays untouched.
__global__ void __launch_bounds__(1024) k_scoremap_topk(const float* __restrict__ sc, long long n, int k,
                                                        float* __restrict__ top, long long* __restrict__ topi) {
  __shared__ float s_v[32];
  __shared__ long long s_i[32];
  __shared__ float prev_v;
  __shared__ long long prev_i;
  if (threadIdx.x == 0) { prev_v = INFINITY; prev_i = -1; }
  __syncthreads();
  for (int r = 0; r < k; ++r) {
    const float pv = prev_v;
    const long long pi = prev_i;
    float bv = -INFINITY;
    long long bi = -1;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
      const float v = sc[i];
      if (!(v == v)) continue;
      const bool after_prev = pi < 0 || v < pv || (v == pv && i > pi);  // strictly after the previous winner
      if (!after_prev) continue;
      if (bi < 0 || v > bv || (v == bv && i < bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { s_v[threadIdx.x >> 5] = bv; s_i[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x < 32) {
      bv = threadIdx.x < (blockDim.x >> 5) ? s_v[threadIdx.x] : -INFINITY;
      bi = threadIdx.x < (blockDim.x >> 5) ? s_i[threadIdx.x] : -1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
      }
      if (threadIdx.x == 0) { top[r] = bi >= 0 ? bv : __int_as_float(0x7fc00000); topi[r] = bi; prev_v = bv; prev_i = bi >= 0 ? bi : (long long)n; }
    }
    __syncthreads();
  }
}

extern "C" int hb2_scoremap_create(hb2_scoremap** out, int64_t n, int device) {
  if (!out || n <= 0) return fail(HB2_ERR_ARG, "bad argument");
  if (hb2_device_count() <= 0) return fail(HB2_ERR_NO_DEVICE, "no CUDA device visible; helicon_b200 has no CPU fallback");
  CK(cudaSetDevice(device));
  auto* m = new hb2_scoremap();
  m->device = device; m->n = n;
  if (cudaMalloc((void**)&m->d_score, (size_t)n * 12) != cudaSuccess) { delete m; return fail(HB2_ERR_CUDA, "cudaMalloc of the score map failed"); }
  m->d_itn = reinterpret_cast<int*>(m->d_score + n);
  m->d_flags = reinterpret_cast<unsigned*>(m->d_score + 2 * n);
  k_scoremap_fill<<<cdiv(n, 256), 256>>>(m->d_score, m->d_itn, m->d_flags, n);
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  *out = m;
  return HB2_OK;
}
extern "C" void hb2_scoremap_destroy(hb2_scoremap* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  if (m->d_score) cudaFree(m->d_score);
  if (m->d_idx) cudaFree(m->d_idx);
  if (m->d_top) cudaFree(m->d_top);
  if (m->d_topi) cudaFree(m->d_topi);
  delete m;
}
extern "C" void* hb2_scoremap_device_ptr(hb2_scoremap* m) { return m ? (void*)m->d_score : nullptr; }
extern "C" int hb2_batch_scatter_scores(hb2_batch* b, hb2_scoremap* m, const int64_t* task_index_host,
                                        const uint32_t* flags_host) {
  if (!b || !b->solved || !m || !task_index_host || !flags_host) return fail(HB2_ERR_ARG, "bad argument or batch not solved");
  if (m->device != b->P->device) return fail(HB2_ERR_ARG, "score map and batch live on different devices");
  CK(cudaSetDevice(m->device));
  const int nc = b->B.nc;
  cudaStream_t st = b->stream;
  if (m->idx_cap < (size_t)2 * nc) {
    CK(cudaStreamSynchronize(st));
    if (m->d_idx) cudaFree(m->d_idx);
    m->idx_cap = std::max<size_t>(2048, (size_t)nc * 4);
    CK(cudaMalloc((void**)&m->d_idx, m->idx_cap * sizeof(long long)));
  }
  std::vector<long long> stage((size_t)2 * nc);
  for (int c = 0; c < nc; ++c) { stage[c] = task_index_host[c]; stage[nc + c] = flags_host[c]; }
  CK(cudaMemcpyAsync(m->d_idx, stage.data(), sizeof(long long) * 2 * nc, cudaMemcpyHostToDevice, st));
  k_scoremap_scatter<<<cdiv(nc, 128), 128, 0, st>>>(b->d_score, b->B.st, m->d_idx, nc, m->n, m->d_score, m->d_itn, m->d_flags);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st));  // task_index_host may go away; the staging buffer is shared by the search's batches
  return HB2_OK;
}
// entries of an earlier, interrupted search (checkpoint.py): packed (index, score bits, iterations, flags) records
__global__ void k_scoremap_restore(const long long* __restrict__ rec, long long n_entries, long long n,
                                   float* __restrict__ sc, int* __restrict__ it, unsigned* __restrict__ fl) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_entries) return;
  const long long t = rec[2 * e];
  if (t < 0 || t >= n) return;
  const unsigned long long w = (unsigned long long)rec[2 * e + 1];  // iterations << 32 | score bits
  sc[t] = __uint_as_float((unsigned)(w & 0xffffffffull));
  it[t] = (int)(unsigned)(w >> 32);
  fl[t] = (unsigned)rec[2 * n_entries + e];
}
extern "C" int hb2_scoremap_restore(hb2_scoremap* m, int64_t n_entries, const int64_t* task_index_host,
                                    const float* scores_host, const int32_t* itn_host, const uint32_t* flags_host) {
  if (!m || n_entries < 0 || (n_entries > 0 && (!task_index_host || !scores_host || !itn_host || !flags_host)))
    return fail(HB2_ERR_ARG, "bad argument");
  if (n_entries == 0) return HB2_OK;
  CK(cudaSetDevice(m->device));
  std::vector<long long> stage((size_t)3 * n_entries);
  for (int64_t e = 0; e < n_entries; ++e) {
    if (task_index_host[e] < 0 || task_index_host[e] >= m->n) return fail(HB2_ERR_ARG, "restored task index outside the map");
    unsigned sb;
    memcpy(&sb, &scores_host[e], 4);
    stage[2 * e] = task_index_host[e];
    stage[2 * e + 1] = (long long)(((unsigned long long)(unsigned)itn_host[e] << 32) | sb);
    stage[2 * n_entries + e] = flags_host[e];
  }
  long long* d = nullptr;
  CK(cudaMalloc((void**)&d, sizeof(long long) * stage.size()));
  cudaError_t e1 = cudaMemcpy(d, stage.data(), sizeof(long long) * stage.size(), cudaMemcpyHostToDevice);
  if (e1 == cudaSuccess) {
    k_scoremap_restore<<<cdiv(n_entries, 256), 256>>>(d, n_entries, m->n, m->d_score, m->d_itn, m->d_flags);
    e1 = cudaGetLastError();
    if (e1 == cudaSuccess) e1 = cudaDeviceSynchronize();
  }
  cudaFree(d);
  if (e1 != cudaSuccess) return fail(HB2_ERR_CUDA, std::string("hb2_scoremap_restore: ") + cudaGetErrorString(e1));
  return HB2_OK;
}
extern "C" int hb2_scoremap_merge(hb2_scoremap* m, const void* gathered_dev, int32_t n_maps, void* stream) {
  if (!m || !gathered_dev || n_maps <= 0) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(m->device));
  k_scoremap_merge<<<cdiv(m->n, 256), 256, 0, (cudaStream_t)stream>>>(m->d_score, m->d_itn, m->d_flags, (const float*)gathered_dev, n_maps, m->n);
  CK(cudaGetLastError());
  return HB2_OK;
}
extern "C" int hb2_scoremap_topk(hb2_scoremap* m, int32_t k, float* top_scores_host, int64_t* top_index_host, void* stream) {
  if (!m || k <= 0 || !top_scores_host || !top_index_host) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (m->top_cap < k) {
    if (m->d_top) cudaFree(m->d_top);
    if (m->d_topi) cudaFree(m->d_topi);
    CK(cudaMalloc((void**)&m->d_top, sizeof(float) * k));
    CK(cudaMalloc((void**)&m->d_topi, sizeof(long long) * k));
    m->top_cap = k;
  }
  k_scoremap_topk<<<1, 1024, 0, st>>>(m->d_score, m->n, k, m->d_top, m->d_topi);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(top_scores_host, m->d_top, sizeof(float) * k, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(top_index_host, m->d_topi, sizeof(long long) * k, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return HB2_OK;
}
extern "C" int hb2_scoremap_read(hb2_scoremap* m, float* scores_host, int32_t* itn_host, uint32_t* flags_host, void* stream) {
  if (!m) return fail(HB2_ERR_ARG, "bad argument");
  CK(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (scores_host) CK(cudaMemcpyAsync(scores_host, m->d_score, sizeof(float) * m->n, cudaMemcpyDeviceToHost, st));
  if (itn_host) CK(cudaMemcpyAsync(itn_host, m->d_itn, sizeof(int) * m->n, cudaMemcpyDeviceToHost, st));
  if (flags_host) CK(cudaMemcpyAsync(flags_host, m->d_flags, sizeof(unsigned) * m->n, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return HB2_OK;
}
