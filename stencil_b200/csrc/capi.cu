// C ABI of stencil_b200 (include/stencil_b200.h): geometry wrappers over the C++ host mirror
// (include/stencil/*.hpp), copy plans over box_copy.cu, jacobi launches, device/peer/IPC plumbing.
#include "stencil_b200.h"

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cuda.h> // CUtensorMap types only: the driver entry point is resolved at run time, libcuda is not linked
#include <cuda_runtime.h>

#include "box_copy.cuh"
#include "astaroth.cuh"
#include "jacobi.cuh"
#include "reduce.cuh"

#include "stencil/geometry.hpp"
#include "stencil/partition_core.hpp"

namespace {

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

int fail(sb_status code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return int(code);
}

#define SB_CUDA(expr)                                                                                                  \
  do {                                                                                                                 \
    cudaError_t e_ = (expr);                                                                                           \
    if (e_ != cudaSuccess) return fail(SB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) {
      ok = false;
      return;
    }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// The compute entry points take pointers and a stream but no device: the launch must happen on the device that owns the
// memory (and the stream), whatever the calling thread's current device is -- a caller that drives several GPUs (or a test
// that ran on another GPU before) would otherwise get "invalid resource handle" from the launch.
int device_of(const void *ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) ? a.device : -1;
}
struct PtrDeviceGuard {
  int prev = -1;
  explicit PtrDeviceGuard(const void *ptr) {
    const int dev = device_of(ptr);
    int cur = -1;
    if (dev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != dev && cudaSetDevice(dev) == cudaSuccess) prev = cur;
  }
  ~PtrDeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

Dim3 d3(const int64_t v[3]) { return Dim3(v[0], v[1], v[2]); }
void put(const Dim3 &d, int64_t out[3]) {
  out[0] = d.x;
  out[1] = d.y;
  out[2] = d.z;
}
Radius radius_of(const int64_t r27[27]) {
  Radius r = Radius::constant(0);
  int i = 0;
  for (int z = -1; z <= 1; ++z)
    for (int y = -1; y <= 1; ++y)
      for (int x = -1; x <= 1; ++x) r.dir(x, y, z) = size_t(r27[i++]);
  return r;
}
bool dir_ok(const int64_t d[3]) {
  for (int a = 0; a < 3; ++a)
    if (d[a] < -1 || d[a] > 1) return false;
  return true;
}

unsigned ceil_log2(unsigned v) {
  unsigned b = 0;
  while ((1ull << b) < v) ++b;
  return b;
}

// Turn one sb_box_copy into >= 1 kernel segments (see box_copy.cuh).
int build_segments(const sb_box_copy &c, std::vector<sb::Seg> &out) {
  const int64_t es = c.elem_size;
  if (es <= 0 || (es & (es - 1)) != 0 || es > 16) return fail(SB_ERR_INVALID, "elem_size %lld must be 1,2,4,8 or 16", (long long)es);
  for (int a = 0; a < 3; ++a) {
    if (c.extent[a] < 0 || c.src_pos[a] < 0 || c.dst_pos[a] < 0) return fail(SB_ERR_INVALID, "negative extent/position");
  }
  if (c.extent[0] == 0 || c.extent[1] == 0 || c.extent[2] == 0) return SB_OK; // empty box: nothing to do
  if (!c.src.ptr || !c.dst.ptr) return fail(SB_ERR_INVALID, "null pointer in box copy");
  if (c.src.pitch <= 0 || c.dst.pitch <= 0 || c.src.ysize <= 0 || c.dst.ysize <= 0)
    return fail(SB_ERR_INVALID, "pitch/ysize must be positive");

  long long row_bytes = c.extent[0] * es;
  long long ny = c.extent[1], nz = c.extent[2];
  long long sp = c.src.pitch, ss = c.src.pitch * c.src.ysize;
  long long dp = c.dst.pitch, ds = c.dst.pitch * c.dst.ysize;
  const char *src = static_cast<const char *>(c.src.ptr) + (c.src_pos[2] * c.src.ysize + c.src_pos[1]) * c.src.pitch + c.src_pos[0] * es;
  char *dst = static_cast<char *>(c.dst.ptr) + (c.dst_pos[2] * c.dst.ysize + c.dst_pos[1]) * c.dst.pitch + c.dst_pos[0] * es;

  // merge dimensions that are contiguous on BOTH sides (full-width rows / full planes)
  const long long kMaxRow = 1ll << 30;
  if (ny > 1 && sp == row_bytes && dp == row_bytes && row_bytes * ny < kMaxRow) {
    row_bytes *= ny;
    ny = 1;
  }
  if (ny == 1 && nz > 1 && ss == row_bytes && ds == row_bytes && row_bytes * nz < kMaxRow) {
    row_bytes *= nz;
    nz = 1;
  }
  if (ny == 1 && nz > 1) { // a single row per plane: planes become the rows
    ny = nz;
    nz = 1;
    sp = ss;
    dp = ds;
  }
  if (row_bytes >= (1ll << 31)) return fail(SB_ERR_INVALID, "row of %lld bytes too long", row_bytes);

  auto emit = [&](const char *s, char *d, long long rb, long long rows_y, long long rows_z, long long spitch, long long sslice,
                  long long dpitch, long long dslice) -> int {
    // keep rows per segment below 2^24 (range of the divide-free row split)
    const long long kMaxRows = (1ll << 24) - 1;
    if (rows_y > kMaxRows) return fail(SB_ERR_INVALID, "more than 2^24 rows per plane");
    long long zmax = kMaxRows / rows_y;
    for (long long z0 = 0; z0 < rows_z; z0 += zmax) {
      const long long zn = (rows_z - z0 < zmax) ? rows_z - z0 : zmax;
      sb::Seg g{};
      g.src = s + z0 * sslice;
      g.dst = d + z0 * dslice;
      g.src_pitch = spitch;
      g.src_slice = sslice;
      g.dst_pitch = dpitch;
      g.dst_slice = dslice;
      g.row_bytes = unsigned(rb);
      g.ny = unsigned(rows_y);
      g.nz = unsigned(zn);
      unsigned long long align = (unsigned long long)(uintptr_t)g.src | (unsigned long long)(uintptr_t)g.dst | (unsigned long long)rb;
      if (rows_y > 1) align |= (unsigned long long)spitch | (unsigned long long)dpitch;
      if (zn > 1) align |= (unsigned long long)sslice | (unsigned long long)dslice;
      unsigned vec = 16;
      while (vec > 1 && (align & (vec - 1))) vec >>= 1;
      g.vec = vec;
      const unsigned nvec = unsigned(rb) / vec;
      unsigned lg = ceil_log2(nvec);
      if (lg > 5) lg = 5;
      g.lg_group = lg;
      const unsigned bits = ceil_log2(unsigned(rows_y));
      g.ny_shift = 24 + bits;
      g.ny_magic = ((1ull << g.ny_shift) + unsigned(rows_y) - 1) / unsigned(rows_y);
      out.push_back(g);
    }
    return SB_OK;
  };

  if (ny == 1 && nz == 1 && row_bytes > 2 * (long long)sb::kTileBytes) {
    // one long contiguous run: cut it into tile-sized "rows"
    const long long chunk = sb::kTileBytes;
    const long long q = row_bytes / chunk, rem = row_bytes % chunk;
    int rc = emit(src, dst, chunk, q, 1, chunk, chunk * q, chunk, chunk * q);
    if (rc != SB_OK) return rc;
    if (rem) rc = emit(src + q * chunk, dst + q * chunk, rem, 1, 1, rem, rem, rem, rem);
    return rc;
  }
  return emit(src, dst, row_bytes, ny, nz, sp, ss, dp, ds);
}

int env_int(const char *name, int dflt);

// ------------------------------------------------------------------------------------------- TMA segments
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      return nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

struct MapKey {
  void *ptr;
  int64_t pitch, ysize, es;
  unsigned bx;
  bool operator==(const MapKey &o) const { return ptr == o.ptr && pitch == o.pitch && ysize == o.ysize && es == o.es && bx == o.bx; }
};

struct TmaBuild {
  std::vector<CUtensorMap> maps;
  std::vector<MapKey> keys;
  std::vector<sb::TmaSeg> segs; // smap/dmap are indices into maps
  std::vector<int> kinds;       // 1 = TMA load + TMA store, 2 = TMA load + vector stores
};

// tensor map of a whole allocation, box = bx x 1 x 1 elements
int tma_map_index(TmaBuild &tb, const sb_pitched &a, int64_t es, unsigned bx) {
  const MapKey key{a.ptr, a.pitch, a.ysize, es, bx};
  for (size_t i = 0; i < tb.keys.size(); ++i)
    if (tb.keys[i] == key) return int(i);
  if (tb.maps.size() >= size_t(sb::kMaxTmaMaps)) return -1; // parameter space holds kMaxTmaMaps descriptors
  CUtensorMapDataType dt = es == 8 ? CU_TENSOR_MAP_DATA_TYPE_UINT64
                           : es == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32
                                     : es == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8;
  const cuuint64_t dims[3] = {cuuint64_t(a.pitch / es), cuuint64_t(a.ysize), cuuint64_t(1) << 20};
  const cuuint64_t strides[2] = {cuuint64_t(a.pitch), cuuint64_t(a.pitch) * cuuint64_t(a.ysize)};
  const cuuint32_t box[3] = {bx, 1, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = encode_tiled_fn()(&m, dt, 3, a.ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                       CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return -1;
  tb.maps.push_back(m);
  tb.keys.push_back(key);
  return int(tb.maps.size()) - 1;
}

// returns true if the copy was taken over by the TMA path
bool try_tma_segment(const sb_box_copy &c, TmaBuild &tb, int plan_device) {
  const int enabled = env_int("SB_TMA", 0); // opt-in: measured slower than the LSU path (profiles/README.md section 4)
  static const int peer_ok = env_int("SB_TMA_PEER", 1); // TMA stores into peer-mapped (NVLink) memory
  if (!enabled || !encode_tiled_fn()) return false;
  if (!peer_ok) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, c.dst.ptr) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    if (at.type == cudaMemoryTypeDevice && at.device != plan_device) return false;
  }
  const int64_t es = c.elem_size;
  if (es != 1 && es != 2 && es != 4 && es != 8) return false;
  const int64_t row_bytes = c.extent[0] * es;
  if (row_bytes < 512) return false; // thin rows stay on the LSU path
  for (const sb_pitched *a : {&c.src, &c.dst}) {
    if ((uintptr_t(a->ptr) & 15) || (a->pitch & 15) || ((a->pitch * a->ysize) & 15) || (a->pitch % es)) return false;
    if (a->pitch * a->ysize >= (int64_t(1) << 40)) return false;
  }
  // MEASURED on B200 (scripts/exp/tma_probe3.cu): the global address a box starts at must itself be 16-byte
  // aligned -- a UINT64 box at x = 1 (or an INT32 box at x = 1..3) raises "illegal instruction" at the
  // UTMALDG, x = 2 (x = 4) is fine.  Rows of an FP64 r=1 halo start 8 bytes into the row, so they are NOT
  // directly TMA-addressable; such segments take the LSU path (or the aligned-down TMA-load kind).
  if ((c.src_pos[0] * es) & 15 || (c.dst_pos[0] * es) & 15) return false;
  // chunk width: the whole row if it fits a box, else its largest divisor that does
  unsigned bx = 0;
  for (int64_t d = std::min<int64_t>(256, c.extent[0]); d >= 1; --d) {
    if (c.extent[0] % d == 0 && (d * es) % 16 == 0 && d * es >= 256) {
      bx = unsigned(d);
      break;
    }
  }
  if (0 == bx) return false;
  const int64_t rows = c.extent[1] * c.extent[2];
  if (rows >= (1 << 24) || c.extent[1] >= (1 << 24)) return false;
  for (int a = 0; a < 3; ++a)
    if (c.src_pos[a] + c.extent[a] >= (int64_t(1) << 20) && a == 2) return false;
  const int si = tma_map_index(tb, c.src, es, bx), di = tma_map_index(tb, c.dst, es, bx);
  if (si < 0 || di < 0) return false;
  sb::TmaSeg t{};
  t.sx0 = int(c.src_pos[0]);
  t.sy0 = int(c.src_pos[1]);
  t.sz0 = int(c.src_pos[2]);
  t.dx0 = int(c.dst_pos[0]);
  t.dy0 = int(c.dst_pos[1]);
  t.dz0 = int(c.dst_pos[2]);
  t.bx = bx;
  t.chunks_per_row = unsigned(c.extent[0] / bx);
  t.chunk_bytes = unsigned(bx * es);
  t.ny = unsigned(c.extent[1]);
  t.nz = unsigned(c.extent[2]);
  const unsigned bits = ceil_log2(t.ny);
  t.ny_shift = 24 + bits;
  t.ny_magic = ((1ull << t.ny_shift) + t.ny - 1) / t.ny;
  t.smap = si;
  t.dmap = di;
  t.cstride = (t.chunk_bytes + 127u) & ~127u; // shared-memory box addresses must be 128-byte aligned
  t.es = unsigned(es);
  tb.segs.push_back(t);
  tb.kinds.push_back(1);
  return true;
}

// kind 2: TMA loads from an aligned-down start + vector stores by the CTA (see box_copy.cuh).  Applies to
// wide rows of 4- or 8-byte elements whose SOURCE allocation is TMA-legal; the destination can be anything.
bool try_tma_load_segment(const sb_box_copy &c, TmaBuild &tb) {
  const int enabled = env_int("SB_TMA", 0) && env_int("SB_TMA_LOAD", 1);
  if (!enabled || !encode_tiled_fn()) return false;
  const int64_t es = c.elem_size;
  if (es != 4 && es != 8) return false;
  if (c.extent[0] * es < 512) return false;
  const sb_pitched &a = c.src;
  if ((uintptr_t(a.ptr) & 15) || (a.pitch & 15) || ((a.pitch * a.ysize) & 15) || (a.pitch % es)) return false;
  if (a.pitch * a.ysize >= (int64_t(1) << 40)) return false;
  const int64_t po = (c.src_pos[0] * es) & 15; // bytes between the aligned-down start and the payload
  const int64_t pre = po / es;
  if (c.src_pos[0] - pre < 0) return false;
  // payload chunk: a divisor of the row, a multiple of 16 bytes, box (pre + bx rounded up to 16 B) <= 256 elements
  unsigned bx = 0, bxa = 0;
  for (int64_t d = std::min<int64_t>(256, c.extent[0]); d >= 1; --d) {
    if (c.extent[0] % d || (d * es) % 16 || d * es < 256) continue;
    const int64_t box_bytes = (po + d * es + 15) & ~int64_t(15);
    if (box_bytes / es > 256) continue;
    bx = unsigned(d);
    bxa = unsigned(box_bytes / es);
    break;
  }
  if (0 == bx) return false;
  if (c.src_pos[0] - pre + c.extent[0] - bx + bxa > a.pitch / es) return false; // the last box must stay inside the row
  const int64_t rows = c.extent[1] * c.extent[2];
  if (rows >= (1 << 24) || c.extent[1] >= (1 << 24) || c.src_pos[2] + c.extent[2] >= (int64_t(1) << 20)) return false;
  const int si = tma_map_index(tb, c.src, es, bxa);
  if (si < 0) return false;
  sb::TmaSeg t{};
  t.smap = si;
  t.dmap = -1;
  t.sx0 = int(c.src_pos[0]);
  t.sy0 = int(c.src_pos[1]);
  t.sz0 = int(c.src_pos[2]);
  t.bx = bx;
  t.chunks_per_row = unsigned(c.extent[0] / bx);
  t.chunk_bytes = unsigned(bx * es); // payload bytes per chunk
  t.ny = unsigned(c.extent[1]);
  t.nz = unsigned(c.extent[2]);
  const unsigned bits = ceil_log2(t.ny);
  t.ny_shift = 24 + bits;
  t.ny_magic = ((1ull << t.ny_shift) + t.ny - 1) / t.ny;
  t.dst = static_cast<char *>(c.dst.ptr) + (c.dst_pos[2] * c.dst.ysize + c.dst_pos[1]) * c.dst.pitch + c.dst_pos[0] * es;
  t.dst_pitch = c.dst.pitch;
  t.dst_slice = c.dst.pitch * c.dst.ysize;
  t.pre = unsigned(pre);
  t.bxa = bxa;
  t.cstride = unsigned((bxa * es + 127) & ~int64_t(127));
  t.es = unsigned(es);
  unsigned long long align = (unsigned long long)(uintptr_t)t.dst | (unsigned long long)po | (unsigned long long)(bx * es);
  if (t.ny > 1) align |= (unsigned long long)t.dst_pitch;
  if (t.nz > 1) align |= (unsigned long long)t.dst_slice;
  t.vec = (align % 8 == 0 && es == 8) ? 8 : ((align % 8 == 0) ? 8 : 4);
  if (t.vec > 4 && (align % 8)) t.vec = 4;
  unsigned long long ph = ((unsigned long long)(uintptr_t)t.dst - (unsigned long long)po);
  if (t.ny > 1) ph |= (unsigned long long)t.dst_pitch;
  if (t.nz > 1) ph |= (unsigned long long)t.dst_slice;
  t.same_phase = (ph % 16 == 0) ? 1u : 0u;
  tb.segs.push_back(t);
  tb.kinds.push_back(2);
  return true;
}

void build_tma_tiles(const std::vector<sb::TmaSeg> &segs, const std::vector<int> &kinds, std::vector<sb::Tile> &tiles) {
  for (size_t si = 0; si < segs.size(); ++si) {
    const sb::TmaSeg &g = segs[si];
    if (kinds[si] == 2) {
      // all threads work on these: normal tile size
      const unsigned row_bytes = g.chunk_bytes * g.chunks_per_row;
      unsigned rows_per_tile = (2 * sb::kTileBytes) / row_bytes;
      if (rows_per_tile < 1) rows_per_tile = 1;
      const unsigned total = g.ny * g.nz;
      for (unsigned r = 0; r < total; r += rows_per_tile) {
        sb::Tile t{};
        t.seg = unsigned(si);
        t.row0 = r;
        t.nrows = (total - r < rows_per_tile) ? total - r : rows_per_tile;
        t.kind = 2;
        tiles.push_back(t);
      }
      continue;
    }
    const unsigned row_bytes = g.chunk_bytes * g.chunks_per_row;
    unsigned rows_per_tile = 65536u / row_bytes; // one thread drives a tile: make it big
    if (rows_per_tile < 1) rows_per_tile = 1;
    const unsigned total = g.ny * g.nz;
    for (unsigned r = 0; r < total; r += rows_per_tile) {
      sb::Tile t{};
      t.seg = unsigned(si);
      t.row0 = r;
      t.nrows = (total - r < rows_per_tile) ? total - r : rows_per_tile;
      t.kind = 1;
      tiles.push_back(t);
    }
  }
}

void build_tiles(const std::vector<sb::Seg> &segs, std::vector<sb::Tile> &tiles) {
  for (size_t si = 0; si < segs.size(); ++si) {
    const sb::Seg &g = segs[si];
    const unsigned rows_per_tile = sb::rows_per_tile_for(g.row_bytes);
    const unsigned total = g.ny * g.nz;
    for (unsigned r = 0; r < total; r += rows_per_tile) {
      sb::Tile t{};
      t.seg = unsigned(si);
      t.row0 = r;
      t.nrows = (total - r < rows_per_tile) ? total - r : rows_per_tile;
      t.kind = 0;
      tiles.push_back(t);
    }
  }
}

int env_int(const char *name, int dflt) {
  const char *s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

struct SlotTable {
  uint32_t *p[64];
};

__global__ void signal_kernel(const __grid_constant__ SlotTable slots, int n, uint32_t value) {
  // all earlier work of this stream is complete (stream order); publish it system-wide
  __threadfence_system();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(slots.p[i]), "r"(value) : "memory");
  }
}

__global__ void wait_kernel(const uint32_t *slots, int n, uint32_t value) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(slots + i) : "memory");
      if ((int32_t)(v - value) >= 0) break; // wrap-safe "v >= value"
      __nanosleep(64);
    } while (true);
  }
  __threadfence_system();
}

} // namespace

struct sb_copy_plan {
  int device = 0;
  sb::Seg *segs_dev = nullptr;
  sb::TmaSeg *tsegs_dev = nullptr;
  sb::TmaMaps *maps_host = nullptr; // passed by value as a __grid_constant__ kernel parameter
  unsigned ntma = 0;
  sb::Tile *tiles_dev = nullptr;
  unsigned ntiles = 0;
  unsigned nsegs = 0;
  int grid = 0;
  int64_t bytes = 0;
};

extern "C" {

const char *sb_last_error(void) { return g_err.c_str(); }
int sb_version(void) { return SB_VERSION; }
uint64_t sb_launch_count(void) { return g_launches.load(); }

// ----------------------------------------------------------------------------------------- geometry
int sb_halo_pos(const int64_t dir[3], const int64_t size[3], const int64_t radius27[27], int halo, int64_t out[3]) {
  if (!dir_ok(dir)) return fail(SB_ERR_INVALID, "direction components must be in -1..1");
  put(stencil::geom::halo_pos(d3(dir), d3(size), radius_of(radius27), halo != 0), out);
  return SB_OK;
}
int sb_halo_extent(const int64_t dir[3], const int64_t size[3], const int64_t radius27[27], int64_t out[3]) {
  if (!dir_ok(dir)) return fail(SB_ERR_INVALID, "direction components must be in -1..1");
  put(stencil::geom::halo_extent(d3(dir), d3(size), radius_of(radius27)), out);
  return SB_OK;
}
int sb_raw_size(const int64_t size[3], const int64_t radius27[27], int64_t out[3]) {
  put(stencil::geom::raw_size(d3(size), radius_of(radius27)), out);
  return SB_OK;
}
int sb_prime_factors(int64_t n, int64_t *out, int cap) {
  if (n < 0) return fail(SB_ERR_INVALID, "n must be >= 0");
  const std::vector<int64_t> f = prime_factors<int64_t>(n);
  if (int(f.size()) > cap) return fail(SB_ERR_INVALID, "output capacity %d too small for %zu factors", cap, f.size());
  for (size_t i = 0; i < f.size(); ++i) out[i] = f[i];
  return int(f.size());
}
int sb_rank_partition(const int64_t size[3], int64_t n, int64_t dim[3], int64_t base[3], int64_t rem[3]) {
  if (n < 1) return fail(SB_ERR_INVALID, "n must be >= 1");
  RankPartition p(d3(size), n);
  const Dim3 d = p.dim();
  put(d, dim);
  put(p.subdomain_size(Dim3(0, 0, 0)), base);
  put(d3(size) % d, rem);
  return SB_OK;
}
int sb_node_partition(const int64_t size[3], const int64_t radius27[27], int64_t nodes, int64_t gpus, int64_t sys_dim[3],
                      int64_t node_dim[3], int64_t base[3], int64_t rem[3]) {
  if (nodes < 1 || gpus < 1) return fail(SB_ERR_INVALID, "nodes and gpus must be >= 1");
  NodePartition p(d3(size), radius_of(radius27), nodes, gpus);
  put(p.sys_dim(), sys_dim);
  put(p.node_dim(), node_dim);
  put(p.subdomain_size(Dim3(0, 0, 0)), base);
  put(d3(size) % p.dim(), rem);
  return SB_OK;
}
int sb_subdomain_size(const int64_t base[3], const int64_t rem[3], const int64_t idx[3], int64_t out[3]) {
  stencil::detail::CutGrid g{d3(base), d3(rem)};
  put(g.size_of(d3(idx)), out);
  return SB_OK;
}
int sb_subdomain_origin(const int64_t base[3], const int64_t rem[3], const int64_t idx[3], int64_t out[3]) {
  stencil::detail::CutGrid g{d3(base), d3(rem)};
  put(g.origin_of(d3(idx)), out);
  return SB_OK;
}
int sb_interior(const int64_t lo[3], const int64_t hi[3], const int64_t radius27[27], int64_t int_lo[3], int64_t int_hi[3]) {
  const Rect3 in = stencil::geom::interior(Rect3(d3(lo), d3(hi)), radius_of(radius27));
  put(in.lo, int_lo);
  put(in.hi, int_hi);
  return SB_OK;
}
int sb_exterior(const int64_t lo[3], const int64_t hi[3], const int64_t radius27[27], int64_t *ext_lo, int64_t *ext_hi) {
  const std::vector<Rect3> slabs = stencil::geom::exterior(Rect3(d3(lo), d3(hi)), radius_of(radius27));
  for (size_t i = 0; i < slabs.size(); ++i) {
    put(slabs[i].lo, ext_lo + 3 * i);
    put(slabs[i].hi, ext_hi + 3 * i);
  }
  return int(slabs.size());
}

// ----------------------------------------------------------------------------------------- box copies
static int one_shot(const sb_box_copy &c, void *stream) {
  PtrDeviceGuard guard(c.src.ptr); // launch where the source lives
  std::vector<sb::Seg> segs;
  int rc = build_segments(c, segs);
  if (rc != SB_OK) return rc;
  for (const sb::Seg &g : segs) {
    sb::launch_box_copy_single(g, static_cast<cudaStream_t>(stream));
    ++g_launches;
  }
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_pack(void *dst, sb_pitched src, const int64_t pos[3], const int64_t extent[3], int64_t elem_size, void *stream) {
  sb_box_copy c{};
  c.dst = sb_pitched{dst, extent[0] * elem_size, extent[1]};
  c.src = src;
  for (int a = 0; a < 3; ++a) {
    c.src_pos[a] = pos[a];
    c.extent[a] = extent[a];
  }
  c.elem_size = elem_size;
  return one_shot(c, stream);
}

int sb_unpack(sb_pitched dst, const void *src, const int64_t pos[3], const int64_t extent[3], int64_t elem_size, void *stream) {
  sb_box_copy c{};
  c.dst = dst;
  c.src = sb_pitched{const_cast<void *>(src), extent[0] * elem_size, extent[1]};
  for (int a = 0; a < 3; ++a) {
    c.dst_pos[a] = pos[a];
    c.extent[a] = extent[a];
  }
  c.elem_size = elem_size;
  return one_shot(c, stream);
}

int sb_translate(sb_pitched dst, const int64_t dst_pos[3], sb_pitched src, const int64_t src_pos[3], const int64_t extent[3],
                 int64_t elem_size, void *stream) {
  sb_box_copy c{};
  c.dst = dst;
  c.src = src;
  for (int a = 0; a < 3; ++a) {
    c.dst_pos[a] = dst_pos[a];
    c.src_pos[a] = src_pos[a];
    c.extent[a] = extent[a];
  }
  c.elem_size = elem_size;
  return one_shot(c, stream);
}

int sb_copy_plan_create(sb_copy_plan **out, int device, const sb_box_copy *copies, int64_t n) {
  if (!out || (n > 0 && !copies) || n < 0) return fail(SB_ERR_INVALID, "bad arguments to sb_copy_plan_create");
  std::vector<sb::Seg> segs;
  TmaBuild tb;
  int64_t bytes = 0;
  for (int64_t i = 0; i < n; ++i) {
    bytes += copies[i].extent[0] * copies[i].extent[1] * copies[i].extent[2] * copies[i].elem_size;
    if (try_tma_segment(copies[i], tb, device)) continue;
    if (try_tma_load_segment(copies[i], tb)) continue;
    int rc = build_segments(copies[i], segs);
    if (rc != SB_OK) return rc;
  }
  std::vector<sb::Tile> tiles;
  build_tma_tiles(tb.segs, tb.kinds, tiles); // big tiles first: they take longest
  build_tiles(segs, tiles);

  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  sb::preload_box_copy_kernels();
  sb_copy_plan *p = new sb_copy_plan();
  p->device = device;
  p->bytes = bytes;
  p->nsegs = unsigned(segs.size());
  p->ntiles = unsigned(tiles.size());
  p->ntma = unsigned(tb.segs.size());
  if (p->ntiles) {
    if (!tb.segs.empty()) {
      static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
      p->maps_host = new sb::TmaMaps();
      std::memset(p->maps_host, 0, sizeof(sb::TmaMaps));
      for (size_t i = 0; i < tb.maps.size(); ++i) std::memcpy(&p->maps_host->m[i][0], &tb.maps[i], sizeof(CUtensorMap));
      SB_CUDA(cudaMalloc(&p->tsegs_dev, tb.segs.size() * sizeof(sb::TmaSeg)));
      SB_CUDA(cudaMemcpy(p->tsegs_dev, tb.segs.data(), tb.segs.size() * sizeof(sb::TmaSeg), cudaMemcpyHostToDevice));
    }
    SB_CUDA(cudaMalloc(&p->segs_dev, (segs.size() + 1) * sizeof(sb::Seg)));
    SB_CUDA(cudaMalloc(&p->tiles_dev, tiles.size() * sizeof(sb::Tile)));
    SB_CUDA(cudaMemcpy(p->segs_dev, segs.data(), segs.size() * sizeof(sb::Seg), cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(p->tiles_dev, tiles.data(), tiles.size() * sizeof(sb::Tile), cudaMemcpyHostToDevice));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int per_sm = env_int("SB_COPY_CTAS_PER_SM", 8);
    const long long cap = (long long)sms * per_sm;
    p->grid = int(p->ntiles < cap ? p->ntiles : cap);
  }
  *out = p;
  return SB_OK;
}

int sb_copy_plan_launch(sb_copy_plan *p, void *stream) {
  if (!p) return fail(SB_ERR_INVALID, "null plan");
  if (0 == p->ntiles) return SB_OK;
  DeviceGuard guard(p->device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", p->device);
  sb::launch_box_copy(p->segs_dev, p->tsegs_dev, p->maps_host, p->tiles_dev, p->ntiles, p->grid, static_cast<cudaStream_t>(stream));
  ++g_launches;
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int64_t sb_copy_plan_bytes(const sb_copy_plan *p) { return p ? p->bytes : 0; }
int64_t sb_copy_plan_num_tiles(const sb_copy_plan *p) { return p ? p->ntiles : 0; }
int64_t sb_copy_plan_num_tma_segments(const sb_copy_plan *p) { return p ? p->ntma : 0; }

int sb_copy_plan_destroy(sb_copy_plan *p) {
  if (!p) return SB_OK;
  DeviceGuard guard(p->device);
  if (p->segs_dev) cudaFree(p->segs_dev);
  if (p->tsegs_dev) cudaFree(p->tsegs_dev);
  delete p->maps_host;
  if (p->tiles_dev) cudaFree(p->tiles_dev);
  delete p;
  return SB_OK;
}

int sb_signal(uint32_t *const *remote_slots, int n, uint32_t value, int device, void *stream) {
  if (n <= 0) return SB_OK;
  if (n > 64) return fail(SB_ERR_INVALID, "at most 64 slots per signal");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SlotTable tab{};
  for (int i = 0; i < n; ++i) tab.p[i] = remote_slots[i];
  signal_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(tab, n, value);
  ++g_launches;
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_wait(const uint32_t *local_slots, int n, uint32_t value, int device, void *stream) {
  if (n <= 0) return SB_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  wait_kernel<<<1, 64, 0, static_cast<cudaStream_t>(stream)>>>(local_slots, n, value);
  ++g_launches;
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// ----------------------------------------------------------------------------------------- jacobi
static int to_alloc_box(const sb_pitched &a, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
                        const int64_t hi[3], int alo[3], int ahi[3]) {
  if (dtype_size != 4 && dtype_size != 8) return fail(SB_ERR_INVALID, "dtype_size must be 4 (float) or 8 (double)");
  if (!a.ptr || a.pitch <= 0 || a.ysize <= 0) return fail(SB_ERR_INVALID, "bad pitched pointer");
  for (int k = 0; k < 3; ++k) {
    const int64_t l = lo[k] - acc_origin[k], h = hi[k] - acc_origin[k];
    if (l < 0 || h > (1ll << 30)) return fail(SB_ERR_INVALID, "region outside the allocation on axis %d", k);
    alo[k] = int(l);
    ahi[k] = int(h);
  }
  return SB_OK;
}

static int jacobi_common(sb::JacobiParams &p, const sb_pitched &dst, const sb_pitched &src, int dtype_size,
                         const int64_t acc_origin[3], const int64_t clo[3], const int64_t chi[3]) {
  if (!dst.ptr || dst.pitch != src.pitch || dst.ysize != src.ysize)
    return fail(SB_ERR_INVALID, "dst and src must have the same pitch and ysize");
  p.dst = static_cast<char *>(dst.ptr);
  p.src = static_cast<const char *>(src.ptr);
  p.pitch = src.pitch;
  p.slice = src.pitch * src.ysize;
  p.raw[0] = int(src.pitch / dtype_size);
  p.raw[1] = int(src.ysize);
  for (int k = 0; k < 3; ++k) p.org[k] = int(acc_origin[k]);
  // sphere placement, bin/jacobi3d.cu:46-51
  const int64_t ex = chi[0] - clo[0];
  p.hot_x = int(clo[0] + ex / 3);
  p.cold_x = int(clo[0] + ex * 2 / 3);
  p.cy = int((clo[1] + chi[1]) / 2);
  p.cz = int((clo[2] + chi[2]) / 2);
  p.rad = int(ex / 10);
  p.zchunk = 0;
  return SB_OK;
}

int sb_jacobi3d_regions(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], int n, const int64_t *lo,
                        const int64_t *hi, const int64_t clo[3], const int64_t chi[3], void *stream) {
  if (n < 0 || n > 8) return fail(SB_ERR_INVALID, "between 0 and 8 regions per launch");
  PtrDeviceGuard guard(dst.ptr);
  sb::JacobiParams p{};
  sb::JacobiRegions r{};
  int zmax = 0;
  r.first[0] = 0;
  int m = 0;
  for (int i = 0; i < n; ++i) {
    int alo[3], ahi[3];
    int rc = to_alloc_box(src, dtype_size, acc_origin, lo + 3 * i, hi + 3 * i, alo, ahi);
    if (rc != SB_OK) return rc;
    long long cells = 1;
    for (int k = 0; k < 3; ++k) {
      if (ahi[k] > alo[k] && alo[k] < 1) return fail(SB_ERR_INVALID, "region needs one ghost cell below it on axis %d", k);
      cells *= (ahi[k] > alo[k]) ? (ahi[k] - alo[k]) : 0;
    }
    if (cells == 0) continue;
    if (cells >= (1ll << 32)) return fail(SB_ERR_INVALID, "region too large for sb_jacobi3d_regions");
    for (int k = 0; k < 3; ++k) {
      r.lo[m][k] = alo[k];
      r.ext[m][k] = ahi[k] - alo[k];
    }
    if (ahi[2] > zmax) zmax = ahi[2];
    r.first[m + 1] = r.first[m] + cells;
    ++m;
  }
  r.n = m;
  if (m == 0) return SB_OK;
  int rc = jacobi_common(p, dst, src, dtype_size, acc_origin, clo, chi);
  if (rc != SB_OK) return rc;
  p.raw[2] = zmax + 1;
  g_launches += uint64_t(sb::launch_jacobi_regions(p, r, dtype_size, static_cast<cudaStream_t>(stream)));
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_jacobi3d(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3],
                const int64_t hi[3], const int64_t clo[3], const int64_t chi[3], void *stream) {
  PtrDeviceGuard guard(dst.ptr);
  sb::JacobiParams p{};
  int rc = to_alloc_box(src, dtype_size, acc_origin, lo, hi, p.lo, p.hi);
  if (rc != SB_OK) return rc;
  for (int k = 0; k < 3; ++k) {
    if (p.lo[k] < 1 && p.hi[k] > p.lo[k]) return fail(SB_ERR_INVALID, "region needs one ghost cell below it on axis %d", k);
  }
  rc = jacobi_common(p, dst, src, dtype_size, acc_origin, clo, chi);
  if (rc != SB_OK) return rc;
  p.dst = static_cast<char *>(dst.ptr);
  p.src = static_cast<const char *>(src.ptr);
  p.pitch = src.pitch;
  p.slice = src.pitch * src.ysize;
  p.raw[0] = int(src.pitch / dtype_size);
  p.raw[1] = int(src.ysize);
  p.raw[2] = p.hi[2] + 1; // planes: the caller guarantees plane hi.z (one ghost plane above) exists
  const int n = sb::launch_jacobi(p, dtype_size, static_cast<cudaStream_t>(stream));
  g_launches += uint64_t(n);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_jacobi3d_fused(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3],
                      const int64_t clo[3], const int64_t chi[3], const sb_halo_push *push, void *stream) {
  return sb_jacobi3d_fused_sync(dst, src, dtype_size, acc_origin, lo, hi, clo, chi, push, nullptr, stream);
}

int sb_jacobi3d_fused_sync(sb_pitched dst, sb_pitched src, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3],
                           const int64_t clo[3], const int64_t chi[3], const sb_halo_push *push, const sb_step_sync *sync, void *stream) {
  if (!push) return fail(SB_ERR_INVALID, "null push table");
  PtrDeviceGuard guard(dst.ptr);
  sb::FusedSync fs{};
  if (sync) {
    for (int f = 0; f < 6; ++f) {
      fs.wait_row[f] = sync->wait_rows[f];
      fs.signal_row[f] = sync->signal_rows[f];
    }
    fs.wait_value = sync->wait_value;
    fs.signal_value = sync->signal_value;
  }
  sb::JacobiParams p{};
  int rc = to_alloc_box(src, dtype_size, acc_origin, lo, hi, p.lo, p.hi);
  if (rc != SB_OK) return rc;
  for (int k = 0; k < 3; ++k) {
    if (p.hi[k] <= p.lo[k]) return SB_OK;
    if (p.lo[k] < 1) return fail(SB_ERR_INVALID, "region needs one ghost cell below it on axis %d", k);
  }
  if (p.hi[0] - p.lo[0] < 16) return fail(SB_ERR_INVALID, "fused step needs at least 16 cells along x");
  rc = jacobi_common(p, dst, src, dtype_size, acc_origin, clo, chi);
  if (rc != SB_OK) return rc;
  p.raw[2] = p.hi[2] + 1;
  for (int d = 0; d < 6; ++d) {
    const sb_pitched &n = push->nbr[d];
    p.push_ptr[d] = nullptr;
    if (!n.ptr) continue;
    const long long npitch = n.pitch, nslice = n.pitch * n.ysize;
    const long long nraw[3] = {npitch / dtype_size, (long long)n.ysize, (long long)push->nbr_zsize[d]};
    const int axis = d / 2;
    if (axis == 0 && push->x_dense[d]) { // dense [y][z] array in the neighbour's memory, my allocation coordinates
      if (n.ysize < p.hi[1] || push->nbr_zsize[d] < p.hi[2]) return fail(SB_ERR_INVALID, "dense x array %d too small", d);
      p.push_ptr[d] = static_cast<char *>(n.ptr);
      p.push_pitch[d] = (long long)push->nbr_zsize[d] * dtype_size;
      p.push_slice[d] = dtype_size;
      p.xdense[d] = 1;
      continue;
    }
    // -axis neighbour: my first cells are its HIGH ghost (index raw-1); +axis neighbour: my last cells are its ghost 0
    const long long fixed = (d % 2 == 0) ? nraw[axis] - 1 : 0;
    if (nraw[axis] < 3) return fail(SB_ERR_INVALID, "neighbour %d allocation too small", d);
    const long long stride[3] = {(long long)dtype_size, npitch, nslice};
    p.push_ptr[d] = static_cast<char *>(n.ptr) + fixed * stride[axis];
    p.push_pitch[d] = npitch;
    p.push_slice[d] = nslice;
    // the two varying coordinates are MY allocation coordinates: they must exist in the neighbour's allocation
    for (int k = 0; k < 3; ++k) {
      if (k != axis && p.hi[k] > nraw[k]) return fail(SB_ERR_INVALID, "neighbour %d is smaller than this subdomain on axis %d", d, k);
    }
  }
  for (int sd = 0; sd < 2; ++sd) {
    p.xghost_ptr[sd] = static_cast<const char *>(push->x_recv[sd]);
    p.xghost_pitch[sd] = (long long)(p.hi[2] + 1) * dtype_size; // [y][z] over this subdomain's planes (raw z = hi.z + 1)
  }
  // A periodic self-neighbour on both sides of an axis needs neither ghost cells nor a push: the kernel reads the
  // opposite face of src in place (x: the edge lane's scalar, y: the row above / below a strip).  With alternating row
  // phases (FP32 rows not a multiple of 16 bytes) the wrapped row must have the parity of the ghost row it replaces.
  auto self = [&](int d) { return push->nbr[d].ptr == dst.ptr && push->nbr[d].pitch == dst.pitch && push->nbr[d].ysize == dst.ysize; };
  if (self(0) && self(1)) p.xwrap = 1; // a request: launch_jacobi_fused keeps the x pushes when the vector layout rules it out
  if (self(2) && self(3) && (src.pitch % 16 == 0 || (p.hi[1] - p.lo[1]) % 2 == 0)) p.ywrap = 1, p.push_ptr[2] = p.push_ptr[3] = nullptr;
  if (self(4) && self(5)) p.zwrap = 1, p.push_ptr[4] = p.push_ptr[5] = nullptr; // planes have one phase: nothing else to check
  const int n = sb::launch_jacobi_fused(p, fs, dtype_size, static_cast<cudaStream_t>(stream));
  if (n == -1) return fail(SB_ERR_INVALID, "a dense received x array needs a 16-byte aligned first compute cell and whole warp strips along x");
  if (n == -2) return fail(SB_ERR_INVALID, "more than %d z chunks or tile rows: too tall for the fused kernel's face groups", SB_FUSED_MAX_GROUPS);
  if (n < 0) return fail(SB_ERR_CUDA, "cannot allocate the face-group counters");
  g_launches += uint64_t(n);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_astaroth_substep(int step, const void *const in[8], void *const out[8], int dtype_size, const int64_t raw[3], const int64_t lo[3],
                        const int64_t hi[3], const sb_astaroth_params *params, int variant, void *stream) {
  if (!in || !out || !raw || !lo || !hi || !params) return fail(SB_ERR_INVALID, "null argument");
  if (step < 0 || step > 2) return fail(SB_ERR_INVALID, "substep %d (Williamson RK3 has substeps 0, 1, 2)", step);
  if (dtype_size != 4 && dtype_size != 8) return fail(SB_ERR_INVALID, "dtype_size %d (4 = float, 8 = double)", dtype_size);
  PtrDeviceGuard guard(out[0]);
  if (variant < 0 || variant > 5) return fail(SB_ERR_INVALID, "variant %d", variant);
  sb::AcFields f;
  for (int i = 0; i < sb::kAcFields; ++i) {
    if (!in[i] || !out[i]) return fail(SB_ERR_INVALID, "field %d is null", i);
    f.in[i] = in[i];
    f.out[i] = out[i];
  }
  int ilo[3], ihi[3];
  for (int k = 0; k < 3; ++k) {
    if (raw[k] <= 0 || raw[k] >= (1ll << 31)) return fail(SB_ERR_INVALID, "raw size");
    if (hi[k] > lo[k] && (lo[k] < 3 || hi[k] > raw[k] - 3))
      return fail(SB_ERR_INVALID, "box [%lld,%lld) on axis %d needs 3 allocated cells on each side (raw %lld)", (long long)lo[k], (long long)hi[k], k,
                  (long long)raw[k]);
    ilo[k] = int(lo[k]);
    ihi[k] = int(hi[k] > lo[k] ? hi[k] : lo[k]);
  }
  sb::AcParams p;
  static_assert(sizeof(sb::AcParams) == sizeof(sb_astaroth_params), "same layout");
  memcpy(&p, params, sizeof(p));
  const int n = sb::launch_astaroth_substep(step, f, dtype_size, raw[0], raw[1], raw[2], ilo, ihi, p, variant, static_cast<cudaStream_t>(stream));
  if (n < 0) return fail(SB_ERR_INVALID, "astaroth substep rejected (code %d)", n);
  g_launches += uint64_t(n);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_fill(sb_pitched dst, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3], double value,
            void *stream) {
  PtrDeviceGuard guard(dst.ptr);
  int alo[3], ahi[3];
  int rc = to_alloc_box(dst, dtype_size, acc_origin, lo, hi, alo, ahi);
  if (rc != SB_OK) return rc;
  g_launches += uint64_t(sb::launch_fill(static_cast<char *>(dst.ptr), dst.pitch, dst.pitch * dst.ysize, alo, ahi, dtype_size, value,
                                         static_cast<cudaStream_t>(stream)));
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int sb_sqdiff(sb_pitched a, sb_pitched b, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3],
              double *out_dev, void *stream) {
  PtrDeviceGuard guard(a.ptr);
  int alo[3], ahi[3];
  int rc = to_alloc_box(a, dtype_size, acc_origin, lo, hi, alo, ahi);
  if (rc != SB_OK) return rc;
  if (b.pitch != a.pitch || b.ysize != a.ysize || !b.ptr || !out_dev) return fail(SB_ERR_INVALID, "mismatched operands");
  g_launches += uint64_t(sb::launch_sqdiff(static_cast<const char *>(a.ptr), static_cast<const char *>(b.ptr), a.pitch,
                                           a.pitch * a.ysize, alo, ahi, dtype_size, out_dev, static_cast<cudaStream_t>(stream)));
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// ----------------------------------------------------------------------------------------- reductions
// SM count of a device (the reduction grid is a fixed multiple of it), cached: it is read on every launch
static int sm_count(int device, int *out) {
  static std::atomic<int> cache[64];
  if (device >= 0 && device < 64 && cache[device].load() > 0) {
    *out = cache[device].load();
    return SB_OK;
  }
  int n = 0;
  SB_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
  if (device >= 0 && device < 64) cache[device].store(n);
  *out = n;
  return SB_OK;
}

int64_t sb_reduce_workspace_bytes(int device) {
  int n = 0;
  const int rc = sm_count(device, &n);
  return rc != SB_OK ? int64_t(rc) : sb::reduce_workspace_bytes(n);
}

int sb_reduce(int kind, const sb_pitched *operands, int dtype_size, const int64_t acc_origin[3], const int64_t lo[3], const int64_t hi[3],
              void *workspace, void *stream) {
  const int n = sb::reduce_num_operands(kind);
  if (n == 0) return fail(SB_ERR_INVALID, "reduction kind %d (0 VALUE, 1 DIFF, 2 VECTOR, 3 EXP, 4 ALFVEN)", kind);
  if (!operands || !acc_origin || !lo || !hi || !workspace) return fail(SB_ERR_INVALID, "null argument to sb_reduce");
  if (reinterpret_cast<uintptr_t>(workspace) % 16 != 0) return fail(SB_ERR_INVALID, "workspace must be 16-byte aligned");
  int alo[3], ahi[3];
  int rc = to_alloc_box(operands[0], dtype_size, acc_origin, lo, hi, alo, ahi);
  if (rc != SB_OK) return rc;
  const char *ops[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int o = 0; o < n; ++o) {
    const sb_pitched &p = operands[o];
    if (!p.ptr) return fail(SB_ERR_INVALID, "operand %d is null", o);
    if (p.pitch != operands[0].pitch || p.ysize != operands[0].ysize)
      return fail(SB_ERR_INVALID, "operand %d: pitch/ysize (%lld, %lld) differ from operand 0 (%lld, %lld)", o, (long long)p.pitch,
                  (long long)p.ysize, (long long)operands[0].pitch, (long long)operands[0].ysize);
    if (reinterpret_cast<uintptr_t>(p.ptr) % unsigned(dtype_size) != 0) return fail(SB_ERR_INVALID, "operand %d is not aligned to its element size", o);
    ops[o] = static_cast<const char *>(p.ptr);
  }
  if (operands[0].pitch % dtype_size != 0) return fail(SB_ERR_INVALID, "pitch %lld is not a multiple of the element size", (long long)operands[0].pitch);
  for (int k = 0; k < 3; ++k)
    if (ahi[k] < alo[k]) return fail(SB_ERR_INVALID, "box has hi < lo on axis %d", k);
  const bool empty = ahi[0] == alo[0] || ahi[1] == alo[1] || ahi[2] == alo[2];
  if (!empty && ahi[0] > operands[0].pitch / dtype_size) return fail(SB_ERR_INVALID, "box ends at x = %d, past the row of %lld elements", ahi[0], (long long)(operands[0].pitch / dtype_size));
  if (!empty && ahi[1] > operands[0].ysize) return fail(SB_ERR_INVALID, "box ends at y = %d, past the %lld rows of a plane", ahi[1], (long long)operands[0].ysize);
  if (int64_t(ahi[1] - alo[1]) * int64_t(ahi[2] - alo[2]) >= (1ll << 31)) return fail(SB_ERR_INVALID, "box has 2^31 rows or more");
  PtrDeviceGuard guard(operands[0].ptr);
  int dev = 0, sms = 0;
  SB_CUDA(cudaGetDevice(&dev));
  rc = sm_count(dev, &sms);
  if (rc != SB_OK) return rc;
  g_launches += uint64_t(sb::launch_reduce(kind, ops, dtype_size, operands[0].pitch, operands[0].pitch * operands[0].ysize, alo, ahi, workspace,
                                           sms, static_cast<cudaStream_t>(stream)));
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// ----------------------------------------------------------------------------------------- device plumbing
int sb_device_count(int *count) {
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) {
    *count = 0;
    cudaGetLastError();
    return fail(SB_ERR_NOGPU, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
  }
  return SB_OK;
}

int sb_malloc(void **ptr, size_t bytes, int device) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaMalloc(ptr, bytes));
  return SB_OK;
}

int sb_free(void *ptr, int device) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaFree(ptr));
  return SB_OK;
}

int sb_memset(void *ptr, int value, size_t bytes, int device, void *stream) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaMemsetAsync(ptr, value, bytes, static_cast<cudaStream_t>(stream)));
  return SB_OK;
}

int sb_memcpy(void *dst, const void *src, size_t bytes, int device, void *stream) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, static_cast<cudaStream_t>(stream)));
  return SB_OK;
}

int sb_stream_sync(int device, void *stream) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return SB_OK;
}

int sb_device_sync(int device) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaDeviceSynchronize());
  return SB_OK;
}

int sb_enable_peer(int src_device, int dst_device, int *ok) {
  *ok = 0;
  if (src_device == dst_device) {
    *ok = 1;
    return SB_OK;
  }
  int can = 0;
  SB_CUDA(cudaDeviceCanAccessPeer(&can, src_device, dst_device));
  if (!can) return SB_OK;
  DeviceGuard guard(src_device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", src_device);
  cudaError_t e = cudaDeviceEnablePeerAccess(dst_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    e = cudaSuccess;
  }
  SB_CUDA(e);
  *ok = 1;
  return SB_OK;
}

int sb_ipc_export(void *ptr, void *handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  SB_CUDA(cudaIpcGetMemHandle(&h, ptr));
  std::memcpy(handle64, &h, sizeof(h));
  return SB_OK;
}

int sb_ipc_import(const void *handle64, int device, void **ptr) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle64, sizeof(h));
  SB_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return SB_OK;
}

int sb_ipc_close(void *ptr, int device) {
  DeviceGuard guard(device);
  if (!guard.ok) return fail(SB_ERR_NOGPU, "cannot select CUDA device %d", device);
  SB_CUDA(cudaIpcCloseMemHandle(ptr));
  return SB_OK;
}

} // extern "C"
