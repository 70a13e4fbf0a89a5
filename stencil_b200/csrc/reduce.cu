// Deterministic one-pass reductions over a box of 1-4 strided allocations (see reduce.cuh, DESIGN.md section 2.5).
//
// Work split: rows (y, z) of the box go round-robin to warps (thin boxes: to threads) by a fixed function of the grid,
// and the grid is a fixed multiple of the SM count, so every lane always sees the same cells in the same order.  Lanes
// accumulate in registers, CTAs reduce through a fixed shuffle tree and write one partial each into the workspace; the
// last CTA to take an integer ticket combines the partials by a fixed tree over CTA indices.  No floating-point atomics.
#include "reduce.cuh"

#include <type_traits>

namespace sb {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kCtasPerSm = 4;
constexpr double kFourPi = 4.0 * 3.14159265358979323846; // AcReal(4.0) * M_PI, astaroth/reductions.cuh:47-50

template <int K> struct NumOps {
  static constexpr int n = (K == kReduceValue || K == kReduceExp) ? 1 : K == kReduceDiff ? 2 : K == kReduceVector ? 3 : 4;
};

struct ReduceArgs {
  const char *op[4]; // allocation bases
  long long pitch, slice;
  int lo[3]; // allocation-relative first cell
  int ex, ey;
  unsigned rows; // ey * ez (0: empty box)
  double *ws;
};

__device__ __forceinline__ double pos_inf() { return __longlong_as_double(0x7ff0000000000000ll); }

// min / max that keep a NaN once they have seen one (fmin / fmax would drop it: a blow-up must show)
__device__ __forceinline__ double nan_min(double m, double f) { return (f < m || f != f) ? f : m; }
__device__ __forceinline__ double nan_max(double m, double f) { return (f > m || f != f) ? f : m; }

struct Acc {
  double mn, mx, s, s2;
  __device__ __forceinline__ void init() {
    mn = pos_inf();
    mx = -pos_inf();
    s = 0.0;
    s2 = 0.0;
  }
  __device__ __forceinline__ void add(double f, double g) {
    mn = nan_min(mn, f);
    mx = nan_max(mx, f);
    s = __dadd_rn(s, f);
    s2 = __dadd_rn(s2, g);
  }
  __device__ __forceinline__ void merge(double omn, double omx, double os, double os2) {
    mn = nan_min(mn, omn);
    mx = nan_max(mx, omx);
    s = __dadd_rn(s, os);
    s2 = __dadd_rn(s2, os2);
  }
  __device__ __forceinline__ void shfl_merge(int o) {
    merge(__shfl_xor_sync(0xffffffffu, mn, o), __shfl_xor_sync(0xffffffffu, mx, o), __shfl_xor_sync(0xffffffffu, s, o),
          __shfl_xor_sync(0xffffffffu, s2, o));
  }
};

// The filters of astaroth/reductions.cuh:18-52 in FP64 with every rounding explicit (no FMA contraction), in the order
// of the table in DESIGN.md section 2.5: f = value for min / max / sum, g = square for sum2.
template <int K> __device__ __forceinline__ void cell(Acc &acc, double a, double b, double c, double d) {
  if constexpr (K == kReduceValue) {
    acc.add(a, __dmul_rn(a, a));
  } else if constexpr (K == kReduceDiff) {
    const double t = __dsub_rn(a, b);
    acc.add(t, __dmul_rn(t, t));
  } else if constexpr (K == kReduceVector) {
    const double s = __dadd_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), __dmul_rn(c, c));
    acc.add(__dsqrt_rn(s), s);
  } else if constexpr (K == kReduceExp) {
    const double e = exp(a);
    acc.add(e, __dmul_rn(e, e));
  } else {
    const double s = __dadd_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), __dmul_rn(c, c));
    const double den = __dmul_rn(kFourPi, exp(d));
    acc.add(__ddiv_rn(__dsqrt_rn(s), __dsqrt_rn(den)), __ddiv_rn(s, den));
  }
}

template <typename T> __device__ __forceinline__ double ld(const char *p) { return double(__ldg(reinterpret_cast<const T *>(p))); }

template <typename T, int K, int N> __device__ __forceinline__ void cell_at(Acc &acc, const char *const (&p)[N], int x) {
  const long long o = (long long)x * (long long)sizeof(T);
  cell<K>(acc, ld<T>(p[0] + o), N > 1 ? ld<T>(p[N > 1 ? 1 : 0] + o) : 0.0, N > 2 ? ld<T>(p[N > 2 ? 2 : 0] + o) : 0.0,
          N > 3 ? ld<T>(p[N > 3 ? 3 : 0] + o) : 0.0);
}

__device__ __forceinline__ double comp(const double2 &v, int c) { return c == 0 ? v.x : v.y; }
__device__ __forceinline__ double comp(const float4 &v, int c) { return double(c == 0 ? v.x : c == 1 ? v.y : c == 2 ? v.z : v.w); }

template <typename T, int K>
__global__ void __launch_bounds__(kThreads, K == kReduceValue ? kCtasPerSm : kCtasPerSm / 2) reduce_kernel(const __grid_constant__ ReduceArgs a) {
  constexpr int N = NumOps<K>::n;
  constexpr int V = 16 / int(sizeof(T));
  constexpr int U = N == 1 ? 8 : 4; // independent 16-byte loads in flight per thread and operand
  using VT = typename std::conditional<sizeof(T) == 8, double2, float4>::type;
  const int lane = threadIdx.x & 31;
  Acc acc;
  acc.init();
  auto row_ptrs = [&](unsigned r, const char *(&p)[N]) {
    const unsigned y = r % unsigned(a.ey), z = r / unsigned(a.ey);
    const long long off = (long long)(a.lo[2] + int(z)) * a.slice + (long long)(a.lo[1] + int(y)) * a.pitch + (long long)a.lo[0] * (long long)sizeof(T);
#pragma unroll
    for (int o = 0; o < N; ++o) p[o] = a.op[o] + off;
  };
  if (a.ex * int(sizeof(T)) < 32) {
    // thin box (the exterior x slabs): a warp would leave most lanes idle on a row, so one thread takes a whole row
    for (unsigned r = blockIdx.x * kThreads + threadIdx.x; r < a.rows; r += gridDim.x * kThreads) {
      const char *p[N];
      row_ptrs(r, p);
      for (int x = 0; x < a.ex; ++x) cell_at<T, K, N>(acc, p, x);
    }
  } else {
    for (unsigned r = blockIdx.x * kWarps + (threadIdx.x >> 5); r < a.rows; r += gridDim.x * kWarps) {
      const char *p[N];
      row_ptrs(r, p);
      // every row has its own 16-byte phase (FP32 radius 1: 2056-byte rows alternate); the vector path needs the same
      // phase in every operand
      const unsigned ph = unsigned(reinterpret_cast<uintptr_t>(p[0])) & 15u;
      bool same = true;
#pragma unroll
      for (int o = 1; o < N; ++o) same = same && (unsigned(reinterpret_cast<uintptr_t>(p[o])) & 15u) == ph;
      if (!same) {
        for (int x = lane; x < a.ex; x += 32) cell_at<T, K, N>(acc, p, x);
        continue;
      }
      const int head = min(a.ex, int(((16u - ph) & 15u) / unsigned(sizeof(T)))); // scalar cells before the first vector
      if (lane < head) cell_at<T, K, N>(acc, p, lane);
      const int nvec = (a.ex - head) / V;
      const VT *vp[N];
#pragma unroll
      for (int o = 0; o < N; ++o) vp[o] = reinterpret_cast<const VT *>(p[o] + (long long)head * (long long)sizeof(T));
      for (int b = 0; b < nvec; b += 32 * U) {
        VT buf[N][U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int i = b + u * 32 + lane;
          if (i < nvec) {
#pragma unroll
            for (int o = 0; o < N; ++o) buf[o][u] = __ldg(vp[o] + i);
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (b + u * 32 + lane < nvec) {
#pragma unroll
            for (int c = 0; c < V; ++c)
              cell<K>(acc, comp(buf[0][u], c), N > 1 ? comp(buf[N > 1 ? 1 : 0][u], c) : 0.0, N > 2 ? comp(buf[N > 2 ? 2 : 0][u], c) : 0.0,
                      N > 3 ? comp(buf[N > 3 ? 3 : 0][u], c) : 0.0);
          }
        }
      }
      const int t0 = head + nvec * V; // scalar tail
      if (lane < a.ex - t0) cell_at<T, K, N>(acc, p, t0 + lane);
    }
  }

  // CTA partial: shuffle tree, then the warps in index order
  __shared__ double sh[kWarps][4];
  __shared__ bool last;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc.shfl_merge(o);
  if (lane == 0) {
    sh[threadIdx.x >> 5][0] = acc.mn;
    sh[threadIdx.x >> 5][1] = acc.mx;
    sh[threadIdx.x >> 5][2] = acc.s;
    sh[threadIdx.x >> 5][3] = acc.s2;
  }
  __syncthreads();
  double *const part = a.ws + 8;
  unsigned *const ticket = reinterpret_cast<unsigned *>(a.ws + 4);
  if (threadIdx.x == 0) {
    Acc c;
    c.init();
    for (int w = 0; w < kWarps; ++w) c.merge(sh[w][0], sh[w][1], sh[w][2], sh[w][3]);
    double *mine = part + 4ll * blockIdx.x;
    mine[0] = c.mn;
    mine[1] = c.mx;
    mine[2] = c.s;
    mine[3] = c.s2;
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;

  // the last CTA: every other partial is visible (written before its CTA's fence and ticket)
  __threadfence();
  acc.init();
  for (unsigned i = threadIdx.x; i < gridDim.x; i += kThreads) {
    const double *q = part + 4ll * i;
    acc.merge(__ldcg(q), __ldcg(q + 1), __ldcg(q + 2), __ldcg(q + 3));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc.shfl_merge(o);
  if (lane == 0) {
    sh[threadIdx.x >> 5][0] = acc.mn;
    sh[threadIdx.x >> 5][1] = acc.mx;
    sh[threadIdx.x >> 5][2] = acc.s;
    sh[threadIdx.x >> 5][3] = acc.s2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Acc c;
    c.init();
    for (int w = 0; w < kWarps; ++w) c.merge(sh[w][0], sh[w][1], sh[w][2], sh[w][3]);
    a.ws[0] = c.mn;
    a.ws[1] = c.mx;
    a.ws[2] = c.s;
    a.ws[3] = c.s2;
    *ticket = 0u; // ready for the next launch on this workspace
  }
}

template <typename T> void go(int kind, const ReduceArgs &a, unsigned grid, cudaStream_t stream) {
  switch (kind) {
  case kReduceValue:
    reduce_kernel<T, kReduceValue><<<grid, kThreads, 0, stream>>>(a);
    break;
  case kReduceDiff:
    reduce_kernel<T, kReduceDiff><<<grid, kThreads, 0, stream>>>(a);
    break;
  case kReduceVector:
    reduce_kernel<T, kReduceVector><<<grid, kThreads, 0, stream>>>(a);
    break;
  case kReduceExp:
    reduce_kernel<T, kReduceExp><<<grid, kThreads, 0, stream>>>(a);
    break;
  default:
    reduce_kernel<T, kReduceAlfven><<<grid, kThreads, 0, stream>>>(a);
    break;
  }
}

} // namespace

int reduce_num_operands(int kind) {
  switch (kind) {
  case kReduceValue:
  case kReduceExp:
    return 1;
  case kReduceDiff:
    return 2;
  case kReduceVector:
    return 3;
  case kReduceAlfven:
    return 4;
  default:
    return 0;
  }
}

int64_t reduce_workspace_bytes(int num_sms) { return 64 + 32ll * kCtasPerSm * num_sms; }

int launch_reduce(int kind, const char *const ops[4], int dtype_size, long long pitch, long long slice, const int lo[3],
                  const int hi[3], void *workspace, int num_sms, cudaStream_t stream) {
  ReduceArgs a;
  const int n = reduce_num_operands(kind);
  for (int o = 0; o < 4; ++o) a.op[o] = ops[o < n ? o : 0];
  a.pitch = pitch;
  a.slice = slice;
  for (int k = 0; k < 3; ++k) a.lo[k] = lo[k];
  const int ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
  const bool empty = ex <= 0 || ey <= 0 || ez <= 0;
  a.ex = empty ? 0 : ex;
  a.ey = empty ? 1 : ey;
  a.rows = empty ? 0u : unsigned(ey) * unsigned(ez);
  a.ws = static_cast<double *>(workspace);
  const unsigned grid = unsigned(kCtasPerSm * num_sms);
  if (dtype_size == 4)
    go<float>(kind, a, grid, stream);
  else
    go<double>(kind, a, grid, stream);
  return 1;
}

} // namespace sb
