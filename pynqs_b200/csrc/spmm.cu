// spmm.cu -- Y = H X for a CSR matrix H (the layout pynqs_hamiltonian_emit writes: crow int64 [n + 1], col int64, val
// float64) and a row-major float64 block X [N, K] (leading dimension ldx), Y [n, K] (ldy), K = 1 .. 8.
//
// Deterministic: Y[i, c] is summed in an order fixed by the length of row i alone -- which lane takes which entry, relative
// to the row's start, and the shuffle tree that combines the lanes -- never by the grid, the stream or float atomics.
// Rows are classed by length, and each class has one summation tree:
//   short  (<= kShortRow entries): 8 lanes per row, four rows per warp at a time; lane j takes entries j, j + 8, ...;
//   medium (<= kLongRow):          a whole warp per row; lane j takes entries j, j + 32, ...;
//   long   (>  kLongRow):          a CTA of kLongThreads per row; thread t takes entries t, t + 256, ..., the warps' sums
//                                  are added in warp order.
// Short and medium rows are taken by spmm_rows_kernel, long rows by spmm_long_kernel (which skips the others).  Neither needs
// a work list: a warp (CTA) checks 32 (256) candidate rows with one load per lane and takes the ones of its class.  The
// candidates of one warp are spaced a grid apart, so rows of similar length that sit together in the matrix (the samples
// of a heavy beta string) spread over the grid.
#include "common.cuh"

namespace pynqs {

constexpr int kRowThreads = 128;
constexpr int kShortRow = 64;
constexpr int kLongRow = 2048;
constexpr int kLongThreads = 256;
// persistent grids: 16 CTAs of 128 threads, or 4 of 256, per SM of a B200 (148 SMs)
constexpr long long kRowWarpsCap = 148LL * 16 * (kRowThreads / 32);
constexpr long long kLongCtasCap = 148LL * 4;

template <int K>
__device__ __forceinline__ void accumulate(double (&acc)[K], const long long *__restrict__ col, const double *__restrict__ val,
                                           const double *__restrict__ X, long long ldx, long long p, long long end, int step) {
  // four entries in flight per lane (two for wide blocks, which load K values each)
#pragma unroll(K <= 4 ? 4 : 2)
  for (; p < end; p += step) {
    const double v = __ldg(val + p);
    const double *x = X + __ldg(col + p) * ldx;
#pragma unroll
    for (int c = 0; c < K; ++c) acc[c] = fma(v, __ldg(x + c), acc[c]);
  }
}

// butterfly over the lanes of an aligned group of `width` lanes: every lane ends with the same bits (x + y == y + x)
template <int K>
__device__ __forceinline__ void group_sum(double (&acc)[K], int width) {
  for (int o = width >> 1; o > 0; o >>= 1) {
#pragma unroll
    for (int c = 0; c < K; ++c) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], o);
  }
}

// lane j < K of the group writes column j (a select, so that acc stays in registers)
template <int K>
__device__ __forceinline__ void store_row(const double (&acc)[K], double *__restrict__ y, int j) {
  double out = 0.0;
#pragma unroll
  for (int c = 0; c < K; ++c)
    if (c == j) out = acc[c];
  if (j < K) y[j] = out;
}

template <int K>
__global__ void __launch_bounds__(kRowThreads) spmm_rows_kernel(const long long *__restrict__ crow, const long long *__restrict__ col,
                                                                const double *__restrict__ val, long long n, const double *__restrict__ X,
                                                                long long ldx, double *__restrict__ Y, long long ldy) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (kRowThreads / 32);
  const long long w = (long long)blockIdx.x * (kRowThreads / 32) + (threadIdx.x >> 5);
  const int grp = lane >> 3, j = lane & 7;
  for (long long q = 0; w + nwarps * 32 * q < n; ++q) {
    const long long r = w + nwarps * (32 * q + lane);  // this lane's candidate row
    long long b = 0, e = 0;
    if (r < n) {
      b = __ldg(crow + r);
      e = __ldg(crow + r + 1);
    }
    u32 shorts = __ballot_sync(0xffffffffu, r < n && e - b <= kShortRow);
    u32 mediums = __ballot_sync(0xffffffffu, r < n && e - b > kShortRow && e - b <= kLongRow);
    while (shorts) {  // four rows at a time: group g takes the g-th remaining one
      u32 m = shorts;
      for (int i = 0; i < grp; ++i) m &= m - 1u;
      const int src = m ? __ffs(m) - 1 : 0;
      const long long rb = __shfl_sync(0xffffffffu, b, src), re = __shfl_sync(0xffffffffu, e, src);
      double acc[K];
#pragma unroll
      for (int c = 0; c < K; ++c) acc[c] = 0.0;
      if (m) accumulate<K>(acc, col, val, X, ldx, rb + j, re, 8);
      group_sum<K>(acc, 8);
      if (m) store_row<K>(acc, Y + (w + nwarps * (32 * q + src)) * ldy, j);
      for (int i = 0; i < 4 && shorts; ++i) shorts &= shorts - 1u;
    }
    while (mediums) {
      const int src = __ffs(mediums) - 1;
      mediums &= mediums - 1u;
      const long long rb = __shfl_sync(0xffffffffu, b, src), re = __shfl_sync(0xffffffffu, e, src);
      double acc[K];
#pragma unroll
      for (int c = 0; c < K; ++c) acc[c] = 0.0;
      accumulate<K>(acc, col, val, X, ldx, rb + lane, re, 32);
      group_sum<K>(acc, 32);
      store_row<K>(acc, Y + (w + nwarps * (32 * q + src)) * ldy, lane);
    }
  }
}

template <int K>
__global__ void __launch_bounds__(kLongThreads) spmm_long_kernel(const long long *__restrict__ crow, const long long *__restrict__ col,
                                                                 const double *__restrict__ val, long long n, const double *__restrict__ X,
                                                                 long long ldx, double *__restrict__ Y, long long ldy) {
  constexpr int kWarps = kLongThreads / 32;
  __shared__ long long s_row[kLongThreads];
  __shared__ int s_cnt;
  __shared__ double s_part[kWarps][K];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const long long G = gridDim.x;
  for (long long q = 0; blockIdx.x + G * kLongThreads * q < n; ++q) {
    if (t == 0) s_cnt = 0;
    __syncthreads();
    const long long r = blockIdx.x + G * (kLongThreads * q + t);
    if (r < n && __ldg(crow + r + 1) - __ldg(crow + r) > kLongRow) s_row[atomicAdd(&s_cnt, 1)] = r;  // the list's order is immaterial
    __syncthreads();
    const int cnt = s_cnt;
    for (int i = 0; i < cnt; ++i) {
      const long long row = s_row[i];
      double acc[K];
#pragma unroll
      for (int c = 0; c < K; ++c) acc[c] = 0.0;
      accumulate<K>(acc, col, val, X, ldx, __ldg(crow + row) + t, __ldg(crow + row + 1), kLongThreads);
      group_sum<K>(acc, 32);
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < K; ++c) s_part[warp][c] = acc[c];
      }
      __syncthreads();
      if (t < K) {
        double s = s_part[0][t];
#pragma unroll
        for (int v = 1; v < kWarps; ++v) s += s_part[v][t];
        Y[row * ldy + t] = s;
      }
      __syncthreads();
    }
  }
}

template <int K>
static void launch_k(const long long *crow, const long long *col, const double *val, long long n, const double *X, long long ldx, double *Y,
                     long long ldy, cudaStream_t st) {
  // up to one warp per row: a matrix of a few thousand long rows still spreads over the whole GPU
  const long long warps = n < kRowWarpsCap ? n : kRowWarpsCap;
  const unsigned rows_grid = (unsigned)((warps + kRowThreads / 32 - 1) / (kRowThreads / 32));
  spmm_rows_kernel<K><<<rows_grid, kRowThreads, 0, st>>>(crow, col, val, n, X, ldx, Y, ldy);
  const unsigned long_grid = (unsigned)(n < kLongCtasCap ? n : kLongCtasCap);
  spmm_long_kernel<K><<<long_grid, kLongThreads, 0, st>>>(crow, col, val, n, X, ldx, Y, ldy);
  count_launch(2);
}

// n > 0; arguments checked by pynqs_csr_spmm
int launch_csr_spmm(const long long *crow, const long long *col, const double *val, long long n, const double *X, long long ldx, int k,
                    double *Y, long long ldy, cudaStream_t st) {
  switch (k) {
    case 1: launch_k<1>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 2: launch_k<2>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 3: launch_k<3>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 4: launch_k<4>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 5: launch_k<5>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 6: launch_k<6>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 7: launch_k<7>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    case 8: launch_k<8>(crow, col, val, n, X, ldx, Y, ldy, st); break;
    default: set_error("csr_spmm: k = %d not in [1, 8]", k); return 1;
  }
  return check_launch("spmm_rows_kernel / spmm_long_kernel");
}

}  // namespace pynqs
