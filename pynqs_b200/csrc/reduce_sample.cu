// reduce_sample.cu -- the stochastic / semi-stochastic branch of the REDUCE method (vmc/energy/eloc.py:257-283):
//
//   hij = |Hmat| with the entries >= eps zeroed (eps > 0: semi-stochastic; those entries are kept exactly; eps is rounded
//         to the integrals' dtype first, as torch compares in the tensor's dtype)
//   p[n, m] = hij / hij.sum(1);   eps_sample draws per sample from p (torch.multinomial, with replacement)
//   Hmat[n, m] <- (count[n, m] / eps_sample) * Hmat[n, m] / p[n, m]     for the drawn (n, m)
//   kept set = {|Hmat| >= eps}  U  {drawn}
//
// The reference materialises comb [n, M, 8L], Hmat [n, M], p [n, M] and the [n, eps_sample] draws.  Here one CTA per
// sample walks the M rows three times without storing them (sum of the sub-eps magnitudes; locate the draws and count;
// locate again and emit): a draw is a point t = u * S in [0, S), S = sum of the sample's sub-eps |H|, and lands on the row
// whose running-sum interval [before, before + |H|) holds it.  The eps_sample points of a sample are sorted in shared
// memory, so a row finds its count with two binary searches.  The re-weighted element of a drawn row is
// sign(H) * S * count / eps_sample (H / p = sign(H) * S), the kept rows keep H.
//
// Random numbers: Philox4x32-10 keyed by the caller's seed, counter = (sample, draw) -- reproducible, independent of the
// launch geometry, but NOT torch's multinomial stream (which differs between its own CPU and CUDA back ends): parity with
// the reference is statistical for seeded runs and exact when the caller supplies the draws (`draws`: row indices
// [n, eps_sample], what torch.multinomial returned), which is how the tests pin it.
//
// Output order per sample: kept rows (ascending m), then drawn rows (ascending m); flat indices s * M + m like the
// reference's gt_eps_idx.  Rows are evaluated with decode_exc / exc_element on the packed integrals (the arithmetic of
// get_comb_hij_fused, bit-identical values).
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace pynqs {

constexpr int kRsThreads = 256;

struct Philox {
  u32 k0, k1;
  __device__ __forceinline__ uint4 operator()(u32 c0, u32 c1, u32 c2, u32 c3) const {
    u32 a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const u32 hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const u32 hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      const u32 n0 = hi1 ^ c1 ^ a, n1 = lo1, n2 = hi0 ^ c3 ^ b, n3 = lo0;
      c0 = n0;
      c1 = n1;
      c2 = n2;
      c3 = n3;
      a += 0x9E3779B9u;
      b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};

__device__ __forceinline__ double uniform53(u32 hi, u32 lo) {  // in (0, 1)
  return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6) + 0.5) * (1.0 / 9007199254740992.0);
}

// number of targets strictly below v (targets ascending)
__device__ __forceinline__ int lower_bound(const double *__restrict__ t, int n, double v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (t[mid] < v) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

struct RsShared {
  double warp_sum[kRsThreads / 32];
  u32 warp_kept[kRsThreads / 32], warp_drawn[kRsThreads / 32];
};

// H of row m of sample x (m = 0: the diagonal), exactly the value get_comb_hij_fused writes
template <int L, typename T>
__device__ __forceinline__ T row_value(const Onv<L> &x, const ExcGeom &g, const OrbLists &lists, const T *__restrict__ h1e,
                                       const T *__restrict__ h2e, T hii, int m, Onv<L> &ket) {
  if (m == 0) {
    ket = x;
    return hii;
  }
  const Exc e = decode_exc(g, lists, m - 1);
  ket = apply_exc<L>(x, e);
  return exc_element<L, T>(x, e, h1e, h2e, g.sorb);
}

// PASS 0: S and the counts (offsets[s] = kept + distinct drawn rows); PASS 1: emit
template <int L, typename T, int PASS>
__global__ void __launch_bounds__(kRsThreads)
reduce_sample_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, const T *__restrict__ h2e, const T *__restrict__ diag, double eps,
                     int n_draw, int n_pow2, unsigned long long seed, const long long *__restrict__ draws, double *__restrict__ row_sum,
                     u32 *__restrict__ kept_cnt, long long *__restrict__ offsets, u64 *__restrict__ x_out, T *__restrict__ h_out,
                     long long *__restrict__ idx_out, long long n, ExcGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *targets = reinterpret_cast<double *>(smem_raw);  // [n_pow2]
  OrbLists &lists = *reinterpret_cast<OrbLists *>(smem_raw + 8 * (size_t)n_pow2);
  __shared__ RsShared sh;
  __shared__ double s_total;
  const long long s = blockIdx.x;
  if (s >= n) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const Onv<L> x = load_onv<L>(bra + s * L);
  if (threadIdx.x < 32) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x);
  __syncthreads();
  const int M = g.nsd + 1;
  const T hii = diag[s];
  const bool semi = eps > 0.0;  // eps == 0: purely stochastic, nothing is kept deterministically (eloc.py:263-270)
  // |H| is compared with eps rounded to the integrals' dtype, as torch compares Hmat and as reduce_kernel does: under float32
  // a row with |H| == float(eps) < eps is kept.  Both passes use this one value, so counts and emitted rows agree.
  const double thr = (double)(T)eps;

  // running sum of the sub-eps magnitudes in row order: the same code (same rounding) in every pass
  auto chunk_scan = [&](double w, double &running, double &before) {
    double incl = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double up = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += up;
    }
    if (lane == 31) sh.warp_sum[warp] = incl;
    __syncthreads();
    double base = running;
#pragma unroll
    for (int q = 0; q < kRsThreads / 32; ++q) {
      const double t = sh.warp_sum[q];
      if (q < warp) base += t;
      running += t;
    }
    before = base + (incl - w);
    __syncthreads();
  };

  double S;
  if (PASS == 0) {
    double running = 0.0, before;
    for (int c0 = 0; c0 < M; c0 += kRsThreads) {
      const int m = c0 + (int)threadIdx.x;
      double w = 0.0;
      if (m < M) {
        Onv<L> ket;
        const double a = fabs((double)row_value<L, T>(x, g, lists, h1e, h2e, hii, m, ket));
        w = (semi && a >= thr) ? 0.0 : a;
      }
      chunk_scan(w, running, before);
    }
    S = running;
    if (threadIdx.x == 0) row_sum[s] = S;
  } else {
    S = row_sum[s];
  }

  // the sample's draws as sorted points: seeded uniforms times S, or the caller's row indices (+ 0.5)
  const Philox rng = {(u32)seed, (u32)(seed >> 32)};
  for (int j = threadIdx.x; j < n_pow2; j += kRsThreads) {
    double t = 1.0e300;
    if (j < n_draw) {
      if (draws != nullptr) {
        t = (double)draws[s * n_draw + j] + 0.5;
      } else {
        const uint4 r = rng((u32)(j >> 1), (u32)s, (u32)((unsigned long long)s >> 32), 0x5eedu);
        t = ((j & 1) ? uniform53(r.z, r.w) : uniform53(r.x, r.y)) * S;
      }
    }
    targets[j] = t;
  }
  __syncthreads();
  for (int k = 2; k <= n_pow2; k <<= 1) {  // bitonic sort, ascending
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pow2; i += kRsThreads) {
        const int p = i ^ j;
        if (p > i) {
          const double a = targets[i], b = targets[p];
          const bool up = (i & k) == 0;
          if ((a > b) == up) {
            targets[i] = b;
            targets[p] = a;
          }
        }
      }
      __syncthreads();
    }
  }

  const long long flat_base = s * (long long)M;
  const long long out_base = PASS == 1 ? offsets[s] : 0;
  const u32 kept_total = PASS == 1 ? kept_cnt[s] : 0u;  // drawn rows go after the kept ones
  u32 kept = 0, drawn = 0;                               // CTA-uniform running counts
  double running = 0.0, before;
  const double scale = S / (double)n_draw;
  for (int c0 = 0; c0 < M; c0 += kRsThreads) {
    const int m = c0 + (int)threadIdx.x;
    Onv<L> ket = x;
    T v = (T)0.0;
    double w = 0.0;
    bool keep = false;
    if (m < M) {
      v = row_value<L, T>(x, g, lists, h1e, h2e, hii, m, ket);
      const double a = fabs((double)v);
      keep = semi && a >= thr;
      w = keep ? 0.0 : a;
    }
    chunk_scan(w, running, before);
    int cnt = 0;
    if (m < M && !keep) {
      if (draws != nullptr) cnt = lower_bound(targets, n_draw, (double)(m + 1)) - lower_bound(targets, n_draw, (double)m);
      else if (w > 0.0) cnt = lower_bound(targets, n_draw, before + w) - lower_bound(targets, n_draw, before);
    }
    const u32 bk = __ballot_sync(0xffffffffu, keep), bd = __ballot_sync(0xffffffffu, cnt > 0);
    if (lane == 0) {
      sh.warp_kept[warp] = (u32)__popc(bk);
      sh.warp_drawn[warp] = (u32)__popc(bd);
    }
    __syncthreads();
    u32 kb = 0, db = 0, kt = 0, dt = 0;
#pragma unroll
    for (int q = 0; q < kRsThreads / 32; ++q) {
      const u32 a = sh.warp_kept[q], b = sh.warp_drawn[q];
      if (q < warp) {
        kb += a;
        db += b;
      }
      kt += a;
      dt += b;
    }
    if (PASS == 1) {
      const u32 below = (1u << lane) - 1u;
      if (keep) {
        const long long o = out_base + kept + kb + (u32)__popc(bk & below);
#pragma unroll
        for (int i = 0; i < L; ++i) x_out[o * L + i] = ket.w[i];
        h_out[o] = v;
        idx_out[o] = flat_base + m;
      } else if (cnt > 0) {
        const long long o = out_base + kept_total + drawn + db + (u32)__popc(bd & below);
#pragma unroll
        for (int i = 0; i < L; ++i) x_out[o * L + i] = ket.w[i];
        // (count / N) * H / p with p = |H| / S
        h_out[o] = (T)((v < (T)0.0 ? -1.0 : 1.0) * scale * (double)cnt);
        idx_out[o] = flat_base + m;
      }
    }
    kept += kt;
    drawn += dt;
    __syncthreads();
  }
  if (PASS == 0 && threadIdx.x == 0) {
    kept_cnt[s] = kept;
    offsets[s] = (long long)kept + (long long)drawn;
  }
  (void)s_total;
}

// ---- host side --------------------------------------------------------------------------------------------------------
struct RsScratch {
  long long diag, row_sum, kept, cub, total;
  size_t cub_bytes;
};

static RsScratch rs_layout(long long n) {
  RsScratch l;
  size_t tmp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp, (const long long *)nullptr, (long long *)nullptr, (int)(n + 1));
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  l.diag = 0;
  l.row_sum = up(8 * n);
  l.kept = l.row_sum + up(8 * n);
  l.cub = l.kept + up(4 * n);
  l.cub_bytes = tmp;
  l.total = l.cub + (long long)tmp + 256;
  return l;
}

long long reduce_sample_scratch_bytes(long long n) { return rs_layout(n < 0 ? 0 : n).total; }

template <int L, typename T>
int launch_diag_plain(const u64 *bra, const T *h1e, const T *h2e, T *out, long long n, long long stride, int sorb, int nele, cudaStream_t st);

template <int L, typename T>
static int launch_rs_LT(const u64 *bra, const T *h1e, const T *h2e, long long n, const ExcGeom &g, double eps, int n_draw,
                        unsigned long long seed, const long long *draws, int emit, void *scratch, long long *offsets, u64 *x_out, T *h_out,
                        long long *idx_out, cudaStream_t st) {
  const RsScratch lay = rs_layout(n);
  char *sc = static_cast<char *>(scratch);
  T *diag = reinterpret_cast<T *>(sc + lay.diag);
  double *row_sum = reinterpret_cast<double *>(sc + lay.row_sum);
  u32 *kept = reinterpret_cast<u32 *>(sc + lay.kept);
  int n_pow2 = 2;
  while (n_pow2 < n_draw) n_pow2 <<= 1;
  const size_t smem = 8 * (size_t)n_pow2 + sizeof(OrbLists);
  if (!emit) {
    if (int rc = launch_diag_plain<L, T>(bra, h1e, h2e, diag, n, 1, g.sorb, g.nele, st)) return rc;
    auto kern = reduce_sample_kernel<L, T, 0>;
    if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("reduce_sample_kernel smem opt-in");
    kern<<<(unsigned)n, kRsThreads, smem, st>>>(bra, h1e, h2e, diag, eps, n_draw, n_pow2, seed, draws, row_sum, kept, offsets, nullptr, nullptr,
                                                nullptr, n, g);
    count_launch();
    if (int rc = check_launch("reduce_sample_kernel (count)")) return rc;
    if (cudaMemsetAsync(offsets + n, 0, 8, st) != cudaSuccess) return check_launch("reduce_sample offsets memset");
    size_t tmp = lay.cub_bytes;
    const cudaError_t e = cub::DeviceScan::ExclusiveSum(sc + lay.cub, tmp, offsets, offsets, (int)(n + 1), st);
    if (e != cudaSuccess) {
      set_error("reduce_sample scan: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
      return 3;
    }
    count_launch(2);
    return 0;
  }
  auto kern = reduce_sample_kernel<L, T, 1>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("reduce_sample_kernel smem opt-in");
  kern<<<(unsigned)n, kRsThreads, smem, st>>>(bra, h1e, h2e, diag, eps, n_draw, n_pow2, seed, draws, row_sum, kept, offsets, x_out, h_out, idx_out,
                                              n, g);
  count_launch();
  return check_launch("reduce_sample_kernel (emit)");
}

template <typename T>
int launch_reduce_sample(const u64 *bra, const T *h1e, const T *h2e, long long n, const ExcGeom &g, double eps, int n_draw,
                         unsigned long long seed, const long long *draws, int emit, void *scratch, long long scratch_bytes, long long *offsets,
                         u64 *x_out, T *h_out, long long *idx_out, cudaStream_t st) {
  if (n == 0) return 0;
  if (n > 0x7fffffffLL - 1) {
    set_error("reduce_sample: at most 2^31 - 2 samples per call (got %lld)", n);
    return 1;
  }
  if (n_draw < 1 || n_draw > 8192) {
    set_error("reduce_sample: eps_sample = %d outside [1, 8192]", n_draw);
    return 1;
  }
  if (scratch_bytes < rs_layout(n).total) {
    set_error("reduce_sample scratch too small: %lld < %lld bytes", scratch_bytes, rs_layout(n).total);
    return 4;
  }
  switch (g.L) {
    case 1: return launch_rs_LT<1, T>(bra, h1e, h2e, n, g, eps, n_draw, seed, draws, emit, scratch, offsets, x_out, h_out, idx_out, st);
    case 2: return launch_rs_LT<2, T>(bra, h1e, h2e, n, g, eps, n_draw, seed, draws, emit, scratch, offsets, x_out, h_out, idx_out, st);
    case 3: return launch_rs_LT<3, T>(bra, h1e, h2e, n, g, eps, n_draw, seed, draws, emit, scratch, offsets, x_out, h_out, idx_out, st);
  }
  set_error("unsupported ONV length L=%d", g.L);
  return 1;
}

template int launch_reduce_sample<double>(const u64 *, const double *, const double *, long long, const ExcGeom &, double, int,
                                          unsigned long long, const long long *, int, void *, long long, long long *, u64 *, double *,
                                          long long *, cudaStream_t);
template int launch_reduce_sample<float>(const u64 *, const float *, const float *, long long, const ExcGeom &, double, int, unsigned long long,
                                         const long long *, int, void *, long long, long long *, u64 *, float *, long long *, cudaStream_t);

}  // namespace pynqs
