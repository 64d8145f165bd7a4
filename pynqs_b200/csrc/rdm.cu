// rdm.cu -- the off-diagonal part of the one- and two-body reduced density matrices of a coefficient vector c over the sorted
// key table, summed over the entries of the square CSR structure (crow, col) of the sample-space Hamiltonian.
//
// Spin orbital P = 2p + sigma (alpha even, beta odd).  With the library's sign (an operator on bit b counts the occupied bits
// below b) and Gamma[A, B, R, S] = sum over pairs (i, j) of conj(c_i) c_j <key_i| a+_A a+_R a_S a_B |key_j>, PySCF's blocks
// are dm1s[p, q] = <a+_qs a_ps>, dm2aa / dm2bb[p, q, r, s] = Gamma over one spin, dm2ab[p, q, r, s] = Gamma[pa, qa, rb, sb].
// An off-diagonal entry (i, j) is a single (bra-only P, ket-only Q) or a double (bra-only P1 > P2, ket-only Q1 > Q2):
//   single  w = conj(c_i) c_j <i| a+_P a_Q |j>:  dm1[q, p] += w;  Gamma[P, Q, r, r] = Gamma[r, r, P, Q] = w n_r and
//           Gamma[r, Q, P, r] = Gamma[P, r, r, Q] = -w n_r for every spectator r occupied in both determinants;
//   double  w = conj(c_i) c_j <i| a+_P1 a+_P2 a_Q2 a_Q1 |j>:  Gamma[P1, Q1, P2, Q2] = Gamma[P2, Q2, P1, Q1] = w and
//           Gamma[P2, Q1, P1, Q2] = Gamma[P1, Q2, P2, Q1] = -w.
// The diagonal entries (the products |c_i|^2 n_p n_r) are not written here: they are dense GEMMs over the occupations, left
// to the caller.  Every dense position is owned by one class -- the diagonal (p p r r / p r r p), one bin of singles
// (p q r r / r r p q / r q p r / p r r q with p != q) or one bin of doubles (four distinct spin orbitals) --, so the reduced
// sums are stored, never added.
//
// Determinism without float atomics: one (bin, i << 32 | j) record per CSR entry, in CSR order (bin_kernel); a stable radix
// sort by bin; run-length encoding of the sorted bins and a scan of the run lengths; then one warp per run (run_kernel) sums
// the run's weights lane-strided in run order and combines the lanes by a butterfly, and sums each spectator's w n_r
// sequentially in run order.  Every order is fixed by the run's contents, which the stable sort fixes by the CSR.
//
// Bins: singles P * sorb + Q in [0, sorb^2); doubles sorb^2 + pair(P1, P2) * npair + pair(Q1, Q2), pair(a, b) = a (a - 1) / 2 + b;
// everything else -- the diagonal, the doubles when only dm1 is wanted, a pair that changes the spin -- the top bin `none`.
// The sort reads the bits up to `none`'s highest one: 11 at 40 spin orbitals for dm1 alone, 20 with dm2.
#include <thrust/iterator/discard_iterator.h>

#include <cub/cub.cuh>

#include "rederive.cuh"

namespace pynqs {

constexpr int kRdmThreads = 128;
constexpr long long kRdmWarpsCap = 148LL * 16 * (kRdmThreads / 32);  // persistent grids: 16 CTAs of 128 threads per SM

struct RdmGeom {
  int sorb, norb;
  u32 npair, dbl0, none;  // spin-orbital pairs, first double bin, the bin of records that add nothing
  bool two;               // dm2 wanted
};

__device__ __forceinline__ u32 pair_index(u32 hi, u32 lo) { return ((hi * (hi - 1)) >> 1) + lo; }

template <int L>
__global__ void __launch_bounds__(kRdmThreads) rdm_bin_kernel(const long long *__restrict__ crow, const long long *__restrict__ col,
                                                              const u64 *__restrict__ key, long long N, RdmGeom g, u32 *__restrict__ bins,
                                                              u64 *__restrict__ pay) {
  const int lane = threadIdx.x & 31;
  const long long nwarps = (long long)gridDim.x * (kRdmThreads / 32);
  for (long long i = (long long)blockIdx.x * (kRdmThreads / 32) + (threadIdx.x >> 5); i < N; i += nwarps) {
    const Onv<L> x = load_onv<L>(key + i * L);
    const long long e = __ldg(crow + i + 1);
    for (long long p = __ldg(crow + i) + lane; p < e; p += 32) {
      const long long j = __ldg(col + p);
      const Onv<L> y = load_onv<L>(key + j * L);
      const int cls = j == i ? 0 : excitation_class<L>(x, y);
      Onv<L> cre, ann;
#pragma unroll
      for (int w = 0; w < L; ++w) {
        cre.w[w] = x.w[w] & ~y.w[w];
        ann.w[w] = y.w[w] & ~x.w[w];
      }
      u32 bin = g.none;
      if (cls == 1) {
        const u32 P = (u32)pop_highest<L>(cre), Q = (u32)pop_highest<L>(ann);
        if (((P ^ Q) & 1u) == 0u) bin = P * (u32)g.sorb + Q;
      } else if (cls == 2 && g.two) {
        u32 P1, P2, Q1, Q2;
        two_set_bits<L>(cre, P1, P2);
        two_set_bits<L>(ann, Q1, Q2);
        if (((P1 & 1u) + (P2 & 1u)) == ((Q1 & 1u) + (Q2 & 1u))) bin = g.dbl0 + pair_index(P1, P2) * g.npair + pair_index(Q1, Q2);
      }
      bins[p] = bin;
      pay[p] = ((u64)i << 32) | (u64)j;
    }
  }
}

// Gamma[A, B, R, S] = v into its block of dm2 ([3][norb^4]: aa, ab, bb); positions outside the three blocks are dropped
template <bool CPLX>
__device__ __forceinline__ void put_gamma(double *__restrict__ dm2, int norb, u32 A, u32 B, u32 R, u32 S, double re, double im) {
  if (((A ^ B) & 1u) || ((R ^ S) & 1u)) return;
  const size_t n = (size_t)norb, blk = n * n * n * n;
  size_t at;
  if ((A & 1u) == (R & 1u)) at = (A & 1u) * 2 * blk + (((size_t)(A >> 1) * n + (B >> 1)) * n + (R >> 1)) * n + (S >> 1);
  else if ((A & 1u) == 0u) at = blk + (((size_t)(A >> 1) * n + (B >> 1)) * n + (R >> 1)) * n + (S >> 1);
  else at = blk + (((size_t)(R >> 1) * n + (S >> 1)) * n + (A >> 1)) * n + (B >> 1);
  if (CPLX) {
    dm2[2 * at] = re;
    dm2[2 * at + 1] = im;
  } else {
    dm2[at] = re;
  }
}

// conj(c_i) c_j of record r, times -1 when odd
template <bool CPLX>
__device__ __forceinline__ void weight(const double *__restrict__ c, u64 r, int odd, double &re, double &im) {
  const long long i = (long long)(r >> 32), j = (long long)(r & 0xffffffffull);
  if (CPLX) {
    const double ar = __ldg(c + 2 * i), ai = __ldg(c + 2 * i + 1), br = __ldg(c + 2 * j), bi = __ldg(c + 2 * j + 1);
    re = fma(ar, br, ai * bi);
    im = fma(ar, bi, -(ai * br));
  } else {
    re = __ldg(c + i) * __ldg(c + j);
    im = 0.0;
  }
  if (odd) {
    re = -re;
    im = -im;
  }
}

__device__ __forceinline__ void lane_sum(double &re, double &im) {
  for (int o = 16; o > 0; o >>= 1) {  // butterfly: every lane ends with the same bits
    re += __shfl_xor_sync(0xffffffffu, re, o);
    im += __shfl_xor_sync(0xffffffffu, im, o);
  }
}

template <int L, bool CPLX>
__device__ __forceinline__ void single_run(const u64 *__restrict__ pay, long long b, long long e, const u64 *__restrict__ key, const double *__restrict__ c,
                           const RdmGeom &g, u32 P, u32 Q, double *__restrict__ dm1, double *__restrict__ dm2) {
  const int lane = threadIdx.x & 31;
  double re = 0.0, im = 0.0;
  double sre[2 * L], sim[2 * L];  // spectator sums of spin orbitals lane + 32 m
#pragma unroll
  for (int m = 0; m < 2 * L; ++m) sre[m] = sim[m] = 0.0;
  for (long long p0 = b; p0 < e; p0 += 32) {
    double wr = 0.0, wi = 0.0;
    Onv<L> y;
#pragma unroll
    for (int w = 0; w < L; ++w) y.w[w] = 0;
    if (p0 + lane < e) {
      const u64 r = __ldg(pay + p0 + lane);
      y = load_onv<L>(key + (long long)(r & 0xffffffffull) * L);
      Onv<L> t = y;  // <i| a+_P a_Q |j>: a_Q, then a+_P
      int s = count_below<L>(t, (int)Q);
      flip_bit<L>(t, (int)Q);
      s += count_below<L>(t, (int)P);
      weight<CPLX>(c, r, s & 1, wr, wi);
      re += wr;
      im += wi;
    }
    if (g.two) {
      const int cnt = e - p0 < 32 ? (int)(e - p0) : 32;
      for (int t = 0; t < cnt; ++t) {
        const double tr = __shfl_sync(0xffffffffu, wr, t), ti = __shfl_sync(0xffffffffu, wi, t);
#pragma unroll
        for (int m = 0; m < 2 * L; ++m) {
          const u64 yw = __shfl_sync(0xffffffffu, y.w[m >> 1], t);
          const u32 r = (u32)(lane + 32 * m);
          if (((yw >> (r & 63)) & 1ull) && r != Q) {
            sre[m] += tr;
            sim[m] += ti;
          }
        }
      }
    }
  }
  lane_sum(re, im);
  const size_t n = (size_t)g.norb;
  if (lane == 0) {
    const size_t at = (P & 1u) * n * n + (size_t)(Q >> 1) * n + (P >> 1);
    if (CPLX) {
      dm1[2 * at] = re;
      dm1[2 * at + 1] = im;
    } else {
      dm1[at] = re;
    }
  }
  if (g.two) {
#pragma unroll
    for (int m = 0; m < 2 * L; ++m) {
      const u32 r = (u32)(lane + 32 * m);
      if (r >= (u32)g.sorb || r == P || r == Q) continue;
      put_gamma<CPLX>(dm2, g.norb, P, Q, r, r, sre[m], sim[m]);
      put_gamma<CPLX>(dm2, g.norb, r, r, P, Q, sre[m], sim[m]);
      put_gamma<CPLX>(dm2, g.norb, r, Q, P, r, -sre[m], -sim[m]);
      put_gamma<CPLX>(dm2, g.norb, P, r, r, Q, -sre[m], -sim[m]);
    }
  }
}

template <int L, bool CPLX>
__device__ __forceinline__ void double_run(const u64 *__restrict__ pay, long long b, long long e, const u64 *__restrict__ key, const double *__restrict__ c,
                           const RdmGeom &g, u32 P1, u32 P2, u32 Q1, u32 Q2, double *__restrict__ dm2) {
  const int lane = threadIdx.x & 31;
  double re = 0.0, im = 0.0;
  for (long long p = b + lane; p < e; p += 32) {
    const u64 r = __ldg(pay + p);
    Onv<L> t = load_onv<L>(key + (long long)(r & 0xffffffffull) * L);  // <i| a+_P1 a+_P2 a_Q2 a_Q1 |j>, right to left
    int s = count_below<L>(t, (int)Q1);
    flip_bit<L>(t, (int)Q1);
    s += count_below<L>(t, (int)Q2);
    flip_bit<L>(t, (int)Q2);
    s += count_below<L>(t, (int)P2);
    flip_bit<L>(t, (int)P2);
    s += count_below<L>(t, (int)P1);
    double wr, wi;
    weight<CPLX>(c, r, s & 1, wr, wi);
    re += wr;
    im += wi;
  }
  lane_sum(re, im);
  if (lane == 0) {
    put_gamma<CPLX>(dm2, g.norb, P1, Q1, P2, Q2, re, im);
    put_gamma<CPLX>(dm2, g.norb, P2, Q2, P1, Q1, re, im);
    put_gamma<CPLX>(dm2, g.norb, P2, Q1, P1, Q2, -re, -im);
    put_gamma<CPLX>(dm2, g.norb, P1, Q2, P2, Q1, -re, -im);
  }
}

template <int L, bool CPLX>
__global__ void __launch_bounds__(kRdmThreads) rdm_run_kernel(const u32 *__restrict__ bins, const u64 *__restrict__ pay,
                                                              const int *__restrict__ starts, const int *__restrict__ num_runs, long long R,
                                                              const u64 *__restrict__ key, const double *__restrict__ c, RdmGeom g,
                                                              double *__restrict__ dm1, double *__restrict__ dm2) {
  const long long nwarps = (long long)gridDim.x * (kRdmThreads / 32);
  const long long nruns = *num_runs;
  for (long long k = (long long)blockIdx.x * (kRdmThreads / 32) + (threadIdx.x >> 5); k < nruns; k += nwarps) {
    const long long b = __ldg(starts + k), e = k + 1 < nruns ? __ldg(starts + k + 1) : R;
    const u32 bin = __ldg(bins + b);
    if (bin == g.none) continue;
    // the run's orbitals, from its first record
    const u64 r = __ldg(pay + b);
    const Onv<L> x = load_onv<L>(key + (long long)(r >> 32) * L), y = load_onv<L>(key + (long long)(r & 0xffffffffull) * L);
    Onv<L> cre, ann;
#pragma unroll
    for (int w = 0; w < L; ++w) {
      cre.w[w] = x.w[w] & ~y.w[w];
      ann.w[w] = y.w[w] & ~x.w[w];
    }
    if (bin < g.dbl0) {
      const u32 P = (u32)pop_highest<L>(cre), Q = (u32)pop_highest<L>(ann);
      single_run<L, CPLX>(pay, b, e, key, c, g, P, Q, dm1, dm2);
    } else {
      u32 P1, P2, Q1, Q2;
      two_set_bits<L>(cre, P1, P2);
      two_set_bits<L>(ann, Q1, Q2);
      double_run<L, CPLX>(pay, b, e, key, c, g, P1, P2, Q1, Q2, dm2);
    }
  }
}

struct RdmScratch {
  long long bins0, bins1, pay0, pay1, starts, num_runs, cub, total;
};

// the radix sort, the run-length encoding and the scan of R items need temporary storage: reserved here, checked against
// cub's own figures at launch
static long long rdm_cub_reserve(long long R) { return 2 * R + (4LL << 20); }

static RdmScratch rdm_layout(long long R) {
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  RdmScratch l;
  l.bins0 = 0;
  l.bins1 = up(l.bins0 + 4 * R);
  l.pay0 = up(l.bins1 + 4 * R);
  l.pay1 = up(l.pay0 + 8 * R);
  l.starts = up(l.pay1 + 8 * R);
  l.num_runs = up(l.starts + 4 * R);
  l.cub = up(l.num_runs + 8);
  l.total = l.cub + rdm_cub_reserve(R);
  return l;
}

long long rdm_scratch_bytes(long long nnz) { return rdm_layout(nnz).total; }

// cub call f(temp, bytes) after checking its temporary storage against the reservation
template <typename F>
static int cub_call(const char *what, char *temp, long long reserved, F f) {
  size_t tmp = 0;
  cudaError_t e = f(nullptr, tmp);
  if (e == cudaSuccess && (long long)tmp > reserved) {
    set_error("rdm %s: %zu bytes of temporary storage needed, %lld reserved", what, tmp, reserved);
    return 4;
  }
  if (e == cudaSuccess) e = f(temp, tmp);
  if (e != cudaSuccess) {
    set_error("rdm %s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
    return 3;
  }
  return 0;
}

template <int L>
static void launch_runs(bool cplx, const u32 *bins, const u64 *pay, const int *starts, const int *num_runs, long long R, const u64 *key,
                        const double *c, const RdmGeom &g, double *dm1, double *dm2, cudaStream_t st) {
  const long long warps = R < kRdmWarpsCap ? R : kRdmWarpsCap;  // at most one run per record
  const unsigned grid = (unsigned)((warps + kRdmThreads / 32 - 1) / (kRdmThreads / 32));
  if (cplx) rdm_run_kernel<L, true><<<grid, kRdmThreads, 0, st>>>(bins, pay, starts, num_runs, R, key, c, g, dm1, dm2);
  else rdm_run_kernel<L, false><<<grid, kRdmThreads, 0, st>>>(bins, pay, starts, num_runs, R, key, c, g, dm1, dm2);
}

// 0 < N, nnz < 2^31; arguments checked, dm1 / dm2 cleared by pynqs_rdm_offdiag
int launch_rdm(const long long *crow, const long long *col, const u64 *key, long long N, long long nnz, int sorb, const double *c, int cplx,
               void *scratch, long long scratch_bytes, double *dm1, double *dm2, cudaStream_t st) {
  const int L = (sorb - 1) / 64 + 1;
  const RdmScratch l = rdm_layout(nnz);
  if (scratch_bytes < l.total) {
    set_error("rdm scratch too small: %lld < %lld bytes", scratch_bytes, l.total);
    return 4;
  }
  RdmGeom g;
  g.sorb = sorb;
  g.norb = sorb / 2;
  g.npair = (u32)(sorb * (sorb - 1) / 2);
  g.dbl0 = (u32)(sorb * sorb);
  g.two = dm2 != nullptr;
  g.none = g.two ? g.dbl0 + g.npair * g.npair : g.dbl0;
  const int end_bit = 32 - __builtin_clz(g.none);
  char *sc = static_cast<char *>(scratch);
  u32 *bins0 = reinterpret_cast<u32 *>(sc + l.bins0);
  u64 *pay0 = reinterpret_cast<u64 *>(sc + l.pay0);
  int *starts = reinterpret_cast<int *>(sc + l.starts);
  int *num_runs = reinterpret_cast<int *>(sc + l.num_runs);
  char *temp = sc + l.cub;
  const long long reserved = rdm_cub_reserve(nnz);
  const int R = (int)nnz;

  const long long warps = N < kRdmWarpsCap ? N : kRdmWarpsCap;
  const unsigned grid = (unsigned)((warps + kRdmThreads / 32 - 1) / (kRdmThreads / 32));
  if (L == 1) rdm_bin_kernel<1><<<grid, kRdmThreads, 0, st>>>(crow, col, key, N, g, bins0, pay0);
  else if (L == 2) rdm_bin_kernel<2><<<grid, kRdmThreads, 0, st>>>(crow, col, key, N, g, bins0, pay0);
  else rdm_bin_kernel<3><<<grid, kRdmThreads, 0, st>>>(crow, col, key, N, g, bins0, pay0);
  count_launch();
  if (int rc = check_launch("rdm_bin_kernel")) return rc;

  cub::DoubleBuffer<u32> kb(bins0, reinterpret_cast<u32 *>(sc + l.bins1));
  cub::DoubleBuffer<u64> vb(pay0, reinterpret_cast<u64 *>(sc + l.pay1));
  if (int rc = cub_call("sort", temp, reserved, [&](void *t, size_t &b) {
        return cub::DeviceRadixSort::SortPairs(t, b, kb, vb, R, 0, end_bit, st);
      }))
    return rc;
  const u32 *bins = kb.Current();
  const u64 *pay = vb.Current();
  if (int rc = cub_call("run-length encoding", temp, reserved, [&](void *t, size_t &b) {
        return cub::DeviceRunLengthEncode::Encode(t, b, bins, thrust::make_discard_iterator(), starts, num_runs, R, st);
      }))
    return rc;
  if (int rc = cub_call("scan", temp, reserved, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, starts, starts, R, st); }))
    return rc;
  count_launch(5);

  if (L == 1) launch_runs<1>(cplx != 0, bins, pay, starts, num_runs, nnz, key, c, g, dm1, dm2, st);
  else if (L == 2) launch_runs<2>(cplx != 0, bins, pay, starts, num_runs, nnz, key, c, g, dm1, dm2, st);
  else launch_runs<3>(cplx != 0, bins, pay, starts, num_runs, nnz, key, c, g, dm1, dm2, st);
  count_launch();
  return check_launch("rdm_run_kernel");
}

}  // namespace pynqs
