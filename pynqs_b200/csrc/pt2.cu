// pt2.cu -- the Epstein-Nesbet second-order correction of sample-space states over the sorted key table T:
//   E_PT2[r] = sum over the externals a of (sum over i in T of <key_i|H|a> C[i, r])^2 / (E[r] - <a|H|a>)
// (the caller divides by sum_i C[i, r]^2).  The externals are the distinct single and double excitations of the table rows
// that are not in the table.
//
// One external is reached from many rows, and its numerator has to be complete before it is squared; the (row, external)
// pairs are far too many to hold at once (7.9 * 10^9 for 10^6 rows of 40 spin orbitals).  So the externals are split into
// 2^log2_parts partitions by the top bits of a 64-bit hash of the determinant, and a pass handles one partition:
//   count  one CTA per table row (reduce_kernel's row enumeration, enum_rows.cuh): a row's excitation is kept when it
//          falls in the partition -- tested first, so only 1 / P of the rows pay for the lookup -- and is not in the table
//          (spin_find, the beta-grouped copy); per-row counts, then an exclusive scan into offsets;
//   emit   the same enumeration writes, per kept excitation, the determinant and the 16-byte payload (<key_i|H|a>, i) at the
//          row's offset, ranked with ballots so the order is ascending (row, excitation index) whatever the timing;
//   sort   the table sort (table.cu), stable, with the payload: equal determinants end up adjacent, in emit order;
//   reduce the run heads of equal determinants (a cub select), then one thread per run sums H * C[i, r] in run order,
//          takes <a|H|a> (diag_element's terms in its order: launch_diag_f64's bits) and adds num^2 / (E[r] - <a|H|a>) to its
//          own partial; a fixed grid, a fixed butterfly per warp, the warps of a block in order and the blocks in order
//          (pt2_finish_kernel) give one partial per root, added to the caller's accumulator.  No float atomics: two calls
//          with the same inputs give identical bits.
// One thread per run: the runs are short on uniform tables (a few sources each), and the numerator is summed strictly in
// run order.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "enum_rows.cuh"
#include "gindex.cuh"

namespace pynqs {

constexpr int kPt2RunThreads = 256;
constexpr int kPt2RunBlocks = 148 * 4;  // fixed: the summation order of the runs depends on it
constexpr int kPt2MaxRoots = 8;

// partition of a determinant: the top log2_parts bits of a 64-bit mix of its two string hashes
template <int L>
__device__ __forceinline__ u32 pt2_part(const Onv<L> &y, u32 log2_parts) {
  if (log2_parts == 0) return 0u;
  u64 h = hash_alpha<L>(y) ^ (hash_beta<L>(y) * 0x9E3779B97F4A7C15ull);
  h ^= h >> 31;
  h *= 0xBF58476D1CE4E5B9ull;
  h ^= h >> 29;
  return (u32)(h >> (64 - log2_parts));
}

struct Pt2Sel {
  const u64 *key;
  long long N;
  GroupView gv;
  bool dup;
  u32 part, log2_parts;
};

template <int L, int CLS, int ROWS, bool EMIT>
__device__ __forceinline__ void pt2_class(const Onv<L> &x, long long s, const EnumEntry<L> *__restrict__ tab, const TableOffsets &to,
                                          const ExcGeom &g, const OrbLists &lists, const double *__restrict__ h1e,
                                          const PrepView<double> &prep, const Pt2Sel &sel, int lo, int hi, u32 &kept, u32 *warp_cnt,
                                          long long out_base, u64 *__restrict__ x_out, u64 *__restrict__ pay_out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kChunk = 32 * ROWS, kWarps = kEnumThreads / 32;
  for (int c0 = lo; c0 < hi; c0 += kWarps * kChunk) {  // same trip count for every warp: there are barriers inside
    const int c = c0 + warp * kChunk;
    Onv<L> row[ROWS];
    double val[ROWS];
    u32 sgn[ROWS];
    class_rows<L, double, EMIT, CLS, ROWS>(x, tab, to, g, lists, h1e, prep, c, hi, row, val, sgn);
    u32 bal[ROWS], wc = 0;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      const bool keep = c + lane + 32 * j < hi && pt2_part<L>(row[j], sel.log2_parts) == sel.part &&
                        spin_find<L>(sel.key, sel.N, sel.gv, sel.dup, row[j]) < 0;
      bal[j] = __ballot_sync(0xffffffffu, keep);
      wc += (u32)__popc(bal[j]);
    }
    if (!EMIT) {
      kept += wc;
      continue;
    }
    if (lane == 0) warp_cnt[warp] = wc;
    __syncthreads();
    u32 before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      const u32 t = warp_cnt[w];
      before += w < warp ? t : 0u;
      total += t;
    }
    u32 pos = kept + before;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      if ((bal[j] >> lane) & 1u) {
        const long long o = out_base + pos + (u32)__popc(bal[j] & ((1u << lane) - 1u));
#pragma unroll
        for (int w = 0; w < L; ++w) x_out[o * L + w] = row[j].w[w];
        *reinterpret_cast<double2 *>(pay_out + 2 * o) = make_double2(flip_sign(1.0 * val[j], sgn[j]), __longlong_as_double(s));
      }
      pos += (u32)__popc(bal[j]);
    }
    kept += total;
    __syncthreads();
  }
}

// one CTA per table row; count: offsets[s] = the row's kept excitations; emit: the records at offsets[s]
template <int L, bool EMIT>
__global__ void __launch_bounds__(kEnumThreads)
pt2_rows_kernel(const double *__restrict__ h1e, PrepView<double> prep, Pt2Sel sel, long long *__restrict__ offsets, u64 *__restrict__ x_out,
                u64 *__restrict__ pay_out, ExcGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  OrbLists &lists = *reinterpret_cast<OrbLists *>(smem_raw);
  EnumEntry<L> *tab = reinterpret_cast<EnumEntry<L> *>(smem_raw + sizeof(OrbLists));
  __shared__ u32 warp_cnt[kEnumThreads / 32];
  __shared__ unsigned long long s_total;
  const long long s = blockIdx.x;
  const Onv<L> x = load_onv<L>(sel.key + s * L);
  if (threadIdx.x < 32) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x);
  if (threadIdx.x == 0) s_total = 0ull;
  __syncthreads();
  const TableOffsets to = table_offsets(g);
  const u32 na = (u32)prep.na, npair = (u32)prep.npair;
  for_each_table_entry(g, lists, to, [&](int t, int kind, u32 e0, u32 e1) {
    EnumEntry<L> e;
    const HitInfo hi = make_hit_info(kind, e0, e1, na, npair);
    e.off = hi.off;
    e.cmp = hi.cmp;
    set_mask<L>(e, e0 & 0xffu, e1 & 0xffu);
    tab[t] = e;
  });
  __syncthreads();

  // row 0 (the table row itself) is never an external
  const long long out_base = EMIT ? offsets[s] : 0;
  u32 kept = 0;
  const int M = g.nsd + 1;
  pt2_class<L, 0, 1, EMIT>(x, s, tab, to, g, lists, h1e, prep, sel, 1, g.d0 + 1, kept, warp_cnt, out_base, x_out, pay_out);
  pt2_class<L, 1, 1, EMIT>(x, s, tab, to, g, lists, h1e, prep, sel, g.d0 + 1, g.d1 + 1, kept, warp_cnt, out_base, x_out, pay_out);
  pt2_class<L, 2, kRowsPerThread, EMIT>(x, s, tab, to, g, lists, h1e, prep, sel, g.d1 + 1, g.d2 + 1, kept, warp_cnt, out_base, x_out, pay_out);
  pt2_class<L, 3, kRowsPerThread, EMIT>(x, s, tab, to, g, lists, h1e, prep, sel, g.d2 + 1, g.d3 + 1, kept, warp_cnt, out_base, x_out, pay_out);
  pt2_class<L, 4, kRowsPerThread, EMIT>(x, s, tab, to, g, lists, h1e, prep, sel, g.d3 + 1, M, kept, warp_cnt, out_base, x_out, pay_out);
  if (!EMIT) {
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_total, (unsigned long long)kept);  // integer tallies: order-free
    __syncthreads();
    if (threadIdx.x == 0) offsets[s] = (long long)s_total;
  }
}

// record i starts a run of equal determinants
template <int L>
struct Pt2Head {
  const u64 *key;
  __device__ __forceinline__ bool operator()(const int &i) const {
    if (i == 0) return true;
    bool same = true;
#pragma unroll
    for (int w = 0; w < L; ++w) same &= key[(long long)i * L + w] == key[(long long)(i - 1) * L + w];
    return !same;
  }
};

// <a|H|a> from D1[p] = h1e[p, p] and D2[p][q] = <pq||pq> in shared memory: the terms of diag_element in its order
// (occupied p ascending, then h1e, then the occupied q < p ascending), so the bits of launch_diag_f64
template <int L>
__device__ __forceinline__ double pt2_diag_table(const Onv<L> &x, const double *d1, const double *d2, int sorb) {
  double v = 0.0;
#pragma unroll
  for (int hp = 0; hp < 2 * L; ++hp) {
    u32 w = (u32)(x.w[hp >> 1] >> (32 * (hp & 1)));
    while (w) {
      const u32 b = (u32)__ffs((int)w) - 1u;
      w &= w - 1u;
      const u32 p = 32u * hp + b;
      v += d1[p];
      const double *row = d2 + p * (u32)sorb;
#pragma unroll
      for (int hq = 0; hq <= hp; ++hq) {
        u32 u = (u32)(x.w[hq >> 1] >> (32 * (hq & 1)));
        if (hq == hp) u &= (1u << b) - 1u;
        const double *rq = row + 32 * hq;
        while (u) {
          const u32 q = (u32)__ffs((int)u) - 1u;
          u &= u - 1u;
          v += rq[q];
        }
      }
    }
  }
  return v;
}

// TAB: the diagonal terms in shared memory (sorb (sorb + 1) doubles), else read from h1e / h2e
template <int L, bool TAB>
__global__ void __launch_bounds__(kPt2RunThreads)
pt2_run_kernel(const u64 *__restrict__ xs, const u64 *__restrict__ ps, const int *__restrict__ starts, const int *__restrict__ num_runs,
               long long R, const double *__restrict__ h1e, const double *__restrict__ h2e, int sorb, int nele,
               const double *__restrict__ C, long long ldc, int k, const double *__restrict__ E, double *__restrict__ partial) {
  extern __shared__ __align__(16) unsigned char pt2_smem[];
  double *d2 = reinterpret_cast<double *>(pt2_smem);
  double *d1 = d2 + sorb * sorb;
  __shared__ double wsum[kPt2RunThreads / 32][kPt2MaxRoots];
  if (TAB) {
    for (int t = threadIdx.x; t < sorb * sorb; t += kPt2RunThreads) {
      const u32 p = (u32)t / (u32)sorb, q = (u32)t - p * (u32)sorb;
      d2[t] = two_body<double>(h2e, p, q, p, q);
    }
    for (int p = threadIdx.x; p < sorb; p += kPt2RunThreads) d1[p] = __ldg(h1e + (size_t)p * sorb + p);
    __syncthreads();
  }
  double e[kPt2MaxRoots], acc[kPt2MaxRoots];
#pragma unroll
  for (int r = 0; r < kPt2MaxRoots; ++r) {
    e[r] = r < k ? __ldg(E + r) : 0.0;
    acc[r] = 0.0;
  }
  const long long nruns = *num_runs;
  for (long long run = (long long)blockIdx.x * kPt2RunThreads + threadIdx.x; run < nruns; run += (long long)kPt2RunBlocks * kPt2RunThreads) {
    const long long b = __ldg(starts + run), end = run + 1 < nruns ? __ldg(starts + run + 1) : R;
    double num[kPt2MaxRoots];
#pragma unroll
    for (int r = 0; r < kPt2MaxRoots; ++r) num[r] = 0.0;
    for (long long p = b; p < end; ++p) {
      const double2 hs = __ldg(reinterpret_cast<const double2 *>(ps) + p);
      const double *c = C + __double_as_longlong(hs.y) * ldc;
#pragma unroll
      for (int r = 0; r < kPt2MaxRoots; ++r)
        if (r < k) num[r] += hs.x * __ldg(c + r);
    }
    const Onv<L> a = load_onv<L>(xs + b * L);
    const double haa = TAB ? pt2_diag_table<L>(a, d1, d2, sorb) : diag_element<L, double>(a, h1e, h2e, sorb, nele);
#pragma unroll
    for (int r = 0; r < kPt2MaxRoots; ++r)
      if (r < k) acc[r] += num[r] * num[r] / (e[r] - haa);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int r = 0; r < kPt2MaxRoots; ++r) {
    for (int o = 16; o > 0; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
    if (lane == 0) wsum[warp][r] = acc[r];
  }
  __syncthreads();
  if (threadIdx.x < kPt2MaxRoots) {
    double t = 0.0;
    for (int w = 0; w < kPt2RunThreads / 32; ++w) t += wsum[w][threadIdx.x];
    partial[blockIdx.x * kPt2MaxRoots + threadIdx.x] = t;
  }
}

// acc[r] += the blocks' partials in block order; externals[0] += the number of runs
__global__ void __launch_bounds__(32) pt2_finish_kernel(const double *__restrict__ partial, const int *__restrict__ num_runs, int k,
                                                        double *__restrict__ acc, long long *__restrict__ externals) {
  const int r = threadIdx.x;
  if (r < k) {
    double t = 0.0;
    for (int b = 0; b < kPt2RunBlocks; ++b) t += partial[b * kPt2MaxRoots + r];
    acc[r] += t;
  }
  if (r == 0 && externals != nullptr) externals[0] += (long long)*num_runs;
}

// ---- scratch: records, sorted records, the table sort's workspace, run starts, partials, cub temporaries ----------------
long long sort_workspace_bytes(long long N);
int launch_sort_table(const u64 *key, const void *psi, long long N, int L, int sorb, int psi_bytes, u64 *key_out, void *psi_out,
                      long long *perm_out, void *ws, long long ws_bytes, cudaStream_t st);

struct Pt2Layout {
  long long x_in, p_in, x_s, p_s, sort, starts, num_runs, partial, cub, total;
  long long sort_bytes, cub_bytes;
};

// the scan of N + 1 offsets and the selection of R run heads: reserved here, checked against cub's own figures at launch
static long long pt2_cub_reserve(long long N, long long R) { return 2 * (N + R) + (4LL << 20); }

static Pt2Layout pt2_layout(long long N, long long R, int L) {
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  Pt2Layout l;
  l.x_in = 0;
  l.p_in = up(l.x_in + 8LL * L * R);
  l.x_s = up(l.p_in + 16 * R);
  l.p_s = up(l.x_s + 8LL * L * R);
  l.sort = up(l.p_s + 16 * R);
  l.sort_bytes = R > 0 ? sort_workspace_bytes(R) : 0;
  l.starts = up(l.sort + l.sort_bytes);
  l.num_runs = up(l.starts + 4 * R);
  l.partial = up(l.num_runs + 8);
  l.cub = up(l.partial + 8LL * kPt2RunBlocks * kPt2MaxRoots);
  l.cub_bytes = pt2_cub_reserve(N, R);
  l.total = l.cub + l.cub_bytes;
  return l;
}

long long pt2_scratch_bytes(long long N, long long R, int L) { return pt2_layout(N, R, L).total; }

template <typename F>
static int pt2_cub(const char *what, char *temp, long long reserved, F f) {
  size_t tmp = 0;
  cudaError_t e = f(nullptr, tmp);
  if (e == cudaSuccess && (long long)tmp > reserved) {
    set_error("pt2 %s: %zu bytes of temporary storage needed, %lld reserved", what, tmp, reserved);
    return 4;
  }
  if (e == cudaSuccess) e = f(temp, tmp);
  if (e != cudaSuccess) {
    set_error("pt2 %s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
    return 3;
  }
  return 0;
}

static int pt2_check_scratch(const Pt2Layout &l, long long scratch_bytes) {
  if (scratch_bytes < l.total) {
    set_error("pt2 scratch too small: %lld < %lld bytes", scratch_bytes, l.total);
    return 4;
  }
  return 0;
}

template <int L, bool EMIT>
static int pt2_rows_L(const double *h1e, const void *prep_ws, const Pt2Sel &sel, long long *offsets, u64 *x_out, u64 *pay_out,
                      const ExcGeom &g, cudaStream_t st) {
  const size_t smem = sizeof(OrbLists) + sizeof(EnumEntry<L>) * (size_t)table_offsets(g).total;
  auto kern = pt2_rows_kernel<L, EMIT>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("pt2_rows_kernel smem opt-in");
  kern<<<(unsigned)sel.N, kEnumThreads, smem, st>>>(h1e, prep_view<double>(prep_ws, g.sorb), sel, offsets, x_out, pay_out, g);
  count_launch();
  return check_launch(EMIT ? "pt2_rows_kernel (emit)" : "pt2_rows_kernel (count)");
}

// 0 < N < 2^31, 0 <= part < 2^log2_parts; arguments checked by pynqs_pt2_count / _emit.  emit = 0: offsets[N + 1] <- the
// exclusive prefix of the rows' counts (offsets[N] = the pass's pairs); emit = 1: the records of the R = offsets[N] pairs
int launch_pt2_rows(const u64 *key, long long N, const double *h1e, const void *prep_ws, const void *group_ws, int part, int log2_parts,
                    long long *offsets, long long R, void *scratch, long long scratch_bytes, const ExcGeom &g, int emit, cudaStream_t st) {
  const Pt2Layout l = pt2_layout(N, R, g.L);
  if (int rc = pt2_check_scratch(l, scratch_bytes)) return rc;
  char *sc = static_cast<char *>(scratch);
  Pt2Sel sel;
  sel.key = key;
  sel.N = N;
  sel.gv = group_view(group_ws, N, g.L);
  sel.dup = false;  // the caller refuses tables with duplicate keys
  sel.part = (u32)part;
  sel.log2_parts = (u32)log2_parts;
  u64 *x_out = reinterpret_cast<u64 *>(sc + l.x_in), *pay_out = reinterpret_cast<u64 *>(sc + l.p_in);
  int rc = 0;
#define PYNQS_PT2_ROWS(LL)                                                                                     \
  case LL:                                                                                                     \
    rc = emit ? pt2_rows_L<LL, true>(h1e, prep_ws, sel, offsets, x_out, pay_out, g, st)                        \
              : pt2_rows_L<LL, false>(h1e, prep_ws, sel, offsets, nullptr, nullptr, g, st);                   \
    break;
  switch (g.L) {
    PYNQS_PT2_ROWS(1)
    PYNQS_PT2_ROWS(2)
    PYNQS_PT2_ROWS(3)
    default: set_error("unsupported ONV length L=%d", g.L); return 1;
  }
#undef PYNQS_PT2_ROWS
  if (rc || emit) return rc;
  if (cudaMemsetAsync(offsets + N, 0, 8, st) != cudaSuccess) return check_launch("pt2 offsets memset");
  rc = pt2_cub("scan", sc + l.cub, l.cub_bytes,
               [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, offsets, offsets, (int)(N + 1), st); });
  count_launch(2);
  return rc;
}

// 0 < R < 2^31: the records sorted by determinant, stable
int launch_pt2_sort(long long N, long long R, int sorb, void *scratch, long long scratch_bytes, cudaStream_t st) {
  const int L = (sorb - 1) / 64 + 1;
  const Pt2Layout l = pt2_layout(N, R, L);
  if (int rc = pt2_check_scratch(l, scratch_bytes)) return rc;
  char *sc = static_cast<char *>(scratch);
  return launch_sort_table(reinterpret_cast<const u64 *>(sc + l.x_in), sc + l.p_in, R, L, sorb, 16, reinterpret_cast<u64 *>(sc + l.x_s),
                           sc + l.p_s, nullptr, sc + l.sort, l.sort_bytes, st);
}

template <int L>
static int pt2_runs_L(const Pt2Layout &l, char *sc, long long R, const double *h1e, const double *h2e, int sorb, int nele, const double *C,
                      long long ldc, int k, const double *E, cudaStream_t st) {
  const u64 *xs = reinterpret_cast<const u64 *>(sc + l.x_s);
  int *starts = reinterpret_cast<int *>(sc + l.starts), *num_runs = reinterpret_cast<int *>(sc + l.num_runs);
  const Pt2Head<L> head{xs};
  if (int rc = pt2_cub("run heads", sc + l.cub, l.cub_bytes, [&](void *t, size_t &b) {
        return cub::DeviceSelect::If(t, b, thrust::counting_iterator<int>(0), starts, num_runs, (int)R, head, st);
      }))
    return rc;
  count_launch();
  const u64 *ps = reinterpret_cast<const u64 *>(sc + l.p_s);
  double *partial = reinterpret_cast<double *>(sc + l.partial);
  const size_t smem = sizeof(double) * ((size_t)sorb * sorb + sorb);
  if (smem <= 100 * 1024) {
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(pt2_run_kernel<L, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("pt2_run_kernel smem opt-in");
    pt2_run_kernel<L, true><<<kPt2RunBlocks, kPt2RunThreads, smem, st>>>(xs, ps, starts, num_runs, R, h1e, h2e, sorb, nele, C, ldc, k, E,
                                                                         partial);
  } else {
    pt2_run_kernel<L, false><<<kPt2RunBlocks, kPt2RunThreads, 0, st>>>(xs, ps, starts, num_runs, R, h1e, h2e, sorb, nele, C, ldc, k, E,
                                                                       partial);
  }
  count_launch();
  return check_launch("pt2_run_kernel");
}

// 0 < R < 2^31, 1 <= k <= 8, the records sorted: acc[r] += this pass's sum over its externals, externals[0] += their number
int launch_pt2_reduce(long long N, long long R, const double *h1e, const double *h2e, int sorb, int nele, const double *C, long long ldc,
                      int k, const double *E, void *scratch, long long scratch_bytes, double *acc, long long *externals, cudaStream_t st) {
  const int L = (sorb - 1) / 64 + 1;
  const Pt2Layout l = pt2_layout(N, R, L);
  if (int rc = pt2_check_scratch(l, scratch_bytes)) return rc;
  char *sc = static_cast<char *>(scratch);
  int rc;
  switch (L) {
    case 1: rc = pt2_runs_L<1>(l, sc, R, h1e, h2e, sorb, nele, C, ldc, k, E, st); break;
    case 2: rc = pt2_runs_L<2>(l, sc, R, h1e, h2e, sorb, nele, C, ldc, k, E, st); break;
    case 3: rc = pt2_runs_L<3>(l, sc, R, h1e, h2e, sorb, nele, C, ldc, k, E, st); break;
    default: set_error("unsupported ONV length L=%d", L); return 1;
  }
  if (rc) return rc;
  pt2_finish_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const double *>(sc + l.partial), reinterpret_cast<const int *>(sc + l.num_runs), k,
                                      acc, externals);
  count_launch();
  return check_launch("pt2_finish_kernel");
}

}  // namespace pynqs
