// enumerate.cu -- connected-determinant enumeration, optionally fused with <x|H|x'>.
//
// Replaces the reference's K1 (get_merged_ovlst_kernel, cuda/kernel.cu:147-166), K2
// (get_comb_SD_kernel, :195-222) and K5 (get_comb_SD_fused_kernel, :224-277) plus the
// `repeat` pre-fill of cuda_tensor.cpp:239.  Differences in design, not in results:
//   * no merged[n, sorb] tensor in HBM: one warp derives the occupied/virtual lists from
//     popcounts of the bra words; all threads then build the per-sample excitation tables
//     (tables.cuh) in shared memory, so a row costs one exact multiply-shift division, two LDS
//     and one coalesced-ish gather from the prepared integrals (prepare.cu);
//   * every output byte is written exactly once: the 32 lanes of a warp own 32 consecutive rows,
//     so one store instruction writes 256 (L = 1) or 512 (L = 2, ulonglong2 per lane) contiguous
//     bytes of comb and 256 contiguous bytes of Hmat;
//   * 64-bit flat indexing (the reference overflows int beyond 2^31 elements);
//   * the diagonal <x|H|x> runs in its own thread-per-sample kernel, so no lane of the
//     enumeration warps serialises nele^2/2 gathers.
// Two kernels: enumerate_kernel (tables + prepared integrals; the production path) and
// enumerate_plain_kernel (decodes every row from the packed arrays; used when no prepared
// workspace is given, and as an on-device cross-check in the tests).
#include "enum_rows.cuh"

namespace pynqs {

template <int L>
__device__ __forceinline__ void store_pair_rows(u64 *dst, const Onv<L> &r0, const Onv<L> &r1) {
  // dst is 16-byte aligned (flat row index even); 2L words contiguous
  u64 buf[2 * L];
#pragma unroll
  for (int i = 0; i < L; ++i) {
    buf[i] = r0.w[i];
    buf[L + i] = r1.w[i];
  }
  ulonglong2 *d2 = reinterpret_cast<ulonglong2 *>(dst);
#pragma unroll
  for (int i = 0; i < L; ++i) d2[i] = make_ulonglong2(buf[2 * i], buf[2 * i + 1]);
}

template <int L>
__device__ __forceinline__ void store_row(u64 *dst, const Onv<L> &r) {
#pragma unroll
  for (int i = 0; i < L; ++i) dst[i] = r.w[i];
}

template <typename T>
__device__ __forceinline__ void store_pair_vals(T *dst, T a, T b);
template <>
__device__ __forceinline__ void store_pair_vals<double>(double *dst, double a, double b) {
  *reinterpret_cast<double2 *>(dst) = make_double2(a, b);
}
template <>
__device__ __forceinline__ void store_pair_vals<float>(float *dst, float a, float b) {
  *reinterpret_cast<float2 *>(dst) = make_float2(a, b);
}

// Rows [lo, hi) of one excitation class.  A warp takes chunks of 32 * ROWS consecutive rows; lane l owns rows
// chunk + l + 32 j, so each store instruction of the warp covers 32 consecutive rows (256 contiguous bytes of
// comb at L = 1 and of Hmat): coalesced, every byte written once.
template <int L, typename T, bool WITH_H, int CLS, int ROWS>
__device__ __forceinline__ void enumerate_class(const Onv<L> &x, const EnumEntry<L> *__restrict__ tab, const TableOffsets &to,
                                                const ExcGeom &g, const OrbLists &lists, const T *__restrict__ h1e,
                                                const PrepView<T> &prep, u64 *__restrict__ comb_s, T *__restrict__ hmat_s,
                                                int lo, int hi, int first_warp = 0) {
  // (first_warp: the warp that takes the first chunk -- the beta singles start where the alpha singles ended, so that the
  //  two serial 31-term sums of a sample's singles run on different warps)
  const int lane = threadIdx.x & 31, warp = ((threadIdx.x >> 5) - first_warp) & (kEnumThreads / 32 - 1);
  constexpr int kChunk = 32 * ROWS;
  for (int c = lo + warp * kChunk; c < hi; c += (kEnumThreads / 32) * kChunk) {
    Onv<L> row[ROWS];
    T val[ROWS];
    u32 sgn[ROWS];
    class_rows<L, T, WITH_H, CLS, ROWS>(x, tab, to, g, lists, h1e, prep, c, hi, row, val, sgn);
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      const int m = c + lane + 32 * j;
      if (m < hi) {
        store_row_vec<L>(comb_s + (size_t)m * L, row[j]);
        if (WITH_H) hmat_s[m] = flip_sign((T)1.0 * val[j], sgn[j]);
      }
    }
  }
}

// One CTA = one tile of one sample.
template <int L, typename T, bool WITH_H>
__global__ void __launch_bounds__(kEnumThreads)
enumerate_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, PrepView<T> prep, u64 *__restrict__ comb,
                 T *__restrict__ hmat, long long n, int tiles_per_sample, int tile_rows, ExcGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  OrbLists &lists = *reinterpret_cast<OrbLists *>(smem_raw);
  EnumEntry<L> *tab = reinterpret_cast<EnumEntry<L> *>(smem_raw + sizeof(OrbLists));

  const long long s = blockIdx.x / tiles_per_sample;
  const int tile = blockIdx.x - (int)(s * tiles_per_sample);
  if (s >= n) return;
  const Onv<L> x = load_onv<L>(bra + s * L);
  if (threadIdx.x < 32) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x);
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

  const long long M = (long long)g.nsd + 1;
  u64 *comb_s = comb + s * M * L;   // this sample's rows
  T *hmat_s = WITH_H ? hmat + s * M : nullptr;
  const long long tb = (long long)tile * tile_rows;
  const int t_lo = (int)tb, t_hi = (int)(tb + tile_rows < M ? tb + tile_rows : M);
  if (tile == 0 && threadIdx.x == 0) store_row_vec<L>(comb_s, x);  // row 0 = bra (its H belongs to diag_kernel)
  auto clip_lo = [&](int v) { return v > t_lo ? v : t_lo; };
  auto clip_hi = [&](int v) { return v < t_hi ? v : t_hi; };
  enumerate_class<L, T, WITH_H, 0, 1>(x, tab, to, g, lists, h1e, prep, comb_s, hmat_s, clip_lo(1), clip_hi(g.d0 + 1));
  enumerate_class<L, T, WITH_H, 1, 1>(x, tab, to, g, lists, h1e, prep, comb_s, hmat_s, clip_lo(g.d0 + 1), clip_hi(g.d1 + 1),
                                      ((g.d0 + 31) >> 5) & (kEnumThreads / 32 - 1));
  enumerate_class<L, T, WITH_H, 2, kRowsPerThread>(x, tab, to, g, lists, h1e, prep, comb_s, hmat_s, clip_lo(g.d1 + 1), clip_hi(g.d2 + 1));
  enumerate_class<L, T, WITH_H, 3, kRowsPerThread>(x, tab, to, g, lists, h1e, prep, comb_s, hmat_s, clip_lo(g.d2 + 1), clip_hi(g.d3 + 1));
  enumerate_class<L, T, WITH_H, 4, kRowsPerThread>(x, tab, to, g, lists, h1e, prep, comb_s, hmat_s, clip_lo(g.d3 + 1), clip_hi((int)M));
}

// ---- plain variant: every row decoded from the packed arrays ----------------------------------------
template <int L, typename T, bool WITH_H>
__global__ void __launch_bounds__(kEnumThreads)
enumerate_plain_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, const T *__restrict__ h2e, u64 *__restrict__ comb,
                       T *__restrict__ hmat, long long n, int tiles_per_sample, int tile_rows, ExcGeom g) {
  __shared__ OrbLists lists;
  const long long s = blockIdx.x / tiles_per_sample;
  const int tile = blockIdx.x - (int)(s * tiles_per_sample);
  if (s >= n) return;
  const Onv<L> x = load_onv<L>(bra + s * L);
  if (threadIdx.x < 32) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x);
  __syncthreads();

  const long long M = (long long)g.nsd + 1;
  const long long base = s * M;
  const int odd = (int)(base & 1);
  const long long m_lo = (long long)tile * tile_rows - odd;
  for (int u = threadIdx.x; u < tile_rows / 2; u += kEnumThreads) {
    const long long m0 = m_lo + 2 * u;
    if (m0 >= M) break;
    Onv<L> row[2];
    T val[2];
    bool ok[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const long long m = m0 + t;
      ok[t] = (m >= 0) && (m < M);
      row[t] = x;
      val[t] = (T)0.0;
      if (ok[t] && m > 0) {
        const Exc e = decode_exc(g, lists, (int)(m - 1));
        row[t] = apply_exc<L>(x, e);
        if (WITH_H) val[t] = exc_element<L, T>(x, e, h1e, h2e, g.sorb);
      }
    }
    if (ok[0] && ok[1]) {
      store_pair_rows<L>(comb + (base + m0) * L, row[0], row[1]);
      if (WITH_H) {
        if (m0 == 0) hmat[base + 1] = val[1];
        else store_pair_vals<T>(hmat + base + m0, val[0], val[1]);
      }
    } else {
#pragma unroll
      for (int t = 0; t < 2; ++t)
        if (ok[t]) {
          store_row<L>(comb + (base + m0 + t) * L, row[t]);
          if (WITH_H && (m0 + t) > 0) hmat[base + m0 + t] = val[t];
        }
    }
  }
}

// thread-per-sample diagonal: out[s * stride] = <x|H|x>
template <int L, typename T>
__global__ void __launch_bounds__(128)
diag_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, const T *__restrict__ h2e, T *__restrict__ out,
            long long n, long long stride, int sorb, int nele) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const Onv<L> x = load_onv<L>(bra + s * L);
  out[s * stride] = diag_element<L, T>(x, h1e, h2e, sorb, nele);
}

// Same sum from a per-CTA table in shared memory: D2[p][q] = <pq||pq> and D1[p] = h1e[p,p] are gathered ONCE per
// CTA (sorb^2 entries) instead of once per sample and term, so a term is a shared-memory load and an add --
// the same values added in the same order as diag_element (cpp_src/cpu/hamiltonian.cpp:33-50).  Each thread
// takes kDiagPerThread samples.  Used when the table fits in shared memory (sorb <= ~160 for float64).
constexpr int kDiagThreads = 128;

template <int L, typename T>
__global__ void __launch_bounds__(kDiagThreads)
diag_table_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, const T *__restrict__ h2e, T *__restrict__ out,
                  long long n, long long stride, int sorb, int nele, int per_thread) {
  extern __shared__ __align__(16) unsigned char diag_smem[];
  T *d2 = reinterpret_cast<T *>(diag_smem);
  T *d1 = d2 + sorb * sorb;
  for (int t = threadIdx.x; t < sorb * sorb; t += kDiagThreads) {
    const u32 p = (u32)t / (u32)sorb, q = (u32)t - p * (u32)sorb;
    d2[t] = two_body<T>(h2e, p, q, p, q);
  }
  for (int p = threadIdx.x; p < sorb; p += kDiagThreads) d1[p] = __ldg(h1e + (size_t)p * sorb + p);
  __syncthreads();
  const long long first = (long long)blockIdx.x * (kDiagThreads * per_thread) + threadIdx.x;
  for (int it = 0; it < per_thread; ++it) {
    const long long s = first + (long long)it * kDiagThreads;
    if (s >= n) return;
    const Onv<L> x = load_onv<L>(bra + s * L);
    int occ = 0;
#pragma unroll
    for (int i = 0; i < L; ++i) occ += __popcll(x.w[i]);
    T v = (T)0.0;
    if (occ == nele) {
      // every occupied orbital p ascending, and for each the occupied q < p ascending: 32-bit words, lowest
      // set bit first (w & (w - 1) clears it)
#pragma unroll
      for (int hp = 0; hp < 2 * L; ++hp) {
        u32 w = (u32)(x.w[hp >> 1] >> (32 * (hp & 1)));
        while (w) {
          const u32 b = (u32)__ffs((int)w) - 1u;
          w &= w - 1u;
          const u32 p = 32u * hp + b;
          v += d1[p];
          const T *row = d2 + p * (u32)sorb;
#pragma unroll
          for (int hq = 0; hq <= hp; ++hq) {
            u32 u = (u32)(x.w[hq >> 1] >> (32 * (hq & 1)));
            if (hq == hp) u &= (1u << b) - 1u;
            const T *rq = row + 32 * hq;
            while (u) {
              const u32 q = (u32)__ffs((int)u) - 1u;
              u &= u - 1u;
              v += rq[q];
            }
          }
        }
      }
    } else {  // electron count differs from nele: the reference's zero-padded list, term by term
      Onv<L> outer = x;
      for (int a = 0; a < nele; ++a) {
        u32 p = 0;
#pragma unroll
        for (int i = 0; i < L; ++i) {
          if (outer.w[i]) {
            const int b = __ffsll((long long)outer.w[i]) - 1;
            outer.w[i] ^= 1ull << b;
            p = (u32)(64 * i + b);
            break;
          }
        }
        v += d1[p];
        Onv<L> inner = x;
        for (int c = 0; c < a; ++c) {
          u32 q = 0;
#pragma unroll
          for (int i = 0; i < L; ++i) {
            if (inner.w[i]) {
              const int b = __ffsll((long long)inner.w[i]) - 1;
              inner.w[i] ^= 1ull << b;
              q = (u32)(64 * i + b);
              break;
            }
          }
          v += d2[p * (u32)sorb + q];
        }
      }
    }
    out[s * stride] = v;
  }
}

template <int L, typename T>
static int launch_diag_LT(const u64 *bra, const T *h1e, const T *h2e, T *out, long long n, long long stride, int sorb, int nele,
                          cudaStream_t st) {
  const size_t smem = sizeof(T) * ((size_t)sorb * sorb + sorb);
  if (smem <= 200 * 1024 && n >= 4096) {  // below that the table build would dominate
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(diag_table_kernel<L, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return check_launch("diag_table_kernel smem opt-in");
    // samples per thread: up to 4, fewer when that would leave SMs without a CTA
    int per_thread = (int)(n / (148LL * 4 * kDiagThreads));
    per_thread = per_thread < 1 ? 1 : (per_thread > 4 ? 4 : per_thread);
    const long long per = (long long)kDiagThreads * per_thread;
    diag_table_kernel<L, T><<<(unsigned)((n + per - 1) / per), kDiagThreads, smem, st>>>(bra, h1e, h2e, out, n, stride, sorb, nele,
                                                                                       per_thread);
    count_launch();
    return check_launch("diag_table_kernel");
  }
  diag_kernel<L, T><<<(unsigned)((n + 127) / 128), 128, 0, st>>>(bra, h1e, h2e, out, n, stride, sorb, nele);
  count_launch();
  return check_launch("diag_kernel");
}

// flag_bit=True companion of get_comb_tensor: states[n, M, sorb] = +-1 of every comb row
// (cpu_tensor.cpp:186-190, excitation.cpp:171-181)
template <int L>
__global__ void __launch_bounds__(256)
states_kernel(const u64 *__restrict__ comb, double *__restrict__ states, long long rows, int sorb) {
  const long long total = rows * sorb;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / sorb;
    const int k = (int)(i - r * sorb);
    const u64 w = comb[r * L + (k >> 6)];
    states[i] = ((w >> (k & 63)) & 1ull) ? 1.0 : -1.0;
  }
}

// rows of one sample per CTA: whole sample when that still gives >= ~8 CTAs per SM, else split
static void choose_tiling(long long n, long long M, int &tiles, int &tile_rows) {
  const long long rows = M;
  long long want_tiles = 1;
  if (n > 0 && n < 148LL * 8) want_tiles = (148LL * 8 + n - 1) / n;
  long long tr = (rows + want_tiles - 1) / want_tiles;
  if (tr < 2048) tr = 2048;
  if (tr > 32768) tr = 32768;
  tr = (tr + 511) / 512 * 512;
  tile_rows = (int)tr;
  tiles = (int)((rows + tr - 1) / tr);
}

template <int L, typename T, bool WITH_H>
static int launch_enumerate_L(const u64 *bra, const T *h1e, const T *h2e, const void *prep_ws, u64 *comb, T *hmat, long long n,
                              const ExcGeom &g, cudaStream_t st) {
  const long long M = (long long)g.nsd + 1;
  int tiles, tile_rows;
  choose_tiling(n, M, tiles, tile_rows);
  const long long blocks = n * tiles;
  if (blocks > 0x7fffffffLL) {
    set_error("enumerate: n * tiles = %lld exceeds the grid limit; split the batch", blocks);
    return 1;
  }
  const bool use_tables = (prep_ws != nullptr) || !WITH_H;
  if (use_tables) {
    const size_t smem = sizeof(OrbLists) + sizeof(EnumEntry<L>) * (size_t)table_offsets(g).total;
    auto kern = enumerate_kernel<L, T, WITH_H>;
    if (smem > 48 * 1024) {
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("enumerate_kernel smem opt-in");
    }
    PrepView<T> pv = prep_view<T>(prep_ws, g.sorb);
    kern<<<(unsigned)blocks, kEnumThreads, smem, st>>>(bra, h1e, pv, comb, hmat, n, tiles, tile_rows, g);
    count_launch();
    if (int rc = check_launch("enumerate_kernel")) return rc;
  } else {
    enumerate_plain_kernel<L, T, WITH_H><<<(unsigned)blocks, kEnumThreads, 0, st>>>(bra, h1e, h2e, comb, hmat, n, tiles, tile_rows, g);
    count_launch();
    if (int rc = check_launch("enumerate_plain_kernel")) return rc;
  }
  if (WITH_H) {
    if (int rc = launch_diag_LT<L, T>(bra, h1e, h2e, hmat, n, M, g.sorb, g.nele, st)) return rc;
  }
  return 0;
}

template <typename T, bool WITH_H>
static int launch_enumerate_T(const u64 *bra, const T *h1e, const T *h2e, const void *prep_ws, u64 *comb, T *hmat, long long n,
                              const ExcGeom &g, cudaStream_t st) {
  switch (g.L) {
    case 1: return launch_enumerate_L<1, T, WITH_H>(bra, h1e, h2e, prep_ws, comb, hmat, n, g, st);
    case 2: return launch_enumerate_L<2, T, WITH_H>(bra, h1e, h2e, prep_ws, comb, hmat, n, g, st);
    case 3: return launch_enumerate_L<3, T, WITH_H>(bra, h1e, h2e, prep_ws, comb, hmat, n, g, st);
  }
  set_error("unsupported ONV length L=%d", g.L);
  return 1;
}

int launch_comb(const u64 *bra, u64 *comb, long long n, const ExcGeom &g, cudaStream_t st) {
  return launch_enumerate_T<double, false>(bra, nullptr, nullptr, nullptr, comb, nullptr, n, g, st);
}

int launch_comb_hij_f64(const u64 *bra, const double *h1e, const double *h2e, const void *prep_ws, u64 *comb, double *hmat,
                        long long n, const ExcGeom &g, cudaStream_t st) {
  return launch_enumerate_T<double, true>(bra, h1e, h2e, prep_ws, comb, hmat, n, g, st);
}

int launch_comb_hij_f32(const u64 *bra, const float *h1e, const float *h2e, const void *prep_ws, u64 *comb, float *hmat,
                        long long n, const ExcGeom &g, cudaStream_t st) {
  return launch_enumerate_T<float, true>(bra, h1e, h2e, prep_ws, comb, hmat, n, g, st);
}

// stand-alone diagonal (used by the fused local-energy op): out[s * stride] = <x_s|H|x_s>
int launch_diag_f64(const u64 *bra, const double *h1e, const double *h2e, double *out, long long n, long long stride, int L,
                    int sorb, int nele, cudaStream_t st) {
  if (n == 0) return 0;
  switch (L) {
    case 1: return launch_diag_LT<1, double>(bra, h1e, h2e, out, n, stride, sorb, nele, st);
    case 2: return launch_diag_LT<2, double>(bra, h1e, h2e, out, n, stride, sorb, nele, st);
    case 3: return launch_diag_LT<3, double>(bra, h1e, h2e, out, n, stride, sorb, nele, st);
  }
  set_error("unsupported ONV length L=%d", L);
  return 1;
}

// the same for either element type (reduce_sample.cu)
template <int L, typename T>
int launch_diag_plain(const u64 *bra, const T *h1e, const T *h2e, T *out, long long n, long long stride, int sorb, int nele, cudaStream_t st) {
  return launch_diag_LT<L, T>(bra, h1e, h2e, out, n, stride, sorb, nele, st);
}
#define PYNQS_DIAG_INST(LL, TT) \
  template int launch_diag_plain<LL, TT>(const u64 *, const TT *, const TT *, TT *, long long, long long, int, int, cudaStream_t);
PYNQS_DIAG_INST(1, double) PYNQS_DIAG_INST(2, double) PYNQS_DIAG_INST(3, double)
PYNQS_DIAG_INST(1, float) PYNQS_DIAG_INST(2, float) PYNQS_DIAG_INST(3, float)
#undef PYNQS_DIAG_INST

int launch_states(const u64 *comb, double *states, long long rows, int sorb, cudaStream_t st) {
  const int L = (sorb - 1) / 64 + 1;
  const long long total = rows * sorb;
  if (total == 0) return 0;
  const unsigned blocks = (unsigned)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  switch (L) {
    case 1: states_kernel<1><<<blocks, 256, 0, st>>>(comb, states, rows, sorb); break;
    case 2: states_kernel<2><<<blocks, 256, 0, st>>>(comb, states, rows, sorb); break;
    default: states_kernel<3><<<blocks, 256, 0, st>>>(comb, states, rows, sorb); break;
  }
  count_launch();
  return check_launch("states_kernel");
}

// ---- REDUCE method: only the connected determinants with |<x|H|x'>| >= eps ----------------------------------
// The reference materialises comb [n, M, 8L] and Hmat [n, M], then keeps torch.where(|Hmat| >= eps)
// (vmc/energy/eloc.py:257-297).  Here nothing of size [n, M] is written: a counting pass, an exclusive scan,
// and an emitting pass that recomputes the rows and writes the kept ones -- determinant, value and flat index
// s * M + m -- in exactly torch.where's order (ascending flat index).  One CTA per sample; inside a CTA the
// rows go through in chunks of 8 warps x 32 ROWS, and the kept rows of a chunk are ranked with ballots
// (inside a warp) and a prefix over the warps' counts (shared memory), so the order does not depend on timing.
template <int L, typename T, int CLS, int ROWS, bool EMIT>
__device__ __forceinline__ void reduce_class(const Onv<L> &x, const EnumEntry<L> *__restrict__ tab, const TableOffsets &to,
                                             const ExcGeom &g, const OrbLists &lists, const T *__restrict__ h1e,
                                             const PrepView<T> &prep, int lo, int hi, T eps, u32 &kept, u32 *warp_cnt,
                                             long long out_base, long long flat_base, u64 *__restrict__ x_out,
                                             T *__restrict__ h_out, long long *__restrict__ idx_out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kChunk = 32 * ROWS, kWarps = kEnumThreads / 32;
  for (int c0 = lo; c0 < hi; c0 += kWarps * kChunk) {  // same trip count for every warp: there are barriers inside
    const int c = c0 + warp * kChunk;
    Onv<L> row[ROWS];
    T val[ROWS];
    u32 sgn[ROWS];
    class_rows<L, T, true, CLS, ROWS>(x, tab, to, g, lists, h1e, prep, c, hi, row, val, sgn);
    u32 bal[ROWS], wc = 0;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      const int m = c + lane + 32 * j;
      bal[j] = __ballot_sync(0xffffffffu, m < hi && fabs(val[j]) >= eps);
      wc += (u32)__popc(bal[j]);
    }
    if (!EMIT) {
      kept += wc;  // per-warp tally, summed at the end
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
        store_row<L>(x_out + o * L, row[j]);
        h_out[o] = flip_sign((T)1.0 * val[j], sgn[j]);
        idx_out[o] = flat_base + (c + lane + 32 * j);
      }
      pos += (u32)__popc(bal[j]);
    }
    kept += total;
    __syncthreads();
  }
}

template <int L, typename T, bool EMIT>
__global__ void __launch_bounds__(kEnumThreads)
reduce_kernel(const u64 *__restrict__ bra, const T *__restrict__ h1e, PrepView<T> prep, const T *__restrict__ diag, T eps,
              long long *__restrict__ offsets, u64 *__restrict__ x_out, T *__restrict__ h_out, long long *__restrict__ idx_out,
              long long n, ExcGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  OrbLists &lists = *reinterpret_cast<OrbLists *>(smem_raw);
  EnumEntry<L> *tab = reinterpret_cast<EnumEntry<L> *>(smem_raw + sizeof(OrbLists));
  __shared__ u32 warp_cnt[kEnumThreads / 32];
  __shared__ unsigned long long s_total;
  const long long s = blockIdx.x;
  if (s >= n) return;
  const Onv<L> x = load_onv<L>(bra + s * L);
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

  const long long M = (long long)g.nsd + 1;
  const long long out_base = EMIT ? offsets[s] : 0, flat_base = s * M;
  // row 0: the sample itself with <x|H|x>
  const T hii = diag[s];
  const bool keep0 = fabs(hii) >= eps;
  u32 kept = 0;
  if (EMIT) {
    kept = keep0 ? 1u : 0u;  // uniform running count of the CTA
    if (keep0 && threadIdx.x == 0) {
      store_row<L>(x_out + out_base * L, x);
      h_out[out_base] = hii;
      idx_out[out_base] = flat_base;
    }
  } else if (threadIdx.x == 0 && keep0) {
    kept = 1u;  // tallies are per warp (lane-uniform); warp 0 carries row 0
  }
  if (!EMIT) kept = __shfl_sync(0xffffffffu, kept, 0);
  const int Mi = (int)M;
  reduce_class<L, T, 0, 1, EMIT>(x, tab, to, g, lists, h1e, prep, 1, g.d0 + 1, eps, kept, warp_cnt, out_base, flat_base, x_out, h_out, idx_out);
  reduce_class<L, T, 1, 1, EMIT>(x, tab, to, g, lists, h1e, prep, g.d0 + 1, g.d1 + 1, eps, kept, warp_cnt, out_base, flat_base, x_out, h_out, idx_out);
  reduce_class<L, T, 2, kRowsPerThread, EMIT>(x, tab, to, g, lists, h1e, prep, g.d1 + 1, g.d2 + 1, eps, kept, warp_cnt, out_base, flat_base, x_out, h_out, idx_out);
  reduce_class<L, T, 3, kRowsPerThread, EMIT>(x, tab, to, g, lists, h1e, prep, g.d2 + 1, g.d3 + 1, eps, kept, warp_cnt, out_base, flat_base, x_out, h_out, idx_out);
  reduce_class<L, T, 4, kRowsPerThread, EMIT>(x, tab, to, g, lists, h1e, prep, g.d3 + 1, Mi, eps, kept, warp_cnt, out_base, flat_base, x_out, h_out, idx_out);
  if (!EMIT) {
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_total, (unsigned long long)kept);
    __syncthreads();
    if (threadIdx.x == 0) offsets[s] = (long long)s_total;  // counts; the scan turns them into offsets
  }
}

}  // namespace pynqs

#include <cub/device/device_scan.cuh>

namespace pynqs {

struct ReduceScratch {
  long long diag, cub, total;
  size_t cub_bytes;
};

static ReduceScratch reduce_scratch_layout(long long n) {
  ReduceScratch l;
  size_t tmp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp, (const long long *)nullptr, (long long *)nullptr, (int)(n + 1));
  l.diag = 0;
  l.cub = (8 * n + 255) / 256 * 256 + 256;
  l.cub_bytes = tmp;
  l.total = l.cub + (long long)tmp + 256;
  return l;
}

long long reduce_scratch_bytes(long long n) { return reduce_scratch_layout(n < 0 ? 0 : n).total; }

template <int L, typename T, bool EMIT>
static int launch_reduce_LT(const u64 *bra, const T *h1e, const T *h2e, const void *prep_ws, long long n, const ExcGeom &g, double eps,
                            void *scratch, long long *offsets, u64 *x_out, T *h_out, long long *idx_out, cudaStream_t st) {
  const ReduceScratch lay = reduce_scratch_layout(n);
  char *sc = static_cast<char *>(scratch);
  T *diag = reinterpret_cast<T *>(sc + lay.diag);
  if (int rc = launch_diag_LT<L, T>(bra, h1e, h2e, diag, n, 1, g.sorb, g.nele, st)) return rc;
  const size_t smem = sizeof(OrbLists) + sizeof(EnumEntry<L>) * (size_t)table_offsets(g).total;
  auto kern = reduce_kernel<L, T, EMIT>;
  if (smem > 48 * 1024 && cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("reduce_kernel smem opt-in");
  const PrepView<T> pv = prep_view<T>(prep_ws, g.sorb);
  kern<<<(unsigned)n, kEnumThreads, smem, st>>>(bra, h1e, pv, diag, (T)eps, offsets, x_out, h_out, idx_out, n, g);
  count_launch();
  if (int rc = check_launch("reduce_kernel")) return rc;
  if (!EMIT) {
    if (cudaMemsetAsync(offsets + n, 0, 8, st) != cudaSuccess) return check_launch("reduce offsets memset");
    size_t tmp = lay.cub_bytes;
    const cudaError_t e = cub::DeviceScan::ExclusiveSum(sc + lay.cub, tmp, offsets, offsets, (int)(n + 1), st);
    if (e != cudaSuccess) {
      set_error("reduce scan: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
      return 3;
    }
    count_launch(2);
  }
  return 0;
}

// emit = 0: offsets[n + 1] <- exclusive prefix of the per-sample counts (offsets[n] = number of kept rows);
// emit = 1: the kept rows at those offsets
template <typename T>
int launch_reduce(const u64 *bra, const T *h1e, const T *h2e, const void *prep_ws, long long n, const ExcGeom &g, double eps, int emit,
                  void *scratch, long long scratch_bytes, long long *offsets, u64 *x_out, T *h_out, long long *idx_out,
                  cudaStream_t st) {
  if (n == 0) return 0;
  if (n > 0x7fffffffLL - 1) {
    set_error("reduce: at most 2^31 - 2 samples per call (got %lld)", n);
    return 1;
  }
  if (scratch_bytes < reduce_scratch_layout(n).total) {
    set_error("reduce scratch too small: %lld < %lld bytes", scratch_bytes, reduce_scratch_layout(n).total);
    return 4;
  }
#define PYNQS_REDUCE_CASE(LL)                                                                                                     \
  case LL:                                                                                                                        \
    return emit ? launch_reduce_LT<LL, T, true>(bra, h1e, h2e, prep_ws, n, g, eps, scratch, offsets, x_out, h_out, idx_out, st)   \
                : launch_reduce_LT<LL, T, false>(bra, h1e, h2e, prep_ws, n, g, eps, scratch, offsets, x_out, h_out, idx_out, st);
  switch (g.L) {
    PYNQS_REDUCE_CASE(1)
    PYNQS_REDUCE_CASE(2)
    PYNQS_REDUCE_CASE(3)
  }
#undef PYNQS_REDUCE_CASE
  set_error("unsupported ONV length L=%d", g.L);
  return 1;
}

template int launch_reduce<double>(const u64 *, const double *, const double *, const void *, long long, const ExcGeom &, double, int,
                                   void *, long long, long long *, u64 *, double *, long long *, cudaStream_t);
template int launch_reduce<float>(const u64 *, const float *, const float *, const void *, long long, const ExcGeom &, double, int,
                                  void *, long long, long long *, u64 *, float *, long long *, cudaStream_t);

// eloc[s] = sum over the kept rows of sample s of (psi_k / psi0) * H_k, psi0 = psi of row 0 (0 when row 0 was not
// kept, as in the reference, where psi_x1[..., 0] then stays 0).  One warp per sample, fixed order.
template <bool CPLX>
__global__ void __launch_bounds__(128)
reduce_eloc_kernel(const double *__restrict__ psi, const double *__restrict__ hij, const long long *__restrict__ idx,
                   const long long *__restrict__ offsets, long long n, long long M, double *__restrict__ eloc,
                   double *__restrict__ psi0_out) {
  const int lane = threadIdx.x & 31;
  const long long s = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (s >= n) return;
  const long long b = offsets[s], e = offsets[s + 1];
  double p0r = 0.0, p0i = 0.0;
  // row 0 of the sample (flat index s * M): first of the kept rows, or -- stochastic branch with a sub-eps diagonal --
  // first of the drawn rows; absent: psi0 = 0 like the reference
  long long k0 = -1;
  for (long long k = b + lane; k < e && k0 < 0; k += 32)
    if (idx[k] == s * M) k0 = k;
  {
    const u32 found = __ballot_sync(0xffffffffu, k0 >= 0);
    if (found) {
      k0 = __shfl_sync(0xffffffffu, k0, __ffs(found) - 1);
      p0r = CPLX ? psi[2 * k0] : psi[k0];
      p0i = CPLX ? psi[2 * k0 + 1] : 0.0;
    }
  }
  double ar = 0.0, ai = 0.0;
  for (long long k = b + lane; k < e; k += 32) {
    const double h = hij[k];
    if (CPLX) {
      // numpy / c10 complex division (same formula as the one-pass kernels)
      const double a = psi[2 * k], bb = psi[2 * k + 1], c = p0r, d = p0i;
      const double ac = fabs(c), ad = fabs(d);
      double qr, qi;
      if (ac >= ad) {
        if (ac == 0.0 && ad == 0.0) {
          qr = a / ac;
          qi = bb / ad;
        } else {
          const double rat = d / c, scl = 1.0 / (c + d * rat);
          qr = (a + bb * rat) * scl;
          qi = (bb - a * rat) * scl;
        }
      } else {
        const double rat = c / d, scl = 1.0 / (d + c * rat);
        qr = (a * rat + bb) * scl;
        qi = (bb * rat - a) * scl;
      }
      ar += qr * h;
      ai += qi * h;
    } else {
      ar += (psi[k] / p0r) * h;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ar += __shfl_xor_sync(0xffffffffu, ar, o);
    if (CPLX) ai += __shfl_xor_sync(0xffffffffu, ai, o);
  }
  if (lane == 0) {
    if (CPLX) {
      eloc[2 * s] = ar;
      eloc[2 * s + 1] = ai;
      psi0_out[2 * s] = p0r;
      psi0_out[2 * s + 1] = p0i;
    } else {
      eloc[s] = ar;
      psi0_out[s] = p0r;
    }
  }
}

int launch_reduce_eloc(const double *psi, int cplx, const double *hij, const long long *idx, const long long *offsets, long long n,
                       long long M, double *eloc, double *psi0, cudaStream_t st) {
  if (n == 0) return 0;
  const unsigned blocks = (unsigned)((n + 3) / 4);
  if (cplx) reduce_eloc_kernel<true><<<blocks, 128, 0, st>>>(psi, hij, idx, offsets, n, M, eloc, psi0);
  else reduce_eloc_kernel<false><<<blocks, 128, 0, st>>>(psi, hij, idx, offsets, n, M, eloc, psi0);
  count_launch();
  return check_launch("reduce_eloc_kernel");
}

}  // namespace pynqs
