// hamiltonian.cu -- the sample-space Hamiltonian H[i, j] = <bra_i|H|key_j> as a CSR matrix, built from the hit lists of
// the one-pass scan (eloc_scan.cu, eloc_block.cu) instead of the dense get_hij_torch(bra, key) matrix.
//
// Row i holds exactly the table rows that eloc_sample_space sums over for sample i: bra_i itself (if it is in the table)
// and every single / double excitation of it that is in the table.  Two calls, the count / emit protocol of the REDUCE
// method:
//   count: the scan phase per batch, then hamiltonian_row_kernel<EMIT = false> (one warp per sample) counts the hits that
//          decode to a single or double excitation, plus the diagonal; a device exclusive scan turns the counts into the
//          row offsets.
//   emit : the scan phase again (the hit lists are not kept between the calls), hamiltonian_row_kernel<EMIT = true>
//          writes (table row, <x|H|x'>) of every entry into the row's slice -- doubles by double_element, singles one at a
//          time by the whole warp (single_element_warp), the diagonal from launch_diag_f64: the evaluation kernel's
//          arithmetic, so the values are bit-identical to get_hij_torch --, then cub::DeviceSegmentedSort orders every row
//          by column.
// Samples flagged for the reference's route (a queue or the hit buffer overflowed; every sample of a table with duplicate
// keys) take it here too: x and all nsd excitations, classic binary search, values by exc_element.  Both calls walk a row
// the same way, so a row's count does not depend on which route it took in which call.  The columns of a row are
// distinct, so the sorted result does not depend on the order the entries were written in.
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include <cub/cub.cuh>

#include "eloc.cuh"
#include "lut.cuh"

namespace pynqs {

constexpr int kHamThreads = 128;  // one warp per sample; 8 CTAs per SM (64 registers) keep the emit kernels free of spills

// EMIT = false: offsets[s] = number of entries of row s.  EMIT = true: the entries of row s into col / val
// [offsets[s], offsets[s + 1]), unsorted.
template <int L, bool HALF, bool EMIT>
__global__ void __launch_bounds__(kHamThreads, 8)
hamiltonian_row_kernel(const u64 *__restrict__ bra, long long n, const double *__restrict__ h1e, const double *__restrict__ h2e,
                       const u64 *__restrict__ key, long long N, GroupView gv, const HitRun *__restrict__ runs,
                       const u32 *__restrict__ run_cnt, int run_stride, const u32 *__restrict__ hits, const u32 *__restrict__ self_pos,
                       const double *__restrict__ hii, long long *__restrict__ offsets, long long *__restrict__ col,
                       double *__restrict__ val, ExcGeom g) {
  __shared__ OrbLists s_lists[kHamThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long s = (long long)blockIdx.x * (kHamThreads / 32) + warp;
  if (s >= n) return;
  OrbLists &lists = s_lists[warp];
  const Onv<L> x = load_onv<L>(bra + s * L);
  const int nruns = (int)run_cnt[s];
  const HitRun *my_runs = runs + s * run_stride;
  bool redo = false;
  for (int w = lane; w < nruns; w += 32) redo |= (my_runs[w].cnt & kOverflow) != 0;
  redo = __any_sync(0xffffffffu, redo);

  long long at = EMIT ? offsets[s] : 0;  // next entry of the row
  const long long end = EMIT ? offsets[s + 1] : 0;
  // the entries the lanes hold, written side by side (ballot compaction)
  auto put = [&](bool have, long long c, double v) {
    const u32 m = __ballot_sync(0xffffffffu, have);
    if (EMIT && have) {
      const long long p = at + __popc(m & ((1u << lane) - 1u));
      if (p < end) {
        col[p] = c;
        val[p] = v;
      }
    }
    at += __popc(m);
  };

  if (redo) {
    // the reference's route: x and every excitation in row order, classic binary search in the sorted table
    build_lists<L>(x, g.sorb, g.noA, g.noB, lists, lane);
    __syncwarp();
    const long long id0 = classic_search<L>(key, N, x);
    put(lane == 0 && id0 >= 0, id0, EMIT ? hii[s] : 0.0);
    for (int r0 = 0; r0 < g.nsd; r0 += 32) {
      const int r = r0 + lane;
      long long id = -1;
      double v = 0.0;
      if (r < g.nsd) {
        const Exc e = decode_exc(g, lists, r);
        id = classic_search<L>(key, N, apply_exc<L>(x, e));
        if (EMIT && id >= 0) v = exc_element<L, double>(x, e, h1e, h2e, g.sorb);
      }
      put(id >= 0, id, v);
    }
  } else {
    const u32 sp = self_pos[s];
    put(lane == 0 && sp != kNoSelf, sp != kNoSelf ? (long long)__ldg(gv.rows[0] + sp) : 0, EMIT ? hii[s] : 0.0);
    bool have_lists = false;
    for (int r = 0; r < nruns; ++r) {
      const HitRun run = my_runs[r];
      for (u32 e0 = 0; e0 < run.cnt; e0 += 32) {
        const u32 e = e0 + (u32)lane;
        Onv<L> y = x;
        u32 row = 0;
        int kind = 0;  // 1 single, 2 double, 0 nothing to add
        if (e < run.cnt) kind = decode_hit<L, HALF>(gv, x, hits[run.off + e], y, row);
        double v = 0.0;
        if (EMIT) {
          if (kind == 2) v = double_element<L, double>(x, y, h2e);
          // single excitations (rare): one at a time by the whole warp, terms gathered in parallel
          u32 pend = __ballot_sync(0xffffffffu, kind == 1);
          while (pend) {
            const int src = __ffs(pend) - 1;
            pend &= pend - 1u;
            if (!have_lists) {
              build_lists<L>(x, g.sorb, g.noA, g.noB, lists, lane);
              __syncwarp();
              have_lists = true;
            }
            Onv<L> ys;
#pragma unroll
            for (int w = 0; w < L; ++w) ys.w[w] = __shfl_sync(0xffffffffu, y.w[w], src);
            const double hv = single_element_warp<L, double>(x, ys, h1e, h2e, g.sorb, lists.occ_order, lists.n_occ);
            if (lane == src) v = hv;
          }
        }
        put(kind != 0, (long long)row, v);
      }
    }
  }
  if (!EMIT && lane == 0) offsets[s] = at;
}

// segment bounds of row i for the sort call that takes the rows starting in [lo, hi), relative to lo; other rows are empty
struct RowBound {
  const long long *offsets;
  long long lo, hi;
  int end;  // 0: begin, 1: end of the row
  __host__ __device__ int operator()(int i) const {
    const long long b = offsets[i];
    return (b >= lo && b < hi) ? (int)(offsets[i + end] - lo) : 0;
  }
};

struct HamScratch {
  ElocScratch eloc;
  long long cub, alt_col, alt_val, total;
};

// the device scan of the counts and the segment partition of the sort need O(n) temporary storage: reserved here, checked
// against cub's own figure at launch
static long long cub_reserve(long long n) { return 16 * (n + 1) + (4LL << 20); }

static HamScratch ham_layout(long long n, long long nnz, const ExcGeom &g, bool block) {
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  HamScratch l;
  l.eloc = eloc_scratch_layout(n, g, block);
  l.cub = up(eloc_scratch_bytes(n, g));  // above the hit lists of either scan route
  l.alt_col = up(l.cub + cub_reserve(n));
  l.alt_val = up(l.alt_col + 8 * nnz);
  l.total = l.alt_val + 8 * nnz;
  return l;
}

long long hamiltonian_scratch_bytes(long long n, long long nnz, const ExcGeom &g) { return ham_layout(n, nnz, g, false).total; }

template <bool EMIT>
static int launch_rows(bool half, const u64 *bra, long long nb, const double *h1e, const double *h2e, const u64 *key, long long N,
                       const GroupView &gv, char *sc, const ElocScratch &lay, const double *hii, long long *offsets, long long *col,
                       double *val, const ExcGeom &g, cudaStream_t st) {
  const HitRun *runs = reinterpret_cast<const HitRun *>(sc + lay.runs);
  const u32 *run_cnt = reinterpret_cast<const u32 *>(sc + lay.run_cnt);
  const u32 *hits = reinterpret_cast<const u32 *>(sc + lay.hits);
  const u32 *self_pos = reinterpret_cast<const u32 *>(sc + lay.self_pos);
  const unsigned grid = (unsigned)((nb + kHamThreads / 32 - 1) / (kHamThreads / 32));
#define PYNQS_HAM_ROWS(LL, HH)                                                                                                    \
  hamiltonian_row_kernel<LL, HH, EMIT><<<grid, kHamThreads, 0, st>>>(bra, nb, h1e, h2e, key, N, gv, runs, run_cnt, lay.run_stride, hits, \
                                                                    self_pos, hii, offsets, col, val, g)
  if (half) PYNQS_HAM_ROWS(1, true);
  else if (g.L == 1) PYNQS_HAM_ROWS(1, false);
  else if (g.L == 2) PYNQS_HAM_ROWS(2, false);
  else PYNQS_HAM_ROWS(3, false);
#undef PYNQS_HAM_ROWS
  count_launch();
  return check_launch(EMIT ? "hamiltonian_row_kernel (emit)" : "hamiltonian_row_kernel (count)");
}

// every row sorted by column: cub::DeviceSegmentedSort with 31-bit offsets, so in calls that each take the rows starting in one
// window of `span` entries (the window's rows end below 2^31 entries past its start)
static int sort_rows(long long n, long long nnz, const long long *offsets, long long *col, double *val, char *sc, const HamScratch &hl,
                     const ExcGeom &g, cudaStream_t st) {
  long long span = (1LL << 31) - 1 - ((long long)g.nsd + 1);
  const long long knob = eloc_tuning().sort_chunk;
  if (knob > 0 && knob < span) span = knob;
  long long *alt_col = reinterpret_cast<long long *>(sc + hl.alt_col);
  double *alt_val = reinterpret_cast<double *>(sc + hl.alt_val);
  bool in_alt = false;
  for (long long lo = 0; lo < nnz; lo += span) {
    const long long items = nnz - lo < (1LL << 31) - 1 ? nnz - lo : (1LL << 31) - 1;
    auto begin = thrust::make_transform_iterator(thrust::counting_iterator<int>(0), RowBound{offsets, lo, lo + span, 0});
    auto end = thrust::make_transform_iterator(thrust::counting_iterator<int>(0), RowBound{offsets, lo, lo + span, 1});
    cub::DoubleBuffer<long long> k(col + lo, alt_col + lo);
    cub::DoubleBuffer<double> v(val + lo, alt_val + lo);
    size_t tmp = 0;
    cudaError_t e = cub::DeviceSegmentedSort::SortPairs(nullptr, tmp, k, v, (int)items, (int)n, begin, end, st);
    if (e == cudaSuccess && (long long)tmp > cub_reserve(n)) {
      set_error("hamiltonian sort: %zu bytes of temporary storage needed, %lld reserved", tmp, cub_reserve(n));
      return 4;
    }
    if (e == cudaSuccess) e = cub::DeviceSegmentedSort::SortPairs(sc + hl.cub, tmp, k, v, (int)items, (int)n, begin, end, st);
    if (e != cudaSuccess) {
      set_error("hamiltonian sort: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
      return 3;
    }
    count_launch(3);
    in_alt = k.selector != 0;  // the same for every call: it depends on the key width only
  }
  if (in_alt) {
    if (cudaMemcpyAsync(col, alt_col, 8 * (size_t)nnz, cudaMemcpyDeviceToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(val, alt_val, 8 * (size_t)nnz, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
      return check_launch("hamiltonian sort: copy of the sorted rows");
  }
  return 0;
}

// emit == 0: offsets [n + 1]; emit == 1: col / val [nnz] from the offsets of the count call
int launch_hamiltonian(const u64 *bra, long long n, const double *h1e, const double *h2e, const u64 *key, long long N, const void *group_ws,
                       void *scratch, long long scratch_bytes, long long *offsets, long long nnz, long long *col, double *val,
                       const ExcGeom &g, int emit, cudaStream_t st) {
  if (n >= (1LL << 31) - 1 || nnz < 0) {
    set_error("hamiltonian: bad n = %lld or nnz = %lld (n < 2^31 - 1)", n, nnz);
    return 1;
  }
  if (n == 0 || N == 0) {  // no rows, or rows without entries
    if (!emit && cudaMemsetAsync(offsets, 0, 8 * (size_t)(n + 1), st) != cudaSuccess) return check_launch("hamiltonian offsets memset");
    return 0;
  }
  const bool half = eloc_half_route(N, g);
  const HamScratch hl = ham_layout(n, emit ? nnz : 0, g, half && block_route_wanted(n, g));
  if (scratch_bytes < hl.total) {
    set_error("hamiltonian scratch too small: %lld < %lld bytes", scratch_bytes, hl.total);
    return 4;
  }
  char *sc = static_cast<char *>(scratch);
  const ElocScratch &lay = hl.eloc;
  double *hii = reinterpret_cast<double *>(sc + lay.hii);
  // emit: the diagonal <x|H|x> on a side stream next to the first scan, joined before the first row kernel
  SideLane *join = nullptr;
  if (emit) {
    SideLane *side = side_lane(1);
    const bool forked = side_fork(side, st);
    if (int rc = launch_diag_f64(bra, h1e, h2e, hii, n, 1, g.L, g.sorb, g.nele, forked ? side->stream : st)) return rc;
    join = forked ? side : nullptr;
  }
  const GroupView gv = group_view(group_ws, N, g.L);
  for (long long b0 = 0; b0 < n; b0 += lay.batch) {
    const long long nb = n - b0 < lay.batch ? n - b0 : lay.batch;
    const u64 *xb = bra + b0 * g.L;
    if (int rc = launch_scan_batch(xb, nb, gv, sc, lay, g, half, st)) return rc;
    if (join != nullptr) {
      if (!side_join(join, st)) return check_launch("hamiltonian: join of the diagonal kernel");
      join = nullptr;
    }
    const int rc = emit ? launch_rows<true>(half, xb, nb, h1e, h2e, key, N, gv, sc, lay, hii + b0, offsets + b0, col, val, g, st)
                        : launch_rows<false>(half, xb, nb, h1e, h2e, key, N, gv, sc, lay, nullptr, offsets + b0, nullptr, nullptr, g, st);
    if (rc) return rc;
  }
  if (emit) return sort_rows(n, nnz, offsets, col, val, sc, hl, g, st);
  // counts -> exclusive prefix, offsets[n] = nnz
  if (cudaMemsetAsync(offsets + n, 0, 8, st) != cudaSuccess) return check_launch("hamiltonian offsets memset");
  size_t tmp = 0;
  cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, tmp, offsets, offsets, (int)(n + 1), st);
  if (e == cudaSuccess && (long long)tmp > cub_reserve(n)) {
    set_error("hamiltonian scan: %zu bytes of temporary storage needed, %lld reserved", tmp, cub_reserve(n));
    return 4;
  }
  if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(sc + hl.cub, tmp, offsets, offsets, (int)(n + 1), st);
  if (e != cudaSuccess) {
    set_error("hamiltonian scan: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
    return 3;
  }
  count_launch(2);
  return 0;
}

}  // namespace pynqs
