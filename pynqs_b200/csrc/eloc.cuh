// eloc.cuh -- what the kernels of the one-pass local energy share (eloc_scan.cu, eloc_block.cu, and hamiltonian.cu, which
// reads the same hit lists): the hit lists the scan kernels hand to the evaluation kernel, the device counters of one call,
// the scan phase's launcher and the test / experiment knobs (set through pynqs_set_tuning, never read from the environment).
#pragma once
#include "gindex.cuh"
#include "rederive.cuh"

namespace pynqs {

// A sample's hits are stored as up to `run_stride` runs in the global hit buffer; run_cnt[s] says how many.
struct HitRun {
  u32 off, cnt;  // cnt & kOverflow: a queue or the buffer overflowed -> the sample takes the full route
};
constexpr u32 kOverflow = 0x80000000u;
constexpr u32 kNoSelf = 0xffffffffu;

// hit word: position in the grouped copy | kHitA (alpha-grouped copy) | kHitOwn (found in the scan of one of
// the sample's own strings, folded route only -- the eval kernel checks the class of the key accordingly)
constexpr u32 kHitA = 0x80000000u, kHitOwn = 0x40000000u, kHitPos = 0x3fffffffu;

// device counters of one call (zeroed by the launcher)
struct ElocCounters {
  u32 hit_cursor;    // next free slot of the hit buffer
  u32 tile_count;    // block route: tiles made by the grouping pass
  u32 tile_next;     // ... and handed out so far
  u32 slot_front;    // block route: samples placed in tiles
  u32 n_single;      // samples left to the per-sample kernel (stored at the back of the slot array)
  u32 single_next;
  u32 n_heavy;       // evaluation: samples with long hit lists, handed from the tile kernel to the warp-per-sample kernel
  u32 heavy_next;    // ... and taken so far
  u32 pad[56];
};
static_assert(sizeof(ElocCounters) == 256, "counters are 256 bytes");

// knobs for tests and experiments (defaults are the production values)
struct ElocTuning {
  int scan_threads = 0;        // 0: by the number of groups; else 64 / 128 / 256
  int search_factor = 64;      // a bucket this many times larger than what it could hold is searched, not walked
  int full_keys = 0;           // 1: one-word ONVs take the full-key route of multi-word ONVs
  int block_min_samples = 4096;  // calls with fewer samples go to the per-sample kernel only
  int block_min_group = 8;     // samples sharing a beta string needed for a tile of the block kernel
  int block_enable = 1;
  int eval_tiles = 1;          // 1: large calls evaluate 32 samples per warp; 2: every call does; 0: one warp per sample
  int block_parts = 0;         // block kernel: parts a tile's alpha-beta groups are split into (0: by the number of tiles; 1, 2, 4)
  int lut_pipeline = 1;        // lut_indexed_kernel: next query and its directory slot fetched ahead (0: one query at a time)
  int sort_chunk = 0;          // hamiltonian.cu: entries per segmented-sort call (0: as many as 31-bit offsets allow)
};
ElocTuning &eloc_tuning();

// scratch of one call (eloc_scan.cu): the diagonal elements of all samples, then the hit lists of one batch
struct ElocScratch {
  long long hii, self_pos, run_cnt, heavy, runs, counters, block_ws, hits, total;
  long long hit_cap, batch;
  int splits;      // same for every batch of the call (sized for the first, largest one)
  int warps;       // warps per scan CTA
  int run_stride;  // HitRun records per sample
  bool block;      // samples grouped by beta string first (eloc_block.cu); the per-sample kernel takes the rest
};
bool eloc_half_route(long long N, const ExcGeom &g);  // one-word ONVs scanned through their folded 32-bit strings
bool block_route_wanted(long long n, const ExcGeom &g);
ElocScratch eloc_scratch_layout(long long n, const ExcGeom &g, bool block);
long long eloc_scratch_bytes(long long n, const ExcGeom &g);
// the scan phase of one batch bra[0, nb) (grouping pass + block kernel, per-sample scan kernel): its hit lists in the scratch
int launch_scan_batch(const u64 *bra, long long nb, const GroupView &gv, char *scratch, const ElocScratch &lay, const ExcGeom &g, bool half,
                      cudaStream_t st);
int launch_diag_f64(const u64 *bra, const double *h1e, const double *h2e, double *out, long long n, long long stride, int L, int sorb,
                    int nele, cudaStream_t st);

// One hit of sample x decoded (the evaluation kernels of eloc_scan.cu, hamiltonian.cu): the key y it points to, y's row of the
// sorted table, and the class of the pair -- 1 single, 2 double, 0 nothing (on the folded route a key that passed the 32-bit
// test but is not connected to x; row is then not loaded).  It has no warp-wide operation, and every lane returns from it:
// the callers' ballots that follow need the whole warp.
template <int L, bool HALF>
__device__ __forceinline__ int decode_hit(const GroupView &gv, const Onv<L> &x, u32 h, Onv<L> &y, u32 &row) {
  const bool grouping = (h & kHitA) != 0u;
  const u32 pos = HALF ? (h & kHitPos) : (h & ~kHitA);
  y = load_onv<L>((grouping ? gv.keys[1] : gv.keys[0]) + (size_t)pos * L);
  if (HALF) {  // the scan tested one folded string only: class of the full key vs the scan it came from
    const u64 d = y.w[0] ^ x.w[0];
    const int na = __popcll(d & kEven), nb = __popcll(d & kOdd);
    const int moved = grouping ? nb : na, fixed = grouping ? na : nb;  // own-string scans: one string is x's
    const bool ok = (h & kHitOwn) ? ((fixed == 0) & ((moved == 2) | (moved == 4))) : ((na == 2) & (nb == 2));
    if (!ok) return 0;
  }
  row = __ldg((grouping ? gv.rows[1] : gv.rows[0]) + pos);
  return excitation_class<L>(x, y);
}

// <x|H|y> of lane src's single excitation x -> y, evaluated by the whole warp (every lane passes the same x; every lane gets
// the element).  The warp's orbital lists of x are built at the first single of the sample; have_lists remembers that.
// The caller (hamiltonian_row_kernel) walks its singles (rare) with a ballot and uses the element inside that loop.
template <int L>
__device__ __forceinline__ double single_element_of_lane(const Onv<L> &x, const Onv<L> &y, int src, const double *__restrict__ h1e,
                                                         const double *__restrict__ h2e, const ExcGeom &g, OrbLists &lists, bool &have_lists) {
  if (!have_lists) {
    build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x & 31);
    __syncwarp();
    have_lists = true;
  }
  Onv<L> ys;
#pragma unroll
  for (int w = 0; w < L; ++w) ys.w[w] = __shfl_sync(0xffffffffu, y.w[w], src);
  return single_element_warp<L, double>(x, ys, h1e, h2e, g.sorb, lists.occ_order, lists.n_occ);
}

// inclusive prefix sum of v over the lanes of the warp
__device__ __forceinline__ u32 warp_inclusive_sum(u32 v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 up = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += up;
  }
  return v;
}

// lanes hold consecutive segments of a list, incl = warp_inclusive_sum of their lengths: the lane whose segment holds entry e
// (the first one whose inclusive prefix exceeds e; 31 when e is past the end)
__device__ __forceinline__ int warp_segment_of(u32 incl, u32 e) {
  int r = 0;
#pragma unroll
  for (int step = 16; step > 0; step >>= 1) {
    const u32 v = __shfl_sync(0xffffffffu, incl, r + step - 1);
    if (v <= e) r += step;
  }
  return r;
}

// alpha / beta strings of a one-word ONV from their 32-bit folds (inverse of fold_alpha / fold_beta)
__device__ __forceinline__ u64 unfold_alpha_word(u32 f) { return (u64)(f & 0x55555555u) | ((u64)(f & 0xAAAAAAAAu) << 31); }
__device__ __forceinline__ u64 unfold_beta_word(u32 f) { return ((u64)(f & 0x55555555u) << 1) | ((u64)(f & 0xAAAAAAAAu) << 32); }

}  // namespace pynqs
