// eloc_block.cu -- the scan of the one-pass local energy for samples that SHARE a beta string.
//
// The per-sample kernel (eloc_scan.cu) walks, for every sample, the ~noB*nvB + 2 groups of table keys that can hold a
// connected determinant.  All but one of those groups depend on the sample's BETA string only, and in a VMC sample
// set many samples carry the same beta string (10^6 Fe2S2 samples: at most C(20,15) = 15 504 beta strings, so >= 64
// samples per string).  Here the samples are first grouped by beta string (three small kernels, no sort: the order
// of the samples inside a group is irrelevant), and one warp then takes a TILE of up to 32 samples with the same
// beta string -- one sample per lane -- and walks the shared groups once for all of them:
//
//   * the groups are walked in chunks of 32 keys; the bit planes of a chunk (the 32 keys' folded alpha strings
//     bit-transposed, GroupView::planes) are copied into shared memory with cp.async (coalesced, all copies of a fill in
//     flight at once);
//   * a lane reads the planes of its K = min(noA, nvA) orbitals and counts, for the 32 keys at once, how many of them
//     are on the wrong side (~3 instructions per orbital): the result is the exact mask of its hits in the chunk;
//   * bucket bounds, hashing, duplicate-bucket detection and the copy are paid once per tile, not per sample.
//
// Groups with fewer than `block_min_group` samples stay with the per-sample kernel (a lane-per-sample walk with one lane
// is slower than a lane-per-key walk).
//
// The sample's own-alpha group (beta singles, beta-beta doubles) depends on the sample, not on the tile: it is walked
// per sample with one key per lane, as in the per-sample kernel.
//
// Output: the same hit lists (HitRun records + hit words) the per-sample kernel writes; eloc_eval_kernel reads both.
// One-word ONVs only (folded 32-bit strings); tables with duplicate keys are handed to the evaluation kernel's
// reference route like everywhere else.
#include "eloc.cuh"

namespace pynqs {

constexpr int kBlkWarps = 4;       // warps per CTA; every warp works on its own tile
constexpr int kStageChunks = 32;   // chunks of 32 keys whose bit planes are staged per warp and fill (4 KB)
constexpr int kMaxGroups = 260;    // beta singles of a one-word ONV (<= 16 * 16) + the own group
constexpr int kMaxOrbs = 16;       // orbitals a lane tests: min(noA, nvA) <= 32 / 2
constexpr int kFirstBlock = 64;    // hit-buffer block sizes of a sample: 64, 128, ... (one HitRun each)

struct BlockWarpSmem {
  u32 stage[kStageChunks * 32];  // [chunk][folded orbital]: bit planes of the staged chunks
  uint2 chunk[kStageChunks];     // of every staged chunk: its number (position / 32) and the mask of its keys in the group
  uint2 rng[kMaxGroups];         // bucket [first, end) of every group; group sB = the tile's own beta string
  u32 goff[kMaxGroups];          // first chunk of every group among the chunks of its walk
  unsigned char bpos[32];
};
constexpr int kDupSet = 512;  // open-addressing set of the bucket starts of a walk (lives in the idle stage, next to minq)
static_assert(2 * kDupSet <= kStageChunks * 32 && kDupSet >= 2 * 256, "duplicate-bucket set: twice the largest number of groups");

__host__ __device__ inline u32 sample_log2_buckets(long long n) {
  u32 lg = 10;
  while ((1LL << lg) < 4 * n && lg < 24) ++lg;
  return lg;
}

// ---- grouping pass ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sample_count_kernel(const u64 *__restrict__ bra, long long n, u32 shift, u32 *__restrict__ bcnt) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Onv<1> x;
  x.w[0] = bra[i];
  atomicAdd(bcnt + (string_hash32<1>(x, kOdd) >> shift), 1u);
}

// one thread per bucket: a range of the slot array for its samples and, when there are enough of them, tiles of
// 17..32 samples (balanced); small buckets go to the back of the slot array, for the per-sample kernel
__global__ void __launch_bounds__(256)
sample_alloc_kernel(u32 *__restrict__ bcnt, u32 *__restrict__ bbase, u32 nbuckets, ElocCounters *ctr, uint2 *__restrict__ tiles, u32 min_group,
                    u32 n) {
  const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nbuckets) return;
  const u32 c = bcnt[b];
  if (c == 0) return;
  bcnt[b] = 0;  // becomes the fill counter of the scatter pass
  if (c < min_group) {
    bbase[b] = n - c - atomicAdd(&ctr->n_single, c);
    return;
  }
  const u32 base = atomicAdd(&ctr->slot_front, c);
  bbase[b] = base;
  const u32 nt = (c + 31u) >> 5, lo = c / nt, extra = c - lo * nt;  // `extra` tiles of lo + 1 samples, the rest lo
  u32 t = atomicAdd(&ctr->tile_count, nt), at = base;
  for (u32 k = 0; k < nt; ++k) {
    const u32 sz = lo + (k < extra ? 1u : 0u);
    tiles[t + k] = make_uint2(at, sz);
    at += sz;
  }
}

__global__ void __launch_bounds__(256)
sample_scatter_kernel(const u64 *__restrict__ bra, long long n, u32 shift, u32 *__restrict__ bfill, const u32 *__restrict__ bbase,
                      u32 *__restrict__ slots) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Onv<1> x;
  x.w[0] = bra[i];
  const u32 b = string_hash32<1>(x, kOdd) >> shift;
  slots[bbase[b] + atomicAdd(bfill + b, 1u)] = (u32)i;
}

// ---- the block kernel -------------------------------------------------------------------------------------------------
struct BlockGeom {
  int sorb, noA, noB, nvB;
  int norb;  // orbitals a lane tests: min(noA, nvA)
  int occ;   // 1: the lane's occupied orbitals (a key's missing bits are counted), 0: its virtual ones (a key's extra bits)
};

struct LaneHits {  // where a lane's sample keeps its hits in the global buffer
  u32 base, fill, cap, nrun;
  u32 end;  // run records [.., end) of the sample belong to this part of the tile
  bool over;
};

// what the rarely taken paths of a tile need (kept in local memory; the inner loop never touches it)
struct TileCtx {
  const u64 *keysB;
  u32 *self_pos, *hits;
  HitRun *my_runs;
  ElocCounters *ctr;
  u64 x;
  u32 sid, hit_cap;
  int run_stride;
};

// a lane's current block is full (or there is none yet): close it and take the next, twice as large.  The bookkeeping
// travels by value so that it stays in registers on the caller's side (every emitted hit reads it).
__device__ __noinline__ LaneHits next_hit_block(const TileCtx &c, LaneHits h) {
  if (h.cap) {
    c.my_runs[h.nrun] = HitRun{h.base, h.fill};
    ++h.nrun;
  }
  const u32 ncap = h.cap ? 2u * h.cap : (u32)kFirstBlock;
  if (h.nrun == h.end) {
    h.over = true;
    return h;
  }
  const u32 off = atomicAdd(&c.ctr->hit_cursor, ncap);
  if (off > c.hit_cap || ncap > c.hit_cap - off) {
    h.over = true;
    return h;
  }
  h.base = off;
  h.cap = ncap;
  h.fill = 0;
  return h;
}

__device__ __forceinline__ void emit_hit(const TileCtx &c, LaneHits &h, u32 v) {
  if (h.over) return;
  if (h.fill == h.cap) {
    h = next_hit_block(c, h);
    if (h.over) return;
  }
  c.hits[h.base + h.fill++] = v;
}

__device__ __forceinline__ void cp_async16(u32 *smem_dst, const u32 *gsrc) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// The key test.  All alpha strings of the sector have noA bits, so |a ^ k| = 2 |k & ~a| = 2 |a & ~k|: key k is an alpha
// single of the lane's string a iff exactly one of k's bits lies on a's virtual orbitals (equivalently: exactly one of a's
// occupied orbitals is missing from k), an alpha double iff two do, and k == a iff none does.  A lane counts that number
// on the smaller side, K = min(noA, nvA) orbitals, for 32 keys at once: the bit planes of a chunk (planes[o] = bit o of
// its 32 folded alpha strings) of its K orbitals through a saturating bit-sliced counter.
// KT: K at compile time (OCC: the occupied side); KT < 0: any K up to kMaxOrbs, side chosen at run time.
template <int KT, bool OCC>
struct LaneOrbs {
  u32 pos[KT >= 0 ? (KT > 0 ? KT : 1) : kMaxOrbs];  // the lane's K orbitals (folded positions)
  int k;                                             // KT < 0: K
  u32 flip;                                          // KT < 0: ~0 on the occupied side
};

template <int KT, bool OCC>
__device__ __forceinline__ LaneOrbs<KT, OCC> lane_orbs(u32 fa, u32 all_alpha, const BlockGeom &g) {
  LaneOrbs<KT, OCC> o;
  o.k = g.norb;
  o.flip = g.occ ? 0xffffffffu : 0u;
  u32 s = (KT < 0 ? g.occ != 0 : OCC) ? fa : all_alpha & ~fa;
  constexpr int kn = KT >= 0 ? KT : kMaxOrbs;
#pragma unroll
  for (int k = 0; k < kn; ++k) {
    o.pos[k] = (u32)(__ffs(s) - 1) & 31u;  // (an idle lane's string has no bits: any position will do)
    s &= s - 1u;
  }
  return o;
}

// ones / twos / threes: the keys of the staged chunk with at least 1 / 2 / 3 counted orbitals
template <int KT, bool OCC>
__device__ __forceinline__ void count_orbs(const u32 *st, const LaneOrbs<KT, OCC> &o, u32 &ones, u32 &twos, u32 &threes) {
  ones = twos = threes = 0u;
  constexpr int kn = KT >= 0 ? KT : kMaxOrbs;
#pragma unroll
  for (int k = 0; k < kn; ++k) {
    if (KT < 0 && k >= o.k) break;
    u32 x = st[o.pos[k]];
    if (KT < 0) x ^= o.flip;
    else if (OCC) x = ~x;
    threes |= twos & x;
    twos |= ones & x;
    ones |= x;
  }
}

// Walk the groups [q_lo, q_hi) of the current beta string: S.goff[q_lo .. q_hi] holds the exclusive prefix of their
// sizes in chunks of 32 keys (chunk c = positions 32c .. 32c + 31 of the beta-grouped copy; a group's first and last
// chunk are shared with its neighbours and masked).  Fill after fill: chunk descriptors (lanes over groups), copy of
// their bit planes (8 lanes per chunk, cp.async), test.  Every lane emits its hits in ascending position within a group,
// the groups in the order of q.  live: ~0 for a lane whose sample has the walk's beta string, else 0.
template <bool OWN, int KT, bool OCC>
__device__ __forceinline__ void walk_groups(const TileCtx &c, LaneHits &h, BlockWarpSmem &S, const u32 *__restrict__ planes, int q_lo,
                                            int q_hi, const LaneOrbs<KT, OCC> &o, u32 live) {
  const int lane = threadIdx.x & 31;
  const u32 total = S.goff[q_hi];
  for (u32 f0 = 0; f0 < total; f0 += (u32)kStageChunks) {
    const u32 n = total - f0 < (u32)kStageChunks ? total - f0 : (u32)kStageChunks;
    for (int q = q_lo + lane; q < q_hi; q += 32) {
      const u32 g0 = S.goff[q], g1 = S.goff[q + 1];
      const u32 lo = g0 > f0 ? g0 : f0, hi = g1 < f0 + n ? g1 : f0 + n;
      if (lo < hi) {
        const uint2 r = S.rng[q];
        const u32 c0 = r.x >> 5, c1 = (r.y - 1u) >> 5;
        for (u32 j = lo; j < hi; ++j) {
          const u32 cj = c0 + (j - g0);
          u32 m = 0xffffffffu;
          if (cj == c0) m &= 0xffffffffu << (r.x & 31u);
          if (cj == c1) m &= 0xffffffffu >> (31u - ((r.y - 1u) & 31u));
          S.chunk[j - f0] = make_uint2(cj, m);
        }
      }
    }
    __syncwarp();
    // 8 lanes per chunk, 4 chunks per pass, all passes of the fill in flight (the descriptors are read first: without
    // that every pass would wait for its own load)
    const u32 sub = (u32)lane & 7u;
    {
      u32 cj[kStageChunks / 4];
#pragma unroll
      for (int u = 0; u < kStageChunks / 4; ++u) {
        const u32 j = ((u32)lane >> 3) + 4u * (u32)u;
        cj[u] = j < n ? S.chunk[j].x : 0u;
      }
#pragma unroll
      for (int u = 0; u < kStageChunks / 4; ++u) {
        const u32 j = ((u32)lane >> 3) + 4u * (u32)u;
        if (j < n) cp_async16(&S.stage[32u * j + 4u * sub], planes + 32u * (size_t)cj[u] + 4u * sub);
      }
    }
    cp_async_wait_all();
    __syncwarp();
    for (u32 j = 0; j < n; ++j) {
      const uint2 d = S.chunk[j];
      u32 ones, twos, threes;
      count_orbs<KT, OCC>(S.stage + 32u * j, o, ones, twos, threes);
      const u32 keys = d.y & live, base = d.x << 5;
      u32 m = (OWN ? ones & ~threes : ones & ~twos) & keys;  // own group: singles and doubles; else: singles
      if (OWN) {
        u32 self = ~ones & keys;  // the sample itself (checked on the full key)
        while (self) {
          const u32 p = base + (u32)(__ffs(self) - 1);
          self &= self - 1u;
          if (c.keysB[p] == c.x) c.self_pos[c.sid] = p;
        }
      }
      while (__any_sync(0xffffffffu, m != 0u)) {
        if (m) {
          const u32 p = base + (u32)(__ffs(m) - 1);
          m &= m - 1u;
          emit_hit(c, h, p | (OWN ? kHitOwn : 0u));
        }
      }
    }
    __syncwarp();
  }
}

// chunks of 32 keys that the bucket [r.x, r.y) touches
__device__ __forceinline__ u32 group_chunks(uint2 r) { return r.x == r.y ? 0u : ((r.y - 1u) >> 5) - (r.x >> 5) + 1u; }

// SPLIT: the alpha-beta groups of a tile are split over several warps (see `parts` below); a template parameter so that
// the whole-tile kernel of large calls carries none of the bookkeeping.
template <bool SPLIT, int KT, bool OCC>
__global__ void __launch_bounds__(kBlkWarps * 32)
eloc_block_kernel(const u64 *__restrict__ bra, const u32 *__restrict__ slots, const uint2 *__restrict__ tiles, ElocCounters *ctr, GroupView gv,
                  HitRun *__restrict__ runs, u32 *__restrict__ run_cnt, int run_stride, u32 *__restrict__ hits, u32 *__restrict__ self_pos,
                  u32 hit_cap, BlockGeom g, u32 force_parts) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  BlockWarpSmem &S = reinterpret_cast<BlockWarpSmem *>(smem_raw)[warp];
  const u32 table_has_dup = __ldg(&gv.hdr->has_dup);
  const u32 ntiles = ctr->tile_count;  // final: written by the grouping pass, which finished before this kernel started
  const int sB = g.noB * g.nvB;
  // Few tiles (a rank's share of the samples at 8 GPUs; the launcher decides by the number of samples): with ~1.2 tiles per
  // resident warp the launch takes the time of two tiles.  The alpha-beta groups of a tile are then split into `parts` ranges that different warps walk (part 0 also takes
  // the tile's own group and the samples' own-alpha groups); every part writes its hits to run records of its own
  // (run_stride / parts each), so nothing is shared between the parts but the read-only table.  Every part repeats the
  // tile's set-up (~12 % of a tile), so two parts is where it stops paying: measured for 125 000 samples 0.700 / 0.656 /
  // 0.738 ms with 1 / 2 / 4 parts (profiles/micro/eloc_slice.py).
  u32 parts = 1;
  if (SPLIT) {
    parts = force_parts ? force_parts : 2u;
    if ((u32)run_stride < 2u * parts) parts = 1;
  }
  const u32 runs_per_part = (u32)run_stride / parts;
  const u32 nitems = ntiles * parts;
  const u32 *__restrict__ planes = gv.planes;
  const u32 *__restrict__ halfA = gv.half[1];
  const u64 all_orbs = g.sorb >= 64 ? ~0ull : ((1ull << g.sorb) - 1ull);
  const u32 all_alpha = fold_alpha(all_orbs);
  const u32 all_beta = fold_beta(all_orbs);
  for (;;) {
    u32 t = 0;
    if (lane == 0) t = atomicAdd(&ctr->tile_next, 1u);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= nitems) break;
    const u32 part = t / ntiles;  // part-major: the (heavier) parts 0 are handed out first
    t -= part * ntiles;
    const uint2 tile = tiles[t];
    const bool active = (u32)lane < tile.y;
    const u32 sid = active ? slots[tile.x + lane] : 0u;
    const u64 x = active ? bra[sid] : 0ull;
    const u32 fa = fold_alpha(x), fb = fold_beta(x);
    const LaneOrbs<KT, OCC> orbs = lane_orbs<KT, OCC>(fa, all_alpha, g);
    TileCtx c;
    c.keysB = gv.keys[0];
    c.self_pos = self_pos;
    c.hits = hits;
    c.my_runs = runs + (size_t)sid * run_stride;
    c.ctr = ctr;
    c.x = x;
    c.sid = sid;
    c.hit_cap = hit_cap;
    c.run_stride = run_stride;
    LaneHits h = {0u, 0u, 0u, part * runs_per_part, (part + 1u) * runs_per_part, table_has_dup != 0u};
    const int q_part_lo = (int)((u32)sB * part / parts), q_part_hi = (int)((u32)sB * (part + 1u) / parts);
    u32 remaining = table_has_dup ? 0u : __ballot_sync(0xffffffffu, active);
    // a tile holds the samples of one bucket of the grouping pass: normally one beta string, after a hash collision several
    while (remaining) {
      const int leader = __ffs(remaining) - 1;
      const u32 fbL = __shfl_sync(0xffffffffu, fb, leader);
      const bool mine = active && fb == fbL;
      remaining &= ~__ballot_sync(0xffffffffu, mine);
      const u32 live = mine ? 0xffffffffu : 0u;
      // ---- the groups of this beta string: positions of its occupied / virtual orbitals, then one bucket per single ------
      __syncwarp();
      {
        const u32 bit = 1u << lane, below = bit - 1u;
        if (fbL & bit) S.bpos[__popc(fbL & below)] = (unsigned char)lane;
        else if (all_beta & bit) S.bpos[g.noB + __popc(all_beta & ~fbL & below)] = (unsigned char)lane;
      }
      __syncwarp();
      for (int q = lane; q <= sB; q += 32) {
        u32 f = fbL;
        if (q < sB) {
          const int pb = q / g.noB, hb = q - pb * g.noB;
          f ^= (1u << S.bpos[hb]) ^ (1u << S.bpos[g.noB + pb]);
        }
        Onv<1> y;
        y.w[0] = unfold_beta_word(f);
        const u32 *stp = gv.start[0] + group_bucket<1>(y, 0, gv.shift);
        S.rng[q] = make_uint2(__ldg(stp), __ldg(stp + 1));
      }
      __syncwarp();
      // the own group first (other acceptance test): the keys that carry the tile's beta string itself
      if (lane == 0) {
        S.goff[sB] = 0u;
        S.goff[sB + 1] = group_chunks(S.rng[sB]);
      }
      __syncwarp();
      if (part == 0u) walk_groups<true>(c, h, S, planes, sB, sB + 1, orbs, live);
      // two singles whose strings share a bucket: the folded test cannot tell them apart, so the bucket is walked for one
      // of them only -- the one with the SMALLEST group number, so that every part of a split tile drops the same ones.
      // Buckets are told apart by their first position; the set and the smallest group number of every bucket live in the
      // (now idle) stage buffer, a group's slot of the set in goff (recomputed below)
      u32 *dupset = S.stage;
      u32 *minq = S.stage + kDupSet;
      for (int i = lane; i < kDupSet; i += 32) {
        dupset[i] = 0xffffffffu;
        minq[i] = 0xffffffffu;
      }
      __syncwarp();
      for (int q = lane; q < sB; q += 32) {
        const uint2 r = S.rng[q];
        if (r.x == r.y) continue;
        u32 slot = (r.x * 0x9E3779B1u) >> (32 - 9);
        for (;;) {
          const u32 old = atomicCAS(&dupset[slot], 0xffffffffu, r.x);
          if (old == 0xffffffffu || old == r.x) break;
          slot = (slot + 1u) & (u32)(kDupSet - 1);
        }
        atomicMin(&minq[slot], (u32)q);
        S.goff[q] = slot;
      }
      __syncwarp();
      for (int q = lane; q < sB; q += 32) {
        const uint2 r = S.rng[q];
        if (r.x != r.y && minq[S.goff[q]] != (u32)q) S.rng[q] = make_uint2(0u, 0u);
      }
      __syncwarp();
      // first chunk of every group: exclusive prefix over the groups' sizes in chunks
      {
        u32 running = 0;
        for (int q0 = 0; q0 < sB; q0 += 32) {
          const int q = q0 + lane;
          u32 nb = 0;
          if (q >= q_part_lo && q < q_part_hi) nb = group_chunks(S.rng[q]);  // (the other parts' groups count as empty)
          const u32 incl = warp_inclusive_sum(nb);
          if (q < sB) S.goff[q] = running + incl - nb;
          running += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) S.goff[sB] = running;
      }
      __syncwarp();
      walk_groups<false>(c, h, S, planes, 0, sB, orbs, live);
    }
    // ---- every sample's own-alpha group (beta singles, beta-beta doubles): the group depends on the sample, so every lane
    // walks ITS bucket of the alpha-grouped copy, four independent loads in flight (a lane reads consecutive words: its lines
    // stay in L1; the 32 lanes touch 32 lines per load, which at ~3 loads per sample and key-chunk is nowhere near a limit).
    // No shuffles, no serial dependence between samples.
    if (!table_has_dup && part == 0u) {
      uint2 rA = make_uint2(0u, 0u);
      if (active) {
        Onv<1> y;
        y.w[0] = x;
        const u32 *stp = gv.start[1] + group_bucket<1>(y, 1, gv.shift);
        rA = make_uint2(__ldg(stp), __ldg(stp + 1));
      }
      const u32 longest = __reduce_max_sync(0xffffffffu, rA.y - rA.x);
      const u32 far = ~fb;  // at distance 32 from the lane's beta string
      for (u32 i = 0; i < longest; i += 4) {
        u32 k[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const u32 p = rA.x + i + (u32)u;
          k[u] = p < rA.y ? __ldg(halfA + p) : far;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const u32 d = (u32)__popc(k[u] ^ fb);
          if (d == 2u || d == 4u) emit_hit(c, h, (rA.x + i + (u32)u) | kHitA | kHitOwn);
        }
      }
    }
    if (active) {
      const u32 first = part * runs_per_part;
      if (h.over) {
        c.my_runs[first] = HitRun{0u, kOverflow};
        h.nrun = first + 1u;
      } else if (h.fill) {
        c.my_runs[h.nrun] = HitRun{h.base, h.fill};
        ++h.nrun;
      }
      if (parts == 1u) {
        run_cnt[sid] = h.nrun;
      } else {
        // every part leaves its unused records empty and reports all of them (the same value from every part)
        for (u32 r = h.nrun; r < h.end; ++r) c.my_runs[r] = HitRun{0u, 0u};
        run_cnt[sid] = (u32)run_stride;
      }
    }
    __syncwarp();
  }
}

// ---- host side --------------------------------------------------------------------------------------------------------
using BlockKernel = decltype(&eloc_block_kernel<false, -1, false>);

// K at compile time for the benchmarked Fe2S2 sector (5 virtual alpha orbitals) and the geometries the tests cover
template <bool SPLIT>
static BlockKernel block_kernel(const BlockGeom &bg) {
  if (bg.norb == 5) return bg.occ ? eloc_block_kernel<SPLIT, 5, true> : eloc_block_kernel<SPLIT, 5, false>;
  if (bg.norb == 6 && !bg.occ) return eloc_block_kernel<SPLIT, 6, false>;
  if (bg.norb == 8 && bg.occ) return eloc_block_kernel<SPLIT, 8, true>;
  return eloc_block_kernel<SPLIT, -1, false>;
}

struct BlockLayout {
  u32 log2_buckets;
  long long bcnt, bbase, slots, tiles, total;
};

BlockLayout block_layout(long long n) {
  BlockLayout l;
  l.log2_buckets = sample_log2_buckets(n);
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  long long o = 0;
  l.bcnt = o;
  o = up(o + 4LL * (1LL << l.log2_buckets));
  l.bbase = o;
  o = up(o + 4LL * (1LL << l.log2_buckets));
  l.slots = o;
  o = up(o + 4 * n);
  l.tiles = o;
  o = up(o + 8 * (n / 4 + 64));
  l.total = o;
  return l;
}

long long block_scratch_bytes(long long n) { return block_layout(n).total; }
int block_run_stride() { return 8; }

// grouping pass + block kernel over all n samples; the samples it leaves to the per-sample kernel are the last
// ctr->n_single entries of the slot array (returned through *slots_out)
int launch_eloc_block(const u64 *bra, long long n, const GroupView &gv, char *block_ws, ElocCounters *ctr, HitRun *runs, u32 *run_cnt,
                      int run_stride, u32 *hits, u32 *self_pos, u32 hit_cap, const ExcGeom &g, const u32 **slots_out, cudaStream_t st) {
  const BlockLayout l = block_layout(n);
  u32 *bcnt = reinterpret_cast<u32 *>(block_ws + l.bcnt), *bbase = reinterpret_cast<u32 *>(block_ws + l.bbase);
  u32 *slots = reinterpret_cast<u32 *>(block_ws + l.slots);
  uint2 *tiles = reinterpret_cast<uint2 *>(block_ws + l.tiles);
  *slots_out = slots;
  const u32 nbuckets = 1u << l.log2_buckets, shift = 32u - l.log2_buckets;
  if (cudaMemsetAsync(bcnt, 0, 4 * (size_t)nbuckets, st) != cudaSuccess) return check_launch("eloc block memset");
  const unsigned sb = (unsigned)((n + 255) / 256);
  sample_count_kernel<<<sb, 256, 0, st>>>(bra, n, shift, bcnt);
  int min_group = eloc_tuning().block_min_group;
  if (min_group < 4) min_group = 4;  // tiles[] holds n / 4 + 64 entries
  sample_alloc_kernel<<<(nbuckets + 255) / 256, 256, 0, st>>>(bcnt, bbase, nbuckets, ctr, tiles, (u32)min_group, (u32)n);
  sample_scatter_kernel<<<sb, 256, 0, st>>>(bra, n, shift, bcnt, bbase, slots);
  count_launch(3);
  if (int rc = check_launch("eloc grouping pass")) return rc;
  BlockGeom bg;
  bg.sorb = g.sorb;
  bg.noA = g.noA;
  bg.noB = g.noB;
  bg.nvB = g.nvB;
  bg.occ = g.noA < g.nvA;
  bg.norb = bg.occ ? g.noA : g.nvA;
  const size_t smem = sizeof(BlockWarpSmem) * kBlkWarps;
  long long ctas = (n + 32 * kBlkWarps - 1) / (32 * kBlkWarps);
  const long long cap = 148LL * (long long)((227 * 1024) / (sizeof(BlockWarpSmem) * kBlkWarps + 1024));
  if (ctas > cap) ctas = cap;
  // fewer than ~2 tiles (of ~26 samples) per resident warp: split the tiles (the knob block_parts forces 1, 2 or 4 parts)
  const int forced = eloc_tuning().block_parts;
  const bool split = forced ? forced > 1 : n < 2 * 26 * ctas * kBlkWarps;
  const BlockKernel kern = split ? block_kernel<true>(bg) : block_kernel<false>(bg);
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("eloc_block_kernel smem opt-in");
  kern<<<(unsigned)ctas, kBlkWarps * 32, smem, st>>>(bra, slots, tiles, ctr, gv, runs, run_cnt, run_stride, hits, self_pos, hit_cap, bg,
                                                     (u32)(forced == 3 ? 2 : forced));
  count_launch();
  return check_launch("eloc_block_kernel");
}

}  // namespace pynqs
