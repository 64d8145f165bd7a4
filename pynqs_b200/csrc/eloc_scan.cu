// eloc_scan.cu -- sample-space local energy without materialising comb / Hmat.
//
// Replaces what the reference does in three native calls plus ~6 torch passes over [n, M]
// (vmc/energy/eloc.py:326-397: get_comb_hij_fused -> WavefunctionLUT.lookup -> scatter ->
// divide -> multiply -> sum).  Nothing of size [n, M] ever reaches HBM, and the connected
// determinants are never formed: the kernels walk the string-grouped copies of the table
// (gindex.cuh) and pick out, with XOR + popcount, the keys that ARE connected to the sample.
//
//   eloc_scan_kernel   one CTA per (sample, slice of its groups).  Groups of a sample x:
//         g < sB : the bucket of the beta string of x's g-th beta single; a key there is an
//                  alpha-beta double of x iff its beta part equals that string and its alpha part
//                  is at distance 2 from x's;
//         g = sB : the bucket of x's own beta string: alpha singles (distance 2), alpha-alpha
//                  doubles (4) and x itself (0);
//         g = sB+1: the bucket of x's own alpha string: beta singles and beta-beta doubles.
//       Small groups are cut into 32-key chunks and the chunks of a sample form one flat list that
//       the warps consume evenly (lanes take consecutive keys: coalesced loads, ~16 instructions per
//       32 keys, no hashing and no searching); one-word ONVs are tested on 32-bit folded strings.
//       Larger groups are walked by one warp each; buckets much larger than the number of
//       determinants they could contain are searched instead (binary search inside the bucket, the
//       reference's own algorithm on a short range).  Hits go to per-warp queues (ballot + popcount
//       compaction) and from there to a global hit buffer in a deterministic order.
//   eloc_eval_kernel   one warp per sample: for every hit, <x|H|x'> re-derived from the two bit
//       strings (rederive.cuh: same arithmetic, same order of additions as the fused operator)
//       times psi(x') / psi(x), summed over a fixed lane assignment and a shuffle tree.
//
// Exactness: a key is a hit iff it is one of the reference's connected determinants and is in the
// table -- the same set binary_search_BigInteger would find.  Tables with duplicate keys, and
// samples whose hits overflow the queues, take the reference's route instead (enumerate every
// excitation, classic binary search); no floating point atomics anywhere.
#include "eloc.cuh"
#include "lut.cuh"
#include "rederive.cuh"
#include "tables.cuh"

namespace pynqs {

constexpr int kMaxScanWarps = 8;   // scan kernel: 2, 4 or 8 warps per CTA, by the number of groups of a sample
constexpr int kQueue = 512;        // hits per warp before the sample falls back to the full route
constexpr int kEvalThreads = 128;  // eval kernel: 4 samples per CTA

struct Cplx {
  double re, im;
};

// numpy / c10 complex division (torch/headeronly/util/complex.h operator/=)
__device__ __forceinline__ Cplx cdiv(Cplx x, Cplx y) {
  const double a = x.re, b = x.im, c = y.re, d = y.im;
  const double ac = fabs(c), ad = fabs(d);
  Cplx r;
  if (ac >= ad) {
    if (ac == 0.0 && ad == 0.0) {
      r.re = a / ac;
      r.im = b / ad;
    } else {
      const double rat = d / c, scl = 1.0 / (c + d * rat);
      r.re = (a + b * rat) * scl;
      r.im = (b - a * rat) * scl;
    }
  } else {
    const double rat = c / d, scl = 1.0 / (d + c * rat);
    r.re = (a * rat + b) * scl;
    r.im = (b * rat - a) * scl;
  }
  return r;
}

template <bool CPLX>
__device__ __forceinline__ Cplx load_psi(const double *__restrict__ psi, long long id) {
  Cplx v;
  if (CPLX) {
    const double2 t = __ldg(reinterpret_cast<const double2 *>(psi) + id);
    v.re = t.x;
    v.im = t.y;
  } else {
    v.re = __ldg(psi + id);
    v.im = 0.0;
  }
  return v;
}

// ratio psi'/psi0 times a real H, accumulated
template <bool CPLX>
__device__ __forceinline__ void accumulate(Cplx &acc, Cplx pm, Cplx p0, double h) {
  if (CPLX) {
    const Cplx q = cdiv(pm, p0);
    acc.re += q.re * h;
    acc.im += q.im * h;
  } else {
    acc.re += (pm.re / p0.re) * h;
  }
}

// the entry's two orbitals as an excitation mask (L = 1) or packed o0 | o1 << 8 (L > 1)
template <int L>
__device__ __forceinline__ u64 msk_make(u32 o0, u32 o1) {
  return L == 1 ? ((1ull << o0) | (1ull << o1)) : (u64)(o0 | (o1 << 8));
}
template <int L>
__device__ __forceinline__ Onv<L> msk_apply(const Onv<L> &x, u64 m) {
  Onv<L> y = x;
  if (L == 1) {
    y.w[0] ^= m;
  } else {
    flip_bit<L>(y, (int)(m & 0xffu));
    flip_bit<L>(y, (int)((m >> 8) & 0xffu));
  }
  return y;
}

ElocTuning &eloc_tuning() {
  static ElocTuning t;
  return t;
}

// hit = position in the grouped copy | grouping << 31
__device__ __forceinline__ void push_hits(u32 *queue, u32 &qn, bool hit, u32 value) {
  const u32 m = __ballot_sync(0xffffffffu, hit);
  if (m == 0) return;
  if (hit) {
    const u32 at = qn + (u32)__popc(m & ((1u << (threadIdx.x & 31)) - 1u));
    if (at < (u32)kQueue) queue[at] = value;
  }
  qn += (u32)__popc(m);
}

// distance test of one key against the pattern y: `same` = the bits that must agree (the string that
// defines the group).  Returns the popcount of the difference, or 255 when the strings differ.
template <int L>
__device__ __forceinline__ u32 key_distance(const Onv<L> &k, const Onv<L> &y, u64 same) {
  u32 pc = 0;
  u64 bad = 0;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = k.w[i] ^ y.w[i];
    bad |= d & same;
    pc += (u32)__popcll(d);
  }
  return bad ? 255u : pc;
}

// walk the keys [s, e) of one bucket, this warp's share of it (warp `part` of `parts`): two keys per lane in flight
template <int L>
__device__ __forceinline__ void scan_bucket(const u64 *__restrict__ keys, u32 s, u32 e, const Onv<L> &y, u64 same, u32 allow, u32 gbit,
                                            u32 *queue, u32 &qn, u32 *self_pos, u32 part, u32 parts) {
  const u32 lane = threadIdx.x & 31;
  for (u32 k0 = s + 64u * part; k0 < e; k0 += 64u * parts) {
    const u32 p0 = k0 + lane, p1 = p0 + 32;
    u32 d0 = 255u, d1 = 255u;
    Onv<L> a, b;
    if (p0 < e) a = load_onv<L>(keys + (size_t)p0 * L);
    if (p1 < e) b = load_onv<L>(keys + (size_t)p1 * L);
    if (p0 < e) d0 = key_distance<L>(a, y, same);
    if (p1 < e) d1 = key_distance<L>(b, y, same);
    if (self_pos != nullptr) {  // the sample itself (own beta bucket only)
      if (d0 == 0u) *self_pos = p0;
      if (d1 == 0u) *self_pos = p1;
    }
    push_hits(queue, qn, d0 < 8u && ((allow >> d0) & 1u), p0 | gbit);
    push_hits(queue, qn, d1 < 8u && ((allow >> d1) & 1u), p1 | gbit);
  }
}

// large bucket: search each determinant the group could contain (targets enumerated by the lanes)
//   kind 0: alpha-beta doubles on top of a beta single, base = x with that single applied (targets: sA alpha singles)
//   kind 1: own beta string  (targets: x itself, sA alpha singles, noAA * nvAA alpha-alpha doubles)
//   kind 2: own alpha string (targets: sB beta singles, noBB * nvBB beta-beta doubles)
// walk the folded strings [s, e) of one bucket (HALF route), this warp's share of it (warp `part` of `parts`):
// distance of each to `pat`, allowed distances in `allow`; four loads per lane in flight
__device__ __forceinline__ u32 scan_half(const u32 *__restrict__ half, u32 s, u32 e, u32 pat, u32 allow, u32 flags, u32 *queue, u32 qn,
                                         u32 part, u32 parts) {
  const u32 lane = threadIdx.x & 31;
  for (u32 k0 = s + 128u * part; k0 < e; k0 += 128u * parts) {
    u32 d[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const u32 p = k0 + 32u * u + lane;
      d[u] = 31u;
      if (p < e) d[u] = (u32)__popc(__ldg(half + p) ^ pat);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) push_hits(queue, qn, ((allow >> d[u]) & 1u) != 0u, (k0 + 32u * u + lane) | flags);
  }
  return qn;
}

struct SearchGeom {  // per kind: number of single targets, hole pairs, particle pairs and their table offsets
  int nS, nH, nP, oS, oH, oP, self, pad;
};

template <int L>
__device__ __noinline__ u32 search_bucket(const u64 *__restrict__ keys, u32 s, u32 e, const Onv<L> base, const u64 *msk,
                                          const SearchGeom *sg, u32 gbit, u32 *queue, u32 qn, u32 *self_pos, int part, int parts) {
  const int lane = threadIdx.x & 31;
  const int nS = sg->nS, nH = sg->nH, nD = nH * sg->nP, oS = sg->oS, oH = sg->oH, oP = sg->oP;
  const int total = nS + nD + sg->self;
  for (int t0 = 32 * part; t0 < total; t0 += 32 * parts) {  // this warp's share of the targets
    const int t = t0 + lane;
    u32 pos = 0xffffffffu;
    bool self = false;
    if (t < total) {
      Onv<L> y = base;
      if (t < nS) {
        y = msk_apply<L>(y, msk[oS + t]);
      } else if (t < nS + nD) {
        const int u = t - nS, pp = u / nH, hp = u - pp * nH;
        y = msk_apply<L>(msk_apply<L>(y, msk[oH + hp]), msk[oP + pp]);
      } else {
        self = true;
      }
      pos = bucket_search<L>(keys, s, e, y);
    }
    if (self && pos != 0xffffffffu) {
      *self_pos = pos;
      pos = 0xffffffffu;
    }
    push_hits(queue, qn, pos != 0xffffffffu, pos | gbit);
  }
  return qn;
}

// dynamic shared memory of the scan kernel:
//   lists | patterns [nG][L] | tables (search route) | buckets [nG] | duplicate filter | long groups | chunk list | queues
constexpr int kListChunks = 4;     // groups of up to kListChunks * 32 keys go to the flat chunk list
constexpr int kChunkUnroll = 4;    // independent key loads in flight per lane (full keys)
constexpr int kHalfUnroll = 8;     // ... (folded 32-bit strings)
constexpr int kDupList = 32;       // suspects checked exactly (more: every group is checked)
constexpr int kDupLog2 = 9, kDupWords = 1 << kDupLog2;  // set of the bucket ids of a sample's groups (<= 256 of them)

struct ScanSmem {
  u32 ypat, msk, rng, dup, lgrp, clist, queues, total;
  u32 list_chunks;  // groups of up to list_chunks * 32 keys go to the flat chunk list (0: none -- everything by the warp)
  u32 search_factor;  // a bucket this many times larger than the number of determinants it could hold is searched
};
constexpr u32 kScanSmemMax = 200 * 1024;
__host__ __device__ inline ScanSmem scan_smem(const ExcGeom &g, int warps) {
  const size_t sB = (size_t)g.noB * g.nvB, nG = sB + 2;
  ScanSmem m;
  // the chunk list is the one part that can be cut down when a large system would not fit: fewer chunks per
  // group qualify, the rest of the groups is walked one warp per group
  for (int lc = kListChunks;; lc = lc / 2) {
    size_t o = (sizeof(OrbLists) + 15) & ~(size_t)15;
    m.ypat = (u32)o;
    o += 8 * nG * g.L;
    m.msk = (u32)o;
    o += 8 * (size_t)table_offsets(g).total;
    m.rng = (u32)o;
    o += 8 * nG;
    m.dup = (u32)o;
    o += 4 * kDupWords;
    m.lgrp = (u32)o;
    o = (o + 2 * (sB + 2) + 15) & ~(size_t)15;
    m.clist = (u32)o;
    o += 16 * (sB * lc + 8);
    m.queues = (u32)o;
    m.total = (u32)(o + sizeof(u32) * kQueue * warps);
    m.list_chunks = (u32)lc;
    if (m.total <= kScanSmemMax || lc == 0) break;
  }
  m.search_factor = 64u;
  return m;
}

// orbital (bit of the ONV word) of position f of a folded beta string (inverse of fold_beta)
__device__ __forceinline__ u32 unfold_beta(u32 f) { return (f & 1u) ? 32u + f : f + 1u; }

// Small groups are cut into 32-key chunks and all chunks of a sample are processed as one flat, evenly
// divided list (a warp would otherwise idle on its small groups while another one walks a large group);
// larger groups are walked (or searched) by one warp each.
// HALF (L = 1, N < 2^30): the test reads the folded 32-bit strings; a key that passes may sit in the bucket
// by hash collision, which the eval kernel detects on the full key.
template <int L, bool HALF, int THREADS>
__global__ void __launch_bounds__(THREADS)
eloc_scan_kernel(const u64 *__restrict__ bra, long long n, GroupView gv, HitRun *__restrict__ runs, u32 *__restrict__ run_cnt,
                 int run_stride, u32 *__restrict__ hits, u32 *__restrict__ self_pos, ElocCounters *ctr, u32 hit_cap, int splits,
                 const u32 *__restrict__ ids, ExcGeom g, ScanSmem sm) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int sB = g.noB * g.nvB, nG = sB + 2;
  OrbLists &lists = *reinterpret_cast<OrbLists *>(smem_raw);
  u64 *ypat = reinterpret_cast<u64 *>(smem_raw + sm.ypat);  // [nG][L] pattern of every group
  u64 *msk = reinterpret_cast<u64 *>(smem_raw + sm.msk);    // excitation tables (search route only)
  uint2 *rng = reinterpret_cast<uint2 *>(smem_raw + sm.rng);  // [nG] bucket of every group
  u32 *dupf = reinterpret_cast<u32 *>(smem_raw + sm.dup);
  unsigned short *lgrp = reinterpret_cast<unsigned short *>(smem_raw + sm.lgrp);  // groups walked by one warp each
  uint4 *clist4 = reinterpret_cast<uint4 *>(smem_raw + sm.clist);  // {first key, bucket end, pattern | group}
  uint2 *clist2 = reinterpret_cast<uint2 *>(smem_raw + sm.clist);  // HALF: {first key, bucket end}
  u32 *queues = reinterpret_cast<u32 *>(smem_raw + sm.queues);
  __shared__ int s_nchunks, s_nlong;
  __shared__ u32 s_flags, s_ndup;
  __shared__ unsigned char s_bpos[32];
  __shared__ unsigned short s_dupq[kDupList];
  __shared__ u32 s_kill[8];
  constexpr int kScanThreads = THREADS, kScanWarps = THREADS / 32;
  __shared__ u32 wtot[80];  // work per (round of THREADS groups, warp); nG <= 2306 -> at most 37 x 2 entries
  __shared__ SearchGeom s_sg[3];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // duplicate keys in the table: the eval kernel takes the reference's route for every sample.  The flag is
  // loaded here and looked at only when the run record is written, so no CTA starts by waiting for it.
  const u32 table_has_dup = __ldg(&gv.hdr->has_dup);
  // work items: (sample, slice of its groups) pairs -- every sample of the call, or (ids != nullptr) the samples
  // the grouping pass of the block route left to this kernel: the last n_single entries of ids[0, n)
  const long long items = ids != nullptr ? (long long)ctr->n_single : n * splits;
  for (long long item = blockIdx.x; item < items; item += gridDim.x) {
  const long long it_s = splits == 1 ? item : item / splits;
  const int split = splits == 1 ? 0 : (int)(item - it_s * splits);
  const long long s = ids != nullptr ? (long long)ids[n - 1 - it_s] : it_s;
  HitRun *my_run = runs + s * run_stride + split * kScanWarps + warp;
  if (threadIdx.x == 0 && split == 0) run_cnt[s] = (u32)(splits * kScanWarps);
  const Onv<L> x = load_onv<L>(bra + s * L);
  // HALF: the beta singles are picked straight out of the folded beta string (n-th set bit); the orbital lists
  // are only built when a group has to be searched
  if (!HALF && threadIdx.x < 64) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x, 64);
  if (HALF) {
    for (int t = threadIdx.x; t < kDupWords; t += kScanThreads) dupf[t] = 0u;
    if (threadIdx.x < 32) {  // positions of the folded beta string: occupied ones first, then the virtual ones
      const u32 occ = fold_beta(x.w[0]);
      const u32 all = fold_beta(g.sorb >= 64 ? ~0ull : ((1ull << g.sorb) - 1ull));
      const u32 bit = 1u << threadIdx.x, below = bit - 1u;
      if (occ & bit) s_bpos[__popc(occ & below)] = (unsigned char)threadIdx.x;
      else if (all & bit) s_bpos[g.noB + __popc(all & ~occ & below)] = (unsigned char)threadIdx.x;
    }
  }
  if (threadIdx.x == 0) s_flags = s_ndup = 0u;
  __syncthreads();

  // ---- the groups of this slice: pattern and bucket of each ---------------------------------------------------
  const int per = (nG + splits - 1) / splits;
  const int g_begin = split * per, g_end = min(nG, g_begin + per), ab_end = min(g_end, sB);
  // a group this large is searched, not walked.  Walking is ~16 instructions per 32 keys with independent
  // loads; a search is ~13 dependent loads per determinant the group could hold: the break-even is at a few
  // thousand keys for the 75 alpha singles of an Fe2S2 alpha-beta group, hence the default factor of 64
  const u32 big_ab = sm.search_factor * (u32)g.sA;
  const u32 big_own_b = sm.search_factor * (u32)(g.sA + g.noAA * g.nvAA + 1), big_own_a = sm.search_factor * (u32)(sB + g.noBB * g.nvBB);
  // (HALF: the buckets of ALL groups, so that every slice agrees on which group walks a shared bucket)
  const int q_lo = HALF ? 0 : g_begin, q_hi = HALF ? nG : g_end;
  constexpr int UN = HALF ? kHalfUnroll : kChunkUnroll;
  // what a group adds to the two work lists: chunks (low half) and one-warp-per-group entries (high half)
  auto work_of = [&](int q, uint2 r) -> u32 {
    if (q < g_begin || q >= g_end || r.y == r.x) return 0u;
    if (q >= sB) return 1u << 16;
    const u32 nc = (r.y - r.x + 31u) >> 5;
    return nc > sm.list_chunks ? (1u << 16) : nc;
  };
  // one round of groups (and not an empty slice): every thread keeps the work scan of its only group
  const bool one_round = q_hi > q_lo && q_hi - q_lo <= kScanThreads;
  u32 my_work = 0, my_incl = 0;
  uint2 my_r = make_uint2(0u, 0u);
  for (int q0 = q_lo; q0 < q_hi; q0 += kScanThreads) {
    const int q = q0 + (int)threadIdx.x;
    uint2 r = make_uint2(0u, 0u);
    if (q < q_hi) {
      Onv<L> y = x;
      if (q < sB) {  // beta single q: hole number q % noB, particle number q / noB
        const u32 pb = fdiv((u32)q, g.by_noB), hb = (u32)q - pb * g.noB;
        if (HALF) {
          // any fixed numbering of the occupied / virtual beta orbitals will do here (every group is treated
          // alike): the order of the set bits of the folded string
          y.w[0] ^= (1ull << unfold_beta(s_bpos[hb])) ^ (1ull << unfold_beta(s_bpos[g.noB + pb]));
        } else {
          flip_bit<L>(y, lists.b[hb] & 0xff);
          flip_bit<L>(y, lists.b[g.noB + pb] & 0xff);
        }
      }
      const int grouping = q == sB + 1 ? 1 : 0;
      const u32 bkt = group_bucket<L>(y, grouping, gv.shift);
      const u32 *st = (grouping ? gv.start[1] : gv.start[0]) + bkt;  // no dynamic index into the param struct
      r = make_uint2(__ldg(st), __ldg(st + 1));
      rng[q] = r;
#pragma unroll
      for (int w = 0; w < L; ++w) ypat[q * L + w] = y.w[w];
      const u32 size = r.y - r.x;
      if (size > (q < sB ? big_ab : (q == sB ? big_own_b : big_own_a))) atomicOr(&s_flags, 1u);  // searched: needs the tables
      if (HALF && q < sB && size && size <= big_ab) {
        // the folded test cannot tell two beta strings in one bucket apart: a bucket must be WALKED for only one
        // of the groups that map to it (searches are exact per group and stay).  Suspects (a later arrival at a
        // bucket that is already in the set) are listed and resolved below.
        // (a small open-addressing set of the bucket ids seen so far: exact, so the check below only runs for
        //  samples that really have two groups in one bucket -- a fraction of a per cent)
        u32 slot = (bkt * 0x9E3779B1u) >> (32 - kDupLog2);
        for (;;) {
          const u32 old = atomicCAS(&dupf[slot], 0u, bkt + 1u);
          if (old == 0u) break;  // first group of this bucket
          if (old == bkt + 1u) {
            const u32 at = atomicAdd(&s_ndup, 1u);
            if (at < (u32)kDupList) s_dupq[at] = (unsigned short)q;
            atomicOr(&s_flags, 2u);
            break;
          }
          slot = (slot + 1u) & (u32)(kDupWords - 1);
        }
      }
    }
    my_work = work_of(q, r);
    my_incl = warp_inclusive_sum(my_work);
    my_r = r;
    const u32 tot = __shfl_sync(0xffffffffu, my_incl, 31);
    if (lane == 0) wtot[(q0 - q_lo) / kScanThreads * kScanWarps + warp] = tot;
  }
  __syncthreads();
  const u32 flags = s_flags;
  if (flags & 2u) {  // rare: filter collision or two groups in one bucket -- keep the lowest group only
    // decisions first (reads of the unchanged buckets, marks in a bit set), then the clearing: no thread reads a
    // bucket that another one is clearing
    if (threadIdx.x < 8) s_kill[threadIdx.x] = 0u;  // one-word ONVs: at most 256 alpha-beta groups
    __syncthreads();
    const u32 nd = s_ndup;
    if (nd <= (u32)kDupList) {
      // one of the groups of a shared bucket arrived first and is not listed, so a suspect marks the HIGHER of
      // every equal pair it finds; the lowest group of a bucket is never marked and everyone else is
      for (u32 i = threadIdx.x; i < nd; i += kScanThreads) {
        const int q = s_dupq[i];
        const uint2 rq = rng[q];
        for (int p = 0; p < sB; ++p) {
          const uint2 rp = rng[p];  // non-empty buckets are equal iff their ranges are
          if (p != q && rp.x == rq.x && rp.y == rq.y) {
            const int m = max(p, q);
            atomicOr(&s_kill[m >> 5], 1u << (m & 31));
          }
        }
      }
    } else {  // list overflow: every group looks for a lower group with the same bucket
      for (int q = threadIdx.x; q < sB; q += kScanThreads) {
        const uint2 rq = rng[q];
        if (rq.x == rq.y || rq.y - rq.x > big_ab) continue;
        for (int p = 0; p < q; ++p) {
          const uint2 rp = rng[p];
          if (rp.x == rq.x && rp.y == rq.y) {
            atomicOr(&s_kill[q >> 5], 1u << (q & 31));
            break;
          }
        }
      }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < sB; q += kScanThreads)
      if ((s_kill[q >> 5] >> (q & 31)) & 1u) rng[q] = make_uint2(0u, 0u);
    __syncthreads();
    for (int q0 = q_lo; q0 < q_hi; q0 += kScanThreads) {  // the work counts again
      const int q = q0 + (int)threadIdx.x;
      const u32 tot = __shfl_sync(0xffffffffu, warp_inclusive_sum(work_of(q, q < q_hi ? rng[q] : make_uint2(0u, 0u))), 31);
      if (lane == 0) wtot[(q0 - q_lo) / kScanThreads * kScanWarps + warp] = tot;
    }
    __syncthreads();
  }
  if (flags & 1u) {
    if (HALF) {  // the search route works on the excitation tables, which need the orbital lists
      if (threadIdx.x < 64) build_lists<L>(x, g.sorb, g.noA, g.noB, lists, threadIdx.x, 64);
      __syncthreads();
    }
    const TableOffsets to = table_offsets(g);
    for_each_table_entry(g, lists, to, [&](int t, int, u32 e0, u32 e1) { msk[t] = msk_make<L>(e0 & 0xffu, e1 & 0xffu); });
    if (threadIdx.x == 0) {
      s_sg[0] = SearchGeom{g.sA, 0, 0, to.sa, 0, 0, 0, 0};
      s_sg[1] = SearchGeom{g.sA, g.noAA, g.nvAA, to.sa, to.hpa, to.ppa, 1, 0};
      s_sg[2] = SearchGeom{sB, g.noBB, g.nvBB, to.sb, to.hpb, to.ppb, 0, 0};
    }
  }
  // every thread places the work of its groups: chunk list in group order, then the long list
  auto place = [&](int q, uint2 r, u32 mine, u32 at) {
    if (mine >> 16) {
      lgrp[at >> 16] = (unsigned short)q;
    } else if (mine) {
      uint4 ent = make_uint4(r.x, r.y, (u32)q, 0u);
      if (L == 1 && !HALF) {
        ent.z = (u32)ypat[q];
        ent.w = (u32)(ypat[q] >> 32);
      }
      for (u32 j = 0; j < mine; ++j) {
        if (HALF) clist2[(at & 0xffffu) + j] = make_uint2(ent.x, ent.y);
        else clist4[(at & 0xffffu) + j] = ent;
        ent.x += 32u;
      }
    }
  };
  u32 all_work = 0;
  if (one_round && !(flags & 2u)) {  // the common case: the scan of the bucket phase is still valid
    u32 before = 0;
#pragma unroll
    for (int w = 0; w < kScanWarps; ++w) {
      const u32 t = wtot[w];
      before += w < warp ? t : 0u;
      all_work += t;
    }
    place(q_lo + (int)threadIdx.x, my_r, my_work, before + my_incl - my_work);
  } else {
    u32 before = 0;  // work of all the (round, warp) pairs before mine
    int slot = 0;
    for (int q0 = q_lo; q0 < q_hi; q0 += kScanThreads) {
      for (int w = 0; w < warp; ++w) before += wtot[slot + w];
      const int q = q0 + (int)threadIdx.x;
      const uint2 r = q < q_hi ? rng[q] : make_uint2(0u, 0u);
      const u32 mine = work_of(q, r);
      place(q, r, mine, before + warp_inclusive_sum(mine) - mine);
      for (int w = warp; w < kScanWarps; ++w) before += wtot[slot + w];
      slot += kScanWarps;
    }
    all_work = before;
  }
  {
    // pad the chunk list to a whole number of unrolled iterations with empty chunks
    const u32 nch = all_work & 0xffffu, padded = (nch + (u32)UN - 1u) / (u32)UN * (u32)UN;
    if (threadIdx.x < padded - nch) {
      if (HALF) clist2[nch + threadIdx.x] = make_uint2(0u, 0u);
      else clist4[nch + threadIdx.x] = make_uint4(0u, 0u, (u32)g_begin, 0u);
    }
    if (threadIdx.x == 0) {
      s_nchunks = (int)padded;
      s_nlong = (int)(all_work >> 16);
    }
  }
  __syncthreads();

  u32 *queue = queues + warp * kQueue;
  u32 qn = 0;
  // ---- (1) the flat chunk list: UN independent chunks per warp and iteration ---------------------------------------
  const int nchunks = s_nchunks;
  if (HALF) {
    const u32 *__restrict__ halfB = gv.half[0];
    const u32 ax = fold_alpha(x.w[0]);
    for (int c0 = warp * UN; c0 < nchunks; c0 += kScanWarps * UN) {
      u32 h[UN], pos[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const uint2 ent = clist2[c0 + u];
        pos[u] = ent.x + (u32)lane;
        h[u] = ~ax;  // past the bucket end: distance 32
        if (pos[u] < ent.y) h[u] = __ldg(halfB + pos[u]);
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) push_hits(queue, qn, __popc(h[u] ^ ax) == 2, pos[u]);
    }
  } else {
    const u64 *__restrict__ keysB = gv.keys[0];
    for (int c0 = warp * UN; c0 < nchunks; c0 += kScanWarps * UN) {
      Onv<L> k[UN], y[UN];
      u32 pos[UN];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const uint4 ent = clist4[c0 + u];
        pos[u] = ent.x + (u32)lane;
        if (L == 1) {
          y[u].w[0] = (u64)ent.z | ((u64)ent.w << 32);
        } else {
#pragma unroll
          for (int w = 0; w < L; ++w) y[u].w[w] = ypat[ent.z * L + w];
        }
#pragma unroll
        for (int w = 0; w < L; ++w) k[u].w[w] = ~y[u].w[w];  // past the bucket end: a key at distance 64 L
        if (pos[u] < ent.y) k[u] = load_onv<L>(keysB + (size_t)pos[u] * L);
      }
#pragma unroll
      for (int u = 0; u < UN; ++u) push_hits(queue, qn, key_distance<L>(k[u], y[u], kOdd) == 2u, pos[u]);
    }
  }
  // ---- (2) the own groups and the long alpha-beta groups ---------------------------------------------------------
  // Small ones (the two own groups of a sparse table, typically) go to one warp each; large ones are shared by
  // all warps: a sample may have a few groups of thousands of keys next to dozens of small ones, and one warp
  // per group would leave the others idle.
  const int nlong = s_nlong;
  for (int i = 0; i < nlong; ++i) {
    const int q = lgrp[i];
    const uint2 r = rng[q];
    const u32 size = r.y - r.x;
    if (size == 0) continue;
    const bool shared = size > 256u;
    if (!shared && i % kScanWarps != warp) continue;
    const int part = shared ? warp : 0, parts = shared ? kScanWarps : 1;
    Onv<L> y;
#pragma unroll
    for (int w = 0; w < L; ++w) y.w[w] = ypat[q * L + w];
    if (q < sB) {  // alpha-beta doubles on top of beta single q
      if (size > big_ab) qn = search_bucket<L>(gv.keys[0], r.x, r.y, y, msk, &s_sg[0], 0u, queue, qn, nullptr, part, parts);
      else if (HALF) qn = scan_half(gv.half[0], r.x, r.y, fold_alpha(x.w[0]), 1u << 2, 0u, queue, qn, part, parts);
      else scan_bucket<L>(gv.keys[0], r.x, r.y, y, kOdd, 1u << 2, 0u, queue, qn, nullptr, part, parts);
    } else if (q == sB) {  // own beta string: x itself, alpha singles, alpha-alpha doubles
      if (size > big_own_b) {
        qn = search_bucket<L>(gv.keys[0], r.x, r.y, x, msk, &s_sg[1], HALF ? kHitOwn : 0u, queue, qn, self_pos + s, part, parts);
      } else if (HALF) {
        const u32 ax = fold_alpha(x.w[0]);
        for (u32 k0 = r.x + 32u * part; k0 < r.y; k0 += 32u * parts) {
          const u32 pos = k0 + (u32)lane;
          u32 d = 31u;
          if (pos < r.y) d = (u32)__popc(__ldg(gv.half[0] + pos) ^ ax);
          if (d == 0u && gv.keys[0][pos] == x.w[0]) self_pos[s] = pos;  // the sample itself (checked on the full key)
          push_hits(queue, qn, d == 2u || d == 4u, pos | kHitOwn);
        }
      } else {
        scan_bucket<L>(gv.keys[0], r.x, r.y, x, kOdd, (1u << 2) | (1u << 4), 0u, queue, qn, self_pos + s, part, parts);
      }
    } else {  // own alpha string: beta singles, beta-beta doubles
      if (size > big_own_a) {
        qn = search_bucket<L>(gv.keys[1], r.x, r.y, x, msk, &s_sg[2], kHitA | (HALF ? kHitOwn : 0u), queue, qn, nullptr, part, parts);
      } else if (HALF) {
        qn = scan_half(gv.half[1], r.x, r.y, fold_beta(x.w[0]), (1u << 2) | (1u << 4), kHitA | kHitOwn, queue, qn, part, parts);
      } else {
        scan_bucket<L>(gv.keys[1], r.x, r.y, x, kEven, (1u << 2) | (1u << 4), kHitA, queue, qn, nullptr, part, parts);
      }
    }
  }

  // publish this warp's hits (no CTA barrier: every warp owns its run record)
  __syncwarp();
  u32 off = 0;
  bool over = qn > (u32)kQueue || table_has_dup != 0u;
  if (lane == 0 && !over && qn) {
    off = atomicAdd(&ctr->hit_cursor, qn);
    if (off > hit_cap || qn > hit_cap - off) over = true;  // buffer exhausted
  }
  off = __shfl_sync(0xffffffffu, off, 0);
  over = __shfl_sync(0xffffffffu, (int)over, 0) != 0;
  if (lane == 0) {
    const HitRun run = {off, over ? kOverflow : qn};
    *my_run = run;
  }
  if (!over)
    for (u32 e = lane; e < qn; e += 32) hits[off + e] = queue[e];
  __syncthreads();  // the next item reuses the shared arrays
  }
}

// ---- evaluation ---------------------------------------------------------------------------------------------
// Single excitations are rare (under 2 % of the hits of the benchmarked Fe2S2 tables) but cost ~30 two-electron terms each.  The
// passes over the hit list put them on a per-warp queue (ballot + popcount) and go on; when the next pass's singles would not fit,
// and when the hit list ends, the queue is flushed: lane i evaluates entry i (single_element, one lane per single).
template <int L>
struct SingleQueue {
  u64 y[32][L];  // the key
  u32 row[32];   // its row of the sorted table
  u32 j[32];     // 32-samples-per-warp kernel: the sample of the tile it belongs to
};

// the lanes with a single (kind == 1) append it to the queue; flush(qn) empties a queue of qn entries first when they would
// not fit.  Every lane of the warp calls this.
template <int L, typename Flush>
__device__ __forceinline__ void push_singles(SingleQueue<L> &q, u32 &qn, int kind, const Onv<L> &y, u32 row, u32 j, Flush flush) {
  const u32 m = __ballot_sync(0xffffffffu, kind == 1);
  if (m == 0u) return;
  if (qn + (u32)__popc(m) > 32u) {
    flush(qn);
    qn = 0;
  }
  if (kind == 1) {
    const u32 at = qn + (u32)__popc(m & ((1u << (threadIdx.x & 31)) - 1u));
#pragma unroll
    for (int w = 0; w < L; ++w) q.y[at][w] = y.w[w];
    q.row[at] = row;
    q.j[at] = j;
  }
  qn += (u32)__popc(m);
  __syncwarp();
}

// (launch bounds per variant: the 40-register budget that lets 12 CTAs of the real one-word kernel share an SM makes the
//  complex and multi-word variants spill 250-390 bytes; they get 80 registers instead)
template <int L, bool CPLX, bool HALF>
__global__ void __launch_bounds__(kEvalThreads, (CPLX || L > 1) ? 6 : 12)
eloc_eval_kernel(const u64 *__restrict__ bra, long long n, const double *__restrict__ h1e, const double *__restrict__ h2e,
                 const u64 *__restrict__ key, const double *__restrict__ psi, long long N, GroupView gv,
                 const HitRun *__restrict__ runs, const u32 *__restrict__ run_cnt, int run_stride, const u32 *__restrict__ hits,
                 const u32 *__restrict__ self_pos, const double *__restrict__ hii, double *__restrict__ eloc,
                 double *__restrict__ psi0_out, const u32 *__restrict__ list, ElocCounters *ctr, ExcGeom g) {
  __shared__ OrbLists s_lists[kEvalThreads / 32];
  __shared__ SingleQueue<L> s_queue[kEvalThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // work items: every sample of the call (one per warp), or (list != nullptr) the samples the tile kernel put on the list of
  // long hit lists, handed out one by one (their lengths differ by orders of magnitude)
  const long long items = list != nullptr ? (long long)ctr->n_heavy : n;
  for (;;) {
  long long item;
  if (list != nullptr) {
    u32 t = 0;
    if (lane == 0) t = atomicAdd(&ctr->heavy_next, 1u);
    item = (long long)__shfl_sync(0xffffffffu, t, 0);
  } else {
    item = (long long)blockIdx.x * (kEvalThreads / 32) + warp;
  }
  if (item >= items) break;
  const long long s = list != nullptr ? (long long)list[item] : item;
  const Onv<L> x = load_onv<L>(bra + s * L);
  const int nruns = (int)run_cnt[s];
  const HitRun *my_runs = runs + s * run_stride;
  bool redo = false;
  for (int w = lane; w < nruns; w += 32) redo |= (my_runs[w].cnt & kOverflow) != 0;
  redo = __any_sync(0xffffffffu, redo);

  Cplx p0 = {0.0, 0.0}, acc = {0.0, 0.0};
  if (redo) {
    // the reference's route: every excitation in row order, classic binary search in the sorted table
    OrbLists &lists = s_lists[warp];
    build_lists<L>(x, g.sorb, g.noA, g.noB, lists, lane);
    __syncwarp();
    const long long id0 = classic_search<L>(key, N, x);
    if (id0 >= 0) p0 = load_psi<CPLX>(psi, id0);
    if (lane == 0) accumulate<CPLX>(acc, p0, p0, hii[s]);
    for (int r = lane; r < g.nsd; r += 32) {
      const Exc e = decode_exc(g, lists, r);
      const long long id = classic_search<L>(key, N, apply_exc<L>(x, e));
      if (id >= 0) accumulate<CPLX>(acc, load_psi<CPLX>(psi, id), p0, exc_element<L, double>(x, e, h1e, h2e, g.sorb));
    }
  } else {
    const u32 sp = self_pos[s];
    if (sp != kNoSelf) p0 = load_psi<CPLX>(psi, (long long)__ldg(gv.rows[0] + sp));
    if (lane == 0) accumulate<CPLX>(acc, p0, p0, hii[s]);  // row 0: (psi0/psi0) * H_xx
    SingleQueue<L> &q = s_queue[warp];
    u32 qn = 0;
    // lane i: entry i, into its own accumulator (two terms in flight: more spill at the real one-word kernel's 40 registers)
    auto flush = [&](u32 cnt) {
      if ((u32)lane < cnt) {
        Onv<L> yq;
#pragma unroll
        for (int w = 0; w < L; ++w) yq.w[w] = q.y[lane][w];
        accumulate<CPLX>(acc, load_psi<CPLX>(psi, q.row[lane]), p0, single_element<L, 2, double>(x, yq, h1e, h2e, g.sorb));
      }
      __syncwarp();
    };
    // the sample's runs back to back: lane r holds run r and an inclusive prefix of the counts, so the
    // whole list is walked 32 hits at a time whatever the runs' lengths (32 runs per round)
    for (int r0 = 0; r0 < nruns; r0 += 32) {
      HitRun mine = {0u, 0u};
      if (r0 + lane < nruns) mine = my_runs[r0 + lane];
      const u32 incl = warp_inclusive_sum(mine.cnt);
      const u32 total = __shfl_sync(0xffffffffu, incl, 31);
      for (u32 e0 = 0; e0 < total; e0 += 32) {
        const u32 e = e0 + (u32)lane;
        const int r = warp_segment_of(incl, e);  // the run that holds hit e
        const u32 r_incl = __shfl_sync(0xffffffffu, incl, r), r_cnt = __shfl_sync(0xffffffffu, mine.cnt, r);
        const u32 r_off = __shfl_sync(0xffffffffu, mine.off, r);
        // (no early exits: the ballot of the singles needs every lane)
        Onv<L> y = x;
        u32 row = 0;
        int kind = 0;  // 1 single, 2 double, 0 nothing to add
        if (e < total) kind = decode_hit<L, HALF>(gv, x, hits[r_off + (e - (r_incl - r_cnt))], y, row);
        if (kind == 2) accumulate<CPLX>(acc, load_psi<CPLX>(psi, row), p0, double_element<L, double>(x, y, h2e));
        push_singles<L>(q, qn, kind, y, row, 0u, flush);
      }
    }
    if (qn) flush(qn);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc.re += __shfl_xor_sync(0xffffffffu, acc.re, o);
    if (CPLX) acc.im += __shfl_xor_sync(0xffffffffu, acc.im, o);
  }
  if (lane == 0) {
    if (CPLX) {
      eloc[2 * s] = acc.re;
      eloc[2 * s + 1] = acc.im;
      psi0_out[2 * s] = p0.re;
      psi0_out[2 * s + 1] = p0.im;
    } else {
      eloc[s] = acc.re;
      psi0_out[s] = p0.re;
    }
  }
  __syncwarp();  // the next item reuses this warp's orbital lists and queue
  if (list == nullptr) break;
  }
}

// ---- evaluation, 32 samples per warp -------------------------------------------------------------------------------------
// The kernel above gives a sample a whole warp: with ~33 hits per sample its second pass over the hit list runs with one
// lane.  Here a warp takes a TILE of 32 consecutive samples (lane l keeps sample l's bookkeeping) and walks the hit lists of
// all of them back to back, 32 hits per pass whatever sample they belong to: ~1 000 hits = ~33 full passes instead of 64 half
// empty ones.  The products (psi'/psi0) * H of a pass are summed per sample with a segmented shuffle scan (the hits of a
// sample are adjacent) and the segment tails add into the sample's accumulator in shared memory -- a fixed order, no atomics.
// Runs: round r of the outer loop takes run r of every sample of the tile (one or two rounds after the block kernel).
// Samples with long hit lists (a skewed table: thousands of hits for the samples of a heavy string, which sit next to each
// other) would make one warp the tail of the launch: they are put on a list instead and the warp-per-sample kernel above
// takes them, one warp each.  Samples flagged for the reference's route (overflow, duplicate keys) go on that list too, and
// the kernel above takes the reference's route for them.
constexpr u32 kHeavyHits = 256;

struct EvalTileSmem {
  u64 x[32][kMaxL];
  double p0[32][2];
  double acc[32][2];
};

template <int L, bool CPLX, bool HALF>
__global__ void __launch_bounds__(kEvalThreads)
eloc_eval_tile_kernel(const u64 *__restrict__ bra, long long n, const double *__restrict__ h1e, const double *__restrict__ h2e,
                      const double *__restrict__ psi, GroupView gv,
                      const HitRun *__restrict__ runs, const u32 *__restrict__ run_cnt, int run_stride, const u32 *__restrict__ hits,
                      const u32 *__restrict__ self_pos, const double *__restrict__ hii, double *__restrict__ eloc,
                      double *__restrict__ psi0_out, u32 *__restrict__ heavy_list, ElocCounters *ctr, ExcGeom g, int per_warp) {
  __shared__ EvalTileSmem s_tile[kEvalThreads / 32];
  __shared__ SingleQueue<L> s_queue[kEvalThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  EvalTileSmem &T = s_tile[warp];
  SingleQueue<L> &q = s_queue[warp];
  // per_warp: samples a warp takes (32; 16 or 8 when the call has too few samples to fill the GPU with 32 per warp -- the hit
  // lists are walked 32 hits at a time whatever the number of samples they belong to)
  const long long s0 = ((long long)blockIdx.x * (kEvalThreads / 32) + warp) * per_warp;
  if (s0 >= n) return;
  const long long s = s0 + lane;
  const bool valid = lane < per_warp && s < n;
  // ---- this lane's sample ---------------------------------------------------------------------------------------------
  Onv<L> x;
#pragma unroll
  for (int w = 0; w < L; ++w) x.w[w] = valid ? bra[s * L + w] : 0ull;
  const int nruns = valid ? (int)run_cnt[s] : 0;
  const HitRun *my_runs = runs + s * run_stride;
  bool redo = false;
  u32 my_hits = 0;
  for (int r = 0; r < nruns; ++r) {
    const u32 c = my_runs[r].cnt;
    redo |= (c & kOverflow) != 0;
    my_hits += c & ~kOverflow;
  }
  // (the samples flagged for the reference's route go the same way: ~M binary searches each)
  const bool heavy = valid && (redo || my_hits > kHeavyHits);
  if (heavy) heavy_list[atomicAdd(&ctr->n_heavy, 1u)] = (u32)s;
  Cplx p0 = {0.0, 0.0};
  if (valid && !heavy) {
    const u32 sp = self_pos[s];
    if (sp != kNoSelf) p0 = load_psi<CPLX>(psi, (long long)__ldg(gv.rows[0] + sp));
  }
#pragma unroll
  for (int w = 0; w < L; ++w) T.x[lane][w] = x.w[w];
  T.p0[lane][0] = p0.re;
  T.p0[lane][1] = p0.im;
  {
    Cplx a0 = {0.0, 0.0};
    if (valid && !heavy) accumulate<CPLX>(a0, p0, p0, hii[s]);  // row 0: (psi0 / psi0) * H_xx
    T.acc[lane][0] = a0.re;
    T.acc[lane][1] = a0.im;
  }
  __syncwarp();
  const int max_runs = __reduce_max_sync(0xffffffffu, heavy ? 0 : nruns);
  // lane i evaluates entry i; the products go into the samples' accumulators in queue order (lane l adds those of sample l:
  // the entries of one sample need not be adjacent, so segment tails added in parallel would race); four terms in flight
  u32 qn = 0;
  auto flush = [&](u32 cnt) {
    Cplx v = {0.0, 0.0};
    u32 jq = 32;
    if ((u32)lane < cnt) {
      jq = q.j[lane];
      Onv<L> xq, yq;
#pragma unroll
      for (int w = 0; w < L; ++w) {
        xq.w[w] = T.x[jq][w];
        yq.w[w] = q.y[lane][w];
      }
      const Cplx pq = {T.p0[jq][0], T.p0[jq][1]};
      accumulate<CPLX>(v, load_psi<CPLX>(psi, q.row[lane]), pq, single_element<L, 4, double>(xq, yq, h1e, h2e, g.sorb));
    }
    Cplx a = {T.acc[lane][0], T.acc[lane][1]};
    for (u32 i = 0; i < cnt; ++i) {
      const u32 ji = __shfl_sync(0xffffffffu, jq, i);
      const double vr = __shfl_sync(0xffffffffu, v.re, i);
      const double vi = CPLX ? __shfl_sync(0xffffffffu, v.im, i) : 0.0;
      if (ji == (u32)lane) {
        a.re += vr;
        if (CPLX) a.im += vi;
      }
    }
    T.acc[lane][0] = a.re;
    T.acc[lane][1] = a.im;
    __syncwarp();
  };
  for (int r = 0; r < max_runs; ++r) {
    HitRun mine = {0u, 0u};
    if (!heavy && r < nruns) mine = my_runs[r];
    const u32 incl = warp_inclusive_sum(mine.cnt);
    const u32 total = __shfl_sync(0xffffffffu, incl, 31);
    for (u32 e0 = 0; e0 < total; e0 += 32) {
      const u32 e = e0 + (u32)lane;
      const int j = warp_segment_of(incl, e);  // the sample that holds hit e
      const u32 j_incl = __shfl_sync(0xffffffffu, incl, j), j_cnt = __shfl_sync(0xffffffffu, mine.cnt, j);
      const u32 j_off = __shfl_sync(0xffffffffu, mine.off, j);
      Onv<L> xs, y;
#pragma unroll
      for (int w = 0; w < L; ++w) xs.w[w] = T.x[j][w];
      y = xs;
      u32 row = 0;
      int kind = 0;  // 1 single, 2 double, 0 nothing to add
      if (e < total) kind = decode_hit<L, HALF>(gv, xs, hits[j_off + (e - (j_incl - j_cnt))], y, row);
      Cplx v = {0.0, 0.0};
      const Cplx pj = {T.p0[j][0], T.p0[j][1]};
      if (kind == 2) accumulate<CPLX>(v, load_psi<CPLX>(psi, row), pj, double_element<L, double>(xs, y, h2e));
      push_singles<L>(q, qn, kind, y, row, (u32)j, flush);
      // sum of v over the lanes of the same sample (adjacent), then the last lane of every sample adds it in
      const int jkey = e < total ? j : 32 + lane;  // idle lanes: segments of their own
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double ur = __shfl_up_sync(0xffffffffu, v.re, o);
        const double ui = CPLX ? __shfl_up_sync(0xffffffffu, v.im, o) : 0.0;
        const int uj = __shfl_up_sync(0xffffffffu, jkey, o);
        if (lane >= o && uj == jkey) {
          v.re += ur;
          if (CPLX) v.im += ui;
        }
      }
      const int nextj = __shfl_down_sync(0xffffffffu, jkey, 1);
      if (e < total && (lane == 31 || nextj != jkey)) {
        T.acc[j][0] += v.re;
        if (CPLX) T.acc[j][1] += v.im;
      }
      __syncwarp();
    }
  }
  if (qn) flush(qn);
  __syncwarp();
  const Cplx acc = {T.acc[lane][0], T.acc[lane][1]};
  if (valid && !heavy) {
    if (CPLX) {
      eloc[2 * s] = acc.re;
      eloc[2 * s + 1] = acc.im;
      psi0_out[2 * s] = p0.re;
      psi0_out[2 * s + 1] = p0.im;
    } else {
      eloc[s] = acc.re;
      psi0_out[s] = p0.re;
    }
  }
}

// ---- host side --------------------------------------------------------------------------------------------
// splits: CTAs per sample -- more than one only when there are too few samples to fill the GPU
static int scan_threads(int n_groups) {
  const int t = eloc_tuning().scan_threads;
  if (t == 64 || t == 128 || t == 256) return t;
  return n_groups <= 192 ? 128 : 256;
}

static int scan_splits(long long n, int n_groups, int warps) {
  if (n <= 0) return 1;
  long long want = (148LL * 8 + n - 1) / n;
  const long long cap = n_groups / warps > 1 ? n_groups / warps : 1;
  if (want > cap) want = cap;
  return (int)(want < 1 ? 1 : want);
}

// block route (eloc_block.cu)
long long block_scratch_bytes(long long n);
int block_run_stride();
int launch_eloc_block(const u64 *bra, long long n, const GroupView &gv, char *block_ws, ElocCounters *ctr, HitRun *runs, u32 *run_cnt,
                      int run_stride, u32 *hits, u32 *self_pos, u32 hit_cap, const ExcGeom &g, const u32 **slots_out, cudaStream_t st);

// the block route needs one-word ONVs (decided again at launch: it also needs N < 2^30 and the folded route)
bool block_route_wanted(long long n, const ExcGeom &g) {
  const ElocTuning &t = eloc_tuning();
  return t.block_enable && !t.full_keys && g.L == 1 && n >= t.block_min_samples && g.noB * g.nvB + 2 <= 258;
}

ElocScratch eloc_scratch_layout(long long n, const ExcGeom &g, bool block) {
  ElocScratch l;
  l.block = block;
  l.warps = scan_threads(g.noB * g.nvB + 2) / 32;
  if (block) {
    // every sample of the call in one go (the samples of a beta string must stay together); hits per sample the
    // buffer can take before samples fall back to the full route: 384 on average, at most 8 GiB in all
    l.batch = n < (1LL << 24) ? n : (1LL << 24);
    l.splits = 1;
    l.run_stride = block_run_stride() > l.warps ? block_run_stride() : l.warps;
    l.hit_cap = l.batch * 384 + 65536;
  } else {
    // hits per sample the global buffer can take before samples fall back to the full route, and a
    // batch size that keeps the buffer at about 2 GiB
    long long per_sample = (long long)g.nsd / 4;
    per_sample = per_sample < 256 ? 256 : (per_sample > 4096 ? 4096 : per_sample);
    l.batch = (1LL << 29) / per_sample;
    l.batch = l.batch < 1024 ? 1024 : (l.batch > (1LL << 18) ? (1LL << 18) : l.batch);
    const long long nb0 = n < l.batch ? n : l.batch;
    l.splits = scan_splits(nb0, g.noB * g.nvB + 2, l.warps);
    l.run_stride = l.splits * l.warps;
    l.hit_cap = nb0 * per_sample + 65536;
  }
  const long long nb = n < l.batch ? n : l.batch;
  if (l.hit_cap > 0x7fffffffLL) l.hit_cap = 0x7fffffffLL;
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  l.hii = 0;
  l.self_pos = up(l.hii + 8 * n);
  l.run_cnt = up(l.self_pos + 4 * nb);
  l.heavy = up(l.run_cnt + 4 * nb);
  l.runs = up(l.heavy + 4 * nb);
  l.counters = up(l.runs + (long long)sizeof(HitRun) * nb * l.run_stride);
  l.block_ws = l.counters + 256;
  l.hits = up(l.block_ws + (block ? block_scratch_bytes(nb) : 0));
  l.total = l.hits + 4 * l.hit_cap + 256;
  return l;
}

// the caller's scratch serves either route (the route also depends on the table, which this function does not see)
long long eloc_scratch_bytes(long long n, const ExcGeom &g) {
  long long t = eloc_scratch_layout(n, g, false).total;
  if (block_route_wanted(n, g)) {
    const long long tb = eloc_scratch_layout(n, g, true).total;
    if (tb > t) t = tb;
  }
  return t;
}

// The scan phase of one batch of samples bra[0, nb): the grouping pass and the block kernel (block route), then the
// per-sample scan kernel.  Leaves the batch's hit lists in the scratch (runs, run_cnt, hits, self_pos).
template <int L, bool HALF>
static int scan_batch(const u64 *bra, long long nb, const GroupView &gv, char *scratch, const ElocScratch &lay, const ExcGeom &g,
                      cudaStream_t st) {
  u32 *self_pos = reinterpret_cast<u32 *>(scratch + lay.self_pos);
  u32 *run_cnt = reinterpret_cast<u32 *>(scratch + lay.run_cnt);
  HitRun *runs = reinterpret_cast<HitRun *>(scratch + lay.runs);
  ElocCounters *ctr = reinterpret_cast<ElocCounters *>(scratch + lay.counters);
  u32 *hits = reinterpret_cast<u32 *>(scratch + lay.hits);
  ScanSmem sm = scan_smem(g, lay.warps);
  const int f = eloc_tuning().search_factor;  // parity tests: force the search route on small tables
  if (f >= 1 && f <= 4096) sm.search_factor = (u32)f;
  const size_t smem = sm.total;
  if (smem > 227 * 1024) {
    set_error("eloc: %zu bytes of shared memory per CTA needed for sorb = %d, noA = %d, noB = %d (limit 227 KB)", smem, g.sorb, g.noA, g.noB);
    return 1;
  }
  auto scan = lay.warps == 2 ? eloc_scan_kernel<L, HALF, 64> : (lay.warps == 4 ? eloc_scan_kernel<L, HALF, 128> : eloc_scan_kernel<L, HALF, 256>);
  if (smem > 48 * 1024 && cudaFuncSetAttribute(scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return check_launch("eloc_scan_kernel smem opt-in");
  const int splits = lay.splits;
  if (cudaMemsetAsync(ctr, 0, sizeof(ElocCounters), st) != cudaSuccess) return check_launch("eloc counters memset");
  if (cudaMemsetAsync(self_pos, 0xff, 4 * (size_t)nb, st) != cudaSuccess) return check_launch("eloc self memset");
  const u32 *ids = nullptr;
  unsigned grid = (unsigned)(nb * splits);
  if (HALF && lay.block) {
    // samples that share a beta string with enough others: tiles of the block kernel; the rest: per-sample kernel,
    // which finds its work list (and its length) in device memory -- a fixed grid of persistent CTAs
    if (int rc = launch_eloc_block(bra, nb, gv, scratch + lay.block_ws, ctr, runs, run_cnt, lay.run_stride, hits, self_pos,
                                   (u32)lay.hit_cap, g, &ids, st))
      return rc;
    const long long cap = 148LL * 12;
    grid = (unsigned)(nb < cap ? nb : cap);
  }
  scan<<<grid, lay.warps * 32, smem, st>>>(bra, nb, gv, runs, run_cnt, lay.run_stride, hits, self_pos, ctr, (u32)lay.hit_cap, splits, ids,
                                           g, sm);
  count_launch();
  return check_launch("eloc_scan_kernel");
}

int launch_scan_batch(const u64 *bra, long long nb, const GroupView &gv, char *scratch, const ElocScratch &lay, const ExcGeom &g, bool half,
                      cudaStream_t st) {
  if (half) return scan_batch<1, true>(bra, nb, gv, scratch, lay, g, st);
  switch (g.L) {
    case 1: return scan_batch<1, false>(bra, nb, gv, scratch, lay, g, st);
    case 2: return scan_batch<2, false>(bra, nb, gv, scratch, lay, g, st);
    case 3: return scan_batch<3, false>(bra, nb, gv, scratch, lay, g, st);
  }
  set_error("unsupported ONV length L=%d", g.L);
  return 1;
}

bool eloc_half_route(long long N, const ExcGeom &g) { return g.L == 1 && N < (1LL << 30) && !eloc_tuning().full_keys; }

template <int L, bool CPLX, bool HALF>
static int launch_eloc_LC(const u64 *bra, long long n, const double *h1e, const double *h2e, const u64 *key, const double *psi,
                          long long N, const GroupView &gv, char *scratch, const ElocScratch &lay, double *eloc, double *psi0,
                          const ExcGeom &g, cudaStream_t st, SideLane *diag_lane) {
  double *hii = reinterpret_cast<double *>(scratch + lay.hii);
  u32 *self_pos = reinterpret_cast<u32 *>(scratch + lay.self_pos);
  u32 *run_cnt = reinterpret_cast<u32 *>(scratch + lay.run_cnt);
  u32 *heavy = reinterpret_cast<u32 *>(scratch + lay.heavy);
  HitRun *runs = reinterpret_cast<HitRun *>(scratch + lay.runs);
  ElocCounters *ctr = reinterpret_cast<ElocCounters *>(scratch + lay.counters);
  u32 *hits = reinterpret_cast<u32 *>(scratch + lay.hits);
  const int w = CPLX ? 2 : 1;
  for (long long b0 = 0; b0 < n; b0 += lay.batch) {
    const long long nb = n - b0 < lay.batch ? n - b0 : lay.batch;
    if (int rc = scan_batch<L, HALF>(bra + b0 * L, nb, gv, scratch, lay, g, st)) return rc;
    if (diag_lane != nullptr) {  // the diagonal elements (side stream) must be there now
      if (!side_join(diag_lane, st)) return check_launch("eloc: join of the diagonal kernel");
      diag_lane = nullptr;
    }
    // 32 samples per warp; calls too small to fill the GPU that way keep one warp per sample
    if ((nb >= 148LL * 32 * 8 && eloc_tuning().eval_tiles) || eloc_tuning().eval_tiles == 2) {
      // samples per warp: 32 (fewer per warp were measured slower even for a rank's 125 000 samples at 8 GPUs: 178 against
      // 168 us with 8 per warp -- the per-warp bookkeeping outweighs the shorter tail)
      const int per_warp = 32;
      const long long per_cta = (long long)per_warp * (kEvalThreads / 32);
      const unsigned eb = (unsigned)((nb + per_cta - 1) / per_cta);
      eloc_eval_tile_kernel<L, CPLX, HALF><<<eb, kEvalThreads, 0, st>>>(bra + b0 * L, nb, h1e, h2e, psi, gv, runs, run_cnt,
                                                                        lay.run_stride, hits, self_pos, hii + b0, eloc + b0 * w,
                                                                        psi0 + b0 * w, heavy, ctr, g, per_warp);
      count_launch();
      // the samples with long hit lists, one warp each (a fixed grid of persistent warps reads the list's length on the device)
      const long long cap = 148LL * 12;
      const long long want = (nb + kEvalThreads / 32 - 1) / (kEvalThreads / 32);
      eloc_eval_kernel<L, CPLX, HALF><<<(unsigned)(want < cap ? want : cap), kEvalThreads, 0, st>>>(
          bra + b0 * L, nb, h1e, h2e, key, psi, N, gv, runs, run_cnt, lay.run_stride, hits, self_pos, hii + b0, eloc + b0 * w, psi0 + b0 * w,
          heavy, ctr, g);
    } else {
      const unsigned eb = (unsigned)((nb + kEvalThreads / 32 - 1) / (kEvalThreads / 32));
      eloc_eval_kernel<L, CPLX, HALF><<<eb, kEvalThreads, 0, st>>>(bra + b0 * L, nb, h1e, h2e, key, psi, N, gv, runs, run_cnt, lay.run_stride,
                                                                   hits, self_pos, hii + b0, eloc + b0 * w, psi0 + b0 * w, nullptr, ctr, g);
    }
    count_launch();
    if (int rc = check_launch("eloc_eval_kernel")) return rc;
  }
  return 0;
}

int launch_eloc(const u64 *bra, long long n, const double *h1e, const double *h2e, const u64 *key, const double *psi, int cplx,
                long long N, const void *group_ws, void *scratch, long long scratch_bytes, double *eloc, double *psi0,
                const ExcGeom &g, cudaStream_t st) {
  if (n == 0) return 0;
  // folded 32-bit strings: one-word ONVs, two flag bits in the hit word.  The tuning knob full_keys forces the
  // full-key route (the one multi-word ONVs take) -- used by the parity tests to cover both.
  const bool half = eloc_half_route(N, g);
  const ElocScratch lay = eloc_scratch_layout(n, g, half && block_route_wanted(n, g));
  if (scratch_bytes < lay.total) {
    set_error("eloc scratch too small: %lld < %lld bytes", scratch_bytes, lay.total);
    return 4;
  }
  char *sc = static_cast<char *>(scratch);
  // the diagonal <x|H|x> needs neither the table nor the hits: it runs on a side stream next to the scan kernels (which
  // leave more than half of the warp slots free) and is joined before the evaluation
  SideLane *side = side_lane(1);
  const bool forked = side_fork(side, st);
  if (int rc = launch_diag_f64(bra, h1e, h2e, reinterpret_cast<double *>(sc + lay.hii), n, 1, g.L, g.sorb, g.nele, forked ? side->stream : st))
    return rc;
  const GroupView gv = group_view(group_ws, N, g.L);
  SideLane *join = forked ? side : nullptr;  // joined before the first evaluation kernel
#define PYNQS_ELOC_CASE(LL)                                                                                                  \
  case LL:                                                                                                                   \
    return cplx ? launch_eloc_LC<LL, true, false>(bra, n, h1e, h2e, key, psi, N, gv, sc, lay, eloc, psi0, g, st, join)       \
                : launch_eloc_LC<LL, false, false>(bra, n, h1e, h2e, key, psi, N, gv, sc, lay, eloc, psi0, g, st, join);
  if (half) {
    return cplx ? launch_eloc_LC<1, true, true>(bra, n, h1e, h2e, key, psi, N, gv, sc, lay, eloc, psi0, g, st, join)
                : launch_eloc_LC<1, false, true>(bra, n, h1e, h2e, key, psi, N, gv, sc, lay, eloc, psi0, g, st, join);
  }
  switch (g.L) {
    PYNQS_ELOC_CASE(1)
    PYNQS_ELOC_CASE(2)
    PYNQS_ELOC_CASE(3)
  }
#undef PYNQS_ELOC_CASE
  set_error("unsupported ONV length L=%d", g.L);
  return 1;
}

}  // namespace pynqs
