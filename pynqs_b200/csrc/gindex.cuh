// gindex.cuh -- the string-grouped copy of the unique-sample table that the local-energy kernels
// scan (device side).
//
// An ONV is an (alpha string, beta string) pair (even / odd bits).  Every determinant connected to
// a sample x shares a string with x or with a single excitation of x:
//     alpha single / alpha-alpha double : beta string of x,        alpha part at distance 2 / 4
//     beta single  / beta-beta double   : alpha string of x,       beta part at distance 2 / 4
//     alpha-beta double                 : beta string of one of the noB*nvB beta singles of x,
//                                         alpha part at distance 2
// So instead of forming the ~M connected determinants and searching each one in the table
// (binary_search_BigInteger, cpp_src/tensor/cpu_tensor.cpp:589-640 -- ~20 dependent loads per
// determinant, 99 % of them misses for a sparse table), the kernels go the other way round: they
// visit the few GROUPS of table keys that carry one of those strings and test every key of the
// group with XOR + popcount.  A group is a handful of consecutive keys: coalesced loads, no hashing
// of the connected determinants, and what survives the test IS a hit (row known, nothing to verify).
//
// For one-word ONVs (sorb <= 64) each copy also carries the OTHER string of every key folded into
// 32 bits (fold_alpha / fold_beta: injective and popcount-preserving), so that the test of a key
// is one 4-byte load, one XOR and one popcount; what passes is checked against the full key later.
//
// Layout: the table is copied twice, bucketed by hash(beta string) ("B") and by hash(alpha string)
// ("A"): start_g[2^b + 1] (u32), keys_g[N] (the keys in bucket order; inside a bucket ascending,
// because the sort is stable and the input table is sorted), rows_g[N] (row in the sorted table).
// A bucket normally holds one group; when two strings share a bucket the exact test on the keys
// still separates them, so collisions cost a little work and never change a result.
#pragma once
#include "common.cuh"
#include "lut.cuh"

namespace pynqs {

struct GroupHeader {
  u32 log2_buckets;
  u32 has_dup;  // two equal adjacent keys in the sorted table: the kernels fall back to the classic search
  u64 n_keys;
  u32 pad[60];
};
static_assert(sizeof(GroupHeader) == 256, "header is 256 bytes");

struct GroupLayout {
  u32 log2_buckets;
  long long start_off[2], keys_off[2], rows_off[2], half_off[2], pos_off, planes_off, scratch_off, total;
  long long bkt_off[2][2], iota_off;  // build scratch: bucket ids (in / out per grouping), identity rows
  long long cub_off;
  size_t cub_bytes;
};

__host__ __device__ inline u32 group_log2_buckets(long long N) {
  u32 lg = 4;
  while ((1LL << lg) < N && lg < 28) ++lg;
  return lg;
}

struct GroupView {
  const GroupHeader *hdr;
  const u32 *start[2];  // [0] bucketed by beta string, [1] by alpha string
  const u64 *keys[2];
  const u32 *rows[2];
  const u32 *half[2];  // L = 1 only: [0] folded alpha strings in B order, [1] folded beta strings in A order
  const u32 *pos;      // position of every row of the sorted table in the beta-grouped copy (inverse of rows[0])
  const u32 *planes;   // L = 1 only: half[0] bit-transposed, planes[c * 32 + o] = bit o of the keys c * 32 .. c * 32 + 31
  u32 shift;  // 32 - log2_buckets
};

// the alpha (even) / beta (odd) bits of a one-word ONV folded into 32 bits
__device__ __forceinline__ u32 fold_alpha(u64 w) {
  const u64 e = w & kEven;
  return (u32)e | ((u32)(e >> 32) << 1);
}
__device__ __forceinline__ u32 fold_beta(u64 w) {
  const u64 o = w & kOdd;
  return ((u32)o >> 1) | (u32)(o >> 32);
}

// 32-bit hash of one spin string (the words masked to the even or the odd bits)
template <int L>
__device__ __forceinline__ u32 string_hash32(const Onv<L> &x, u64 spin_mask) {
  u32 a = (u32)(x.w[0] & spin_mask), b = (u32)((x.w[0] & spin_mask) >> 32);
#pragma unroll
  for (int i = 1; i < L; ++i) {
    const u64 w = x.w[i] & spin_mask;
    a = (a ^ (a >> 15)) * 0x2C1B3C6Du + (u32)w;
    b = (b ^ (b >> 13)) * 0x297A2D39u + (u32)(w >> 32);
  }
  u32 h = a * 0x27D4EB2Fu + b * 0x165667B1u;
  h ^= h >> 16;
  h *= 0x7FEB352Du;
  h ^= h >> 15;
  h *= 0x846CA68Bu;
  h ^= h >> 16;
  return h;
}

// grouping 0 buckets by the beta string, grouping 1 by the alpha string
template <int L>
__device__ __forceinline__ u32 group_bucket(const Onv<L> &x, int grouping, u32 shift) {
  return string_hash32<L>(x, grouping == 0 ? kOdd : kEven) >> shift;
}

// binary search of y among the ascending keys [lo, hi) of one bucket; position or 0xffffffff
template <int L>
__device__ __forceinline__ u32 bucket_search(const u64 *__restrict__ keys, u32 lo, u32 hi, const Onv<L> &y) {
  while (lo < hi) {
    const u32 mid = lo + ((hi - lo) >> 1);
    const int c = cmp_onv<L>(load_onv<L>(keys + (size_t)mid * L), y);
    if (c == 0) return mid;
    if (c < 0) lo = mid + 1;
    else hi = mid;
  }
  return 0xffffffffu;
}

// table row of y, or -1: the beta-grouped copy, or the classic binary search over a table with duplicate keys
template <int L>
__device__ __forceinline__ long long spin_find(const u64 *__restrict__ key, long long N, const GroupView &gv, bool dup, const Onv<L> &y) {
  if (dup) return classic_search<L>(key, N, y);
  const u32 b = group_bucket<L>(y, 0, gv.shift);
  const u32 pos = bucket_search<L>(gv.keys[0], __ldg(gv.start[0] + b), __ldg(gv.start[0] + b + 1), y);
  return pos == 0xffffffffu ? -1 : (long long)__ldg(gv.rows[0] + pos);
}

// host side (gindex.cu)
// A side stream per device with a pair of events: independent kernels of one call run next to the caller's stream
// (fork: the side stream waits for what the caller's stream has queued; join: the caller's stream waits for the side
// stream).  Capturable in a CUDA graph.  `which` selects one of two lanes (the table build and the local energy never share).
struct SideLane {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
SideLane *side_lane(int which);
bool side_fork(SideLane *s, cudaStream_t st);
bool side_join(SideLane *s, cudaStream_t st);

GroupLayout group_layout(long long N, int L);
GroupView group_view(const void *ws, long long N, int L);

}  // namespace pynqs
