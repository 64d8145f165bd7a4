// gindex.cu -- build of the string-grouped table copies of gindex.cuh.  All asynchronous on the
// caller's stream, no host round trip:
//   1. bucket : every key computes its two bucket ids (hash of its beta string, hash of its alpha
//               string); adjacent equal keys raise has_dup;
//   2. sort   : one stable radix sort per grouping of (bucket id, row) over log2(buckets) bits
//               (cub onesweep) -- rows inside a bucket stay ascending;
//   3. finish : gather the keys into bucket order and write the bucket boundaries (and, L = 1, the bit planes of the
//               beta-grouped copy's folded alpha strings).
#include <mutex>

#include <cub/device/device_radix_sort.cuh>

#include "gindex.cuh"

namespace pynqs {

GroupLayout group_layout(long long N, int L) {
  GroupLayout l;
  l.log2_buckets = group_log2_buckets(N);
  const long long nb = (1LL << l.log2_buckets) + 1;
  auto up = [](long long v) { return (v + 255) & ~255LL; };
  long long o = (long long)sizeof(GroupHeader);
  for (int g = 0; g < 2; ++g) {
    l.start_off[g] = o;
    o = up(o + nb * 4);
  }
  for (int g = 0; g < 2; ++g) {
    l.keys_off[g] = o;
    o = up(o + N * 8 * L);
  }
  for (int g = 0; g < 2; ++g) {
    l.rows_off[g] = o;
    o = up(o + N * 4);
  }
  for (int g = 0; g < 2; ++g) {
    l.half_off[g] = o;
    if (L == 1) o = up(o + N * 4);
  }
  l.pos_off = o;
  o = up(o + N * 4);
  l.planes_off = o;
  if (L == 1) o = up(o + (N + 31) / 32 * 128);
  l.scratch_off = o;
  for (int g = 0; g < 2; ++g)
    for (int k = 0; k < 2; ++k) {
      l.bkt_off[g][k] = o;
      o = up(o + N * 4);
    }
  l.iota_off = o;
  o = up(o + N * 4);
  size_t tmp = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const u32 *)nullptr, (u32 *)nullptr, (const u32 *)nullptr, (u32 *)nullptr,
                                  (int)(N > 0 ? N : 1), 0, 32);
  l.cub_off = o;
  l.cub_bytes = tmp;
  l.total = up(o + 2 * (long long)up((long long)tmp)) + 256;  // one temporary area per (concurrent) sort
  return l;
}

long long group_workspace_bytes(long long N, int L) { return group_layout(N, L).total; }

GroupView group_view(const void *ws, long long N, int L) {
  const GroupLayout l = group_layout(N, L);
  const char *b = static_cast<const char *>(ws);
  GroupView v;
  v.hdr = reinterpret_cast<const GroupHeader *>(b);
  for (int g = 0; g < 2; ++g) {
    v.start[g] = reinterpret_cast<const u32 *>(b + l.start_off[g]);
    v.keys[g] = reinterpret_cast<const u64 *>(b + l.keys_off[g]);
    v.rows[g] = reinterpret_cast<const u32 *>(b + l.rows_off[g]);
    v.half[g] = L == 1 ? reinterpret_cast<const u32 *>(b + l.half_off[g]) : nullptr;
  }
  v.pos = reinterpret_cast<const u32 *>(b + l.pos_off);
  v.planes = L == 1 ? reinterpret_cast<const u32 *>(b + l.planes_off) : nullptr;
  v.shift = 32u - l.log2_buckets;
  return v;
}

template <int L>
__global__ void __launch_bounds__(256)
group_bucket_kernel(const u64 *__restrict__ key, long long N, GroupHeader *hdr, u32 log2_buckets, u32 *__restrict__ bktB,
                    u32 *__restrict__ bktA, u32 *__restrict__ iota) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    hdr->log2_buckets = log2_buckets;
    hdr->n_keys = (u64)N;
  }
  if (i >= N) return;
  const Onv<L> x = load_onv<L>(key + i * L);
  if (i > 0 && eq_onv<L>(load_onv<L>(key + (i - 1) * L), x)) atomicExch(&hdr->has_dup, 1u);
  const u32 shift = 32u - log2_buckets;
  bktB[i] = group_bucket<L>(x, 0, shift);
  bktA[i] = group_bucket<L>(x, 1, shift);
  iota[i] = (u32)i;
}

// blockIdx.y = grouping
template <int L>
__global__ void __launch_bounds__(256)
group_finish_kernel(const u64 *__restrict__ key, long long N, u32 log2_buckets, const u32 *__restrict__ bktB,
                    const u32 *__restrict__ bktA, const u32 *__restrict__ rowsB, const u32 *__restrict__ rowsA, u64 *__restrict__ keysB,
                    u64 *__restrict__ keysA, u32 *__restrict__ startB, u32 *__restrict__ startA, u32 *__restrict__ halfB,
                    u32 *__restrict__ halfA, u32 *__restrict__ posB, u32 *__restrict__ planes) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool ga = blockIdx.y != 0;
  if (L == 1 && !ga && (i & ~31LL) < N) {
    // the folded alpha strings of the warp's 32 positions bit-transposed: one ballot per bit, lane o keeps ballot o
    // (blocks are whole warps, so all 32 lanes are here; the positions past N count as empty strings)
    const u32 fa = i < N ? fold_alpha(key[rowsB[i]]) : 0u;
    u32 plane = 0;
#pragma unroll
    for (int o = 0; o < 32; ++o) {
      const u32 b = __ballot_sync(0xffffffffu, (fa >> o) & 1u);
      if ((threadIdx.x & 31) == o) plane = b;
    }
    planes[i] = plane;  // = planes[(i / 32) * 32 + lane]
  }
  if (i >= N) return;
  const u32 *bkt = ga ? bktA : bktB;
  const u32 *rows = ga ? rowsA : rowsB;
  u64 *keys = ga ? keysA : keysB;
  u32 *start = ga ? startA : startB;
  const u32 row = rows[i];
  if (!ga) posB[row] = (u32)i;  // where the beta-grouped copy keeps every table row
#pragma unroll
  for (int w = 0; w < L; ++w) keys[i * L + w] = key[(long long)row * L + w];
  if (L == 1) {  // the other string of the key, folded
    const u64 k0 = key[(long long)row * L];
    if (ga) halfA[i] = fold_beta(k0);
    else halfB[i] = fold_alpha(k0);
  }
  // bucket boundaries: start[t] = first position whose bucket id is >= t
  const u32 b = bkt[i];
  const long long first = i == 0 ? 0 : (long long)bkt[i - 1] + 1;
  for (long long t = first; t <= (long long)b; ++t) start[t] = (u32)i;
  if (i == N - 1) {
    const long long nb = 1LL << log2_buckets;
    for (long long t = (long long)b + 1; t <= nb; ++t) start[t] = (u32)N;
  }
}

__global__ void __launch_bounds__(256) group_empty_kernel(GroupHeader *hdr, u32 log2_buckets, u32 *startB, u32 *startA) {
  const long long nb = (1LL << log2_buckets) + 1;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    hdr->log2_buckets = log2_buckets;
    hdr->n_keys = 0;
  }
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nb; t += (long long)gridDim.x * blockDim.x)
    startB[t] = startA[t] = 0u;
}

// The two sorts are independent and far too small to fill the GPU (10^6 keys: ~16 us per pass): the second one
// runs on a side stream, forked from and joined back into the caller's stream with events (capturable).
static std::mutex g_side_mutex;
static SideLane g_side[2][64];

SideLane *side_lane(int which) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(g_side_mutex);
  SideLane &s = g_side[which & 1][dev];
  if (s.stream == nullptr) {
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
      s.stream = nullptr;
      cudaGetLastError();
      return nullptr;
    }
  }
  return &s;
}

bool side_fork(SideLane *s, cudaStream_t st) {
  const bool ok = s != nullptr && cudaEventRecord(s->fork, st) == cudaSuccess && cudaStreamWaitEvent(s->stream, s->fork, 0) == cudaSuccess;
  if (!ok) cudaGetLastError();
  return ok;
}

bool side_join(SideLane *s, cudaStream_t st) {
  return cudaEventRecord(s->join, s->stream) == cudaSuccess && cudaStreamWaitEvent(st, s->join, 0) == cudaSuccess;
}

int launch_group_build(const u64 *key, long long N, int L, void *ws, long long ws_bytes, cudaStream_t st) {
  if (N >= (1LL << 31)) {
    set_error("the grouped table supports fewer than 2^31 keys (got %lld)", N);
    return 1;
  }
  if (L < 1 || L > 3) {
    set_error("unsupported ONV length L=%d", L);
    return 1;
  }
  const GroupLayout l = group_layout(N, L);
  if (ws_bytes < l.total) {
    set_error("group index workspace too small: %lld < %lld bytes", ws_bytes, l.total);
    return 4;
  }
  char *b = static_cast<char *>(ws);
  GroupHeader *hdr = reinterpret_cast<GroupHeader *>(b);
  u32 *start[2] = {reinterpret_cast<u32 *>(b + l.start_off[0]), reinterpret_cast<u32 *>(b + l.start_off[1])};
  u64 *keys[2] = {reinterpret_cast<u64 *>(b + l.keys_off[0]), reinterpret_cast<u64 *>(b + l.keys_off[1])};
  u32 *rows[2] = {reinterpret_cast<u32 *>(b + l.rows_off[0]), reinterpret_cast<u32 *>(b + l.rows_off[1])};
  u32 *bkt[2][2] = {{reinterpret_cast<u32 *>(b + l.bkt_off[0][0]), reinterpret_cast<u32 *>(b + l.bkt_off[0][1])},
                    {reinterpret_cast<u32 *>(b + l.bkt_off[1][0]), reinterpret_cast<u32 *>(b + l.bkt_off[1][1])}};
  u32 *iota = reinterpret_cast<u32 *>(b + l.iota_off);
  u32 *half[2] = {reinterpret_cast<u32 *>(b + l.half_off[0]), reinterpret_cast<u32 *>(b + l.half_off[1])};
  u32 *posB = reinterpret_cast<u32 *>(b + l.pos_off);
  u32 *planes = reinterpret_cast<u32 *>(b + l.planes_off);
  if (cudaMemsetAsync(hdr, 0, sizeof(GroupHeader), st) != cudaSuccess) return check_launch("group header memset");
  if (N == 0) {
    group_empty_kernel<<<148, 256, 0, st>>>(hdr, l.log2_buckets, start[0], start[1]);
    count_launch();
    return check_launch("group_empty_kernel");
  }
  const unsigned blocks = (unsigned)((N + 255) / 256);
  switch (L) {
    case 1: group_bucket_kernel<1><<<blocks, 256, 0, st>>>(key, N, hdr, l.log2_buckets, bkt[0][0], bkt[1][0], iota); break;
    case 2: group_bucket_kernel<2><<<blocks, 256, 0, st>>>(key, N, hdr, l.log2_buckets, bkt[0][0], bkt[1][0], iota); break;
    case 3: group_bucket_kernel<3><<<blocks, 256, 0, st>>>(key, N, hdr, l.log2_buckets, bkt[0][0], bkt[1][0], iota); break;
    default: set_error("unsupported ONV length L=%d", L); return 1;
  }
  count_launch();
  SideLane *side = side_lane(0);
  const bool forked = side_fork(side, st);
  const long long cub_stride = (l.cub_bytes + 255) / 256 * 256;
  for (int g = 0; g < 2; ++g) {
    size_t tmp = l.cub_bytes;
    const cudaStream_t sg = (g == 1 && forked) ? side->stream : st;
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(b + l.cub_off + g * cub_stride, tmp, (const u32 *)bkt[g][0], bkt[g][1],
                                                          (const u32 *)iota, rows[g], (int)N, 0, (int)l.log2_buckets, sg);
    if (e != cudaSuccess) {
      set_error("group sort: CUDA error %d (%s)", (int)e, cudaGetErrorString(e));
      return 3;
    }
    count_launch(((int)l.log2_buckets + 7) / 8 + 2);
  }
  if (forked && !side_join(side, st)) return check_launch("group build join");
  const dim3 grid(blocks, 2);
#define PYNQS_FINISH(LL)                                                                                                           \
  group_finish_kernel<LL><<<grid, 256, 0, st>>>(key, N, l.log2_buckets, bkt[0][1], bkt[1][1], rows[0], rows[1], keys[0], keys[1], \
                                                start[0], start[1], half[0], half[1], posB, planes)
  switch (L) {
    case 1: PYNQS_FINISH(1); break;
    case 2: PYNQS_FINISH(2); break;
    default: PYNQS_FINISH(3); break;
  }
#undef PYNQS_FINISH
  count_launch();
  return check_launch("group index build");
}

}  // namespace pynqs
