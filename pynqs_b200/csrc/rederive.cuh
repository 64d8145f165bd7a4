// rederive.cuh -- <x|H|y> from the two bit strings alone: the excitation is re-derived from x ^ y
// (diff_type cpu/onstate.cpp:10-20, diff_orb :34-55, dispatch cpu/hamiltonian.cpp:87-102) and then
// evaluated by the same exc_element / diag_element the fused operator uses, so both routes give
// bit-identical values.
#pragma once
#include "common.cuh"

namespace pynqs {

// highest set bit over all words, removing it
template <int L>
__device__ __forceinline__ int pop_highest(Onv<L> &d) {
#pragma unroll
  for (int i = L - 1; i >= 0; --i) {
    if (d.w[i]) {
      const int b = 63 - __clzll((long long)d.w[i]);
      d.w[i] ^= 1ull << b;
      return 64 * i + b;
    }
  }
  return 0;
}

template <int L, typename T>
__device__ __forceinline__ T rederived_element(const Onv<L> &x, const Onv<L> &y, const T *__restrict__ h1e,
                                               const T *__restrict__ h2e, int sorb, int nele) {
  Onv<L> cre, ann;  // bra-only / ket-only orbitals
  int nc = 0, na = 0;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = x.w[i] ^ y.w[i];
    cre.w[i] = d & x.w[i];
    ann.w[i] = d & y.w[i];
    nc += __popcll(cre.w[i]);
    na += __popcll(ann.w[i]);
  }
  if (nc == 0 && na == 0) return diag_element<L, T>(x, h1e, h2e, sorb, nele);
  Exc e;
  if (nc == 1 && na == 1) {
    const int h = pop_highest<L>(cre), p = pop_highest<L>(ann);
    e.h0 = h | ((count_below<L>(x, h) & 1) << 8);
    e.p0 = p | ((count_below<L>(x, p) & 1) << 8);
    e.h1 = e.p1 = 0;
    e.dbl = false;
    return exc_element<L, T>(x, e, h1e, h2e, sorb);
  }
  if (nc == 2 && na == 2) {
    const int h0 = pop_highest<L>(cre), h1 = pop_highest<L>(cre);
    const int p0 = pop_highest<L>(ann), p1 = pop_highest<L>(ann);
    e.h0 = h0 | ((count_below<L>(x, h0) & 1) << 8);
    e.h1 = h1 | ((count_below<L>(x, h1) & 1) << 8);
    e.p0 = p0 | ((count_below<L>(x, p0) & 1) << 8);
    e.p1 = p1 | ((count_below<L>(x, p1) & 1) << 8);
    e.dbl = true;
    return exc_element<L, T>(x, e, h1e, h2e, sorb);
  }
  return (T)0.0;
}

// class of the pair from the popcounts of bra-only / ket-only orbitals: 1 single, 2 double, 0 anything else
// (the diagonal included -- callers treat x == y themselves)
template <int L>
__device__ __forceinline__ int excitation_class(const Onv<L> &x, const Onv<L> &y) {
  int nc = 0, na = 0;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = x.w[i] ^ y.w[i];
    nc += __popcll(d & x.w[i]);
    na += __popcll(d & y.w[i]);
  }
  return (nc == 1 && na == 1) ? 1 : ((nc == 2 && na == 2) ? 2 : 0);
}

// the two set bits of m (exactly two are set): highest and lowest position, without data-dependent branches
template <int L>
__device__ __forceinline__ void two_set_bits(const Onv<L> &m, u32 &hi, u32 &lo) {
  hi = 0;
  lo = 0;
  bool have = false;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 w = m.w[i];
    const bool nz = w != 0;
    const u32 top = (u32)(64 * i + 63 - __clzll((long long)(w | 1ull)));
    const u32 bot = (u32)(64 * i + __ffsll((long long)w) - 1);
    hi = nz ? top : hi;  // later (more significant) words win
    lo = (nz && !have) ? bot : lo;
    have = have || nz;
  }
}

// Double excitation x -> y (two bra-only and two ket-only orbitals) from the bit strings, branch-free so that the
// lanes of a warp stay together: the same value as rederived_element / exc_element.
template <int L, typename T>
__device__ __forceinline__ T double_element(const Onv<L> &x, const Onv<L> &y, const T *__restrict__ h2e) {
  Onv<L> cre, ann;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = x.w[i] ^ y.w[i];
    cre.w[i] = d & x.w[i];
    ann.w[i] = d & y.w[i];
  }
  u32 hh, hl, ph, pl;
  two_set_bits<L>(cre, hh, hl);
  two_set_bits<L>(ann, ph, pl);
  const int par = count_below<L>(x, (int)hh) ^ count_below<L>(x, (int)hl) ^ count_below<L>(x, (int)ph) ^ count_below<L>(x, (int)pl);
  const int cross = (int)(hh < ph) + (int)(hl < ph) + (int)(hh < pl) + (int)(hl < pl);
  const int sg = par ^ cross ^ 1;
  T v = (T)1.0 * __ldg(h2e + pair_offset(hh, hl, ph, pl));
  v *= (sg & 1) ? (T)-1.0 : (T)1.0;
  return v;
}

// Single excitation x -> y evaluated by one lane: the excitation re-derived as in rederived_element, then exc_element's single
// branch -- the same terms (two_body) added in the same order (occupied orbitals by word ascending, bits descending), so the
// same value.  The terms are loaded AHEAD at a time before they are added, instead of one dependent load per addition (each
// term in flight holds a register of the caller's budget).
template <int L, int AHEAD, typename T>
__device__ __forceinline__ T single_element(const Onv<L> &x, const Onv<L> &y, const T *__restrict__ h1e, const T *__restrict__ h2e,
                                            int sorb) {
  Onv<L> cre, ann;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = x.w[i] ^ y.w[i];
    cre.w[i] = d & x.w[i];
    ann.w[i] = d & y.w[i];
  }
  const u32 h = (u32)pop_highest<L>(cre), p = (u32)pop_highest<L>(ann);
  T v = (T)0.0;
  v += __ldg(h1e + (size_t)p * sorb + h);
#pragma unroll
  for (int i = 0; i < L; ++i) {
    u64 rest = x.w[i];
    while (rest) {
      T t[AHEAD];
      int n = 0;
#pragma unroll
      for (int u = 0; u < AHEAD; ++u) {
        t[u] = (T)0.0;
        if (rest) {
          const int b = 63 - __clzll((long long)rest);
          rest ^= 1ull << b;
          const u32 k = (u32)(64 * i + b);
          t[u] = two_body<T>(h2e, h, k, p, k);
          n = u + 1;
        }
      }
#pragma unroll
      for (int u = 0; u < AHEAD; ++u)
        if (u < n) v += t[u];
    }
  }
  const int sg = (count_below<L>(x, (int)h) ^ count_below<L>(x, (int)p) ^ (int)(h < p)) & 1;
  v *= sg ? (T)-1.0 : (T)1.0;
  return v;
}

// Single excitation x -> y evaluated by a whole warp (all lanes pass the same x, y): the two-electron terms
// of cpp_src/cpu/hamiltonian.cpp:52-72 are gathered one per lane and then added in the reference's order
// (occ_order: words ascending, bits descending) through shuffles -- the same additions in the same order as
// exc_element, without its chain of dependent loads.  Every lane returns the element.
template <int L, typename T>
__device__ __forceinline__ T single_element_warp(const Onv<L> &x, const Onv<L> &y, const T *__restrict__ h1e,
                                                 const T *__restrict__ h2e, int sorb, const unsigned char *occ_order, int n_occ) {
  const int lane = threadIdx.x & 31;
  Onv<L> cre, ann;
#pragma unroll
  for (int i = 0; i < L; ++i) {
    const u64 d = x.w[i] ^ y.w[i];
    cre.w[i] = d & x.w[i];
    ann.w[i] = d & y.w[i];
  }
  const u32 h = (u32)pop_highest<L>(cre), p = (u32)pop_highest<L>(ann);
  T v = (T)0.0;
  v += __ldg(h1e + (size_t)p * sorb + h);
  for (int j0 = 0; j0 < n_occ; j0 += 32) {
    const int j = j0 + lane;
    T t = (T)0.0;
    if (j < n_occ) {
      const u32 k = occ_order[j];
      t = two_body<T>(h2e, h, k, p, k);
    }
    const int cnt = min(32, n_occ - j0);
    for (int l = 0; l < cnt; ++l) v += __shfl_sync(0xffffffffu, t, l);
  }
  const int sg = (count_below<L>(x, (int)h) ^ count_below<L>(x, (int)p) ^ (int)(h < p)) & 1;
  v *= sg ? (T)-1.0 : (T)1.0;
  return v;
}

}  // namespace pynqs
