// enum_rows.cuh -- the rows of one excitation class of a sample, from the per-sample excitation tables in shared
// memory (tables.cuh): what enumerate_kernel and reduce_kernel (enumerate.cu) and the PT2 kernels (pt2.cu) enumerate.
#pragma once
#include "prepare.cuh"
#include "tables.cuh"

namespace pynqs {

constexpr int kEnumThreads = 256;

// ---- table entries of the enumeration kernel: excitation mask (L = 1) + HitInfo (tables.cuh) ------
template <int L>
struct __align__(8) EnumEntry {
  u32 off, cmp;
};
#define PYNQS_WIDE_ENTRIES 1  // (8-byte entries + recomputed masks measured slower: 1.04 vs 0.89 ms)
#ifdef PYNQS_WIDE_ENTRIES  // one-word ONVs: the excitation mask stored next to the HitInfo (16-byte entries, one LDS.128)
template <>
struct __align__(16) EnumEntry<1> {
  u64 mask;
  u32 off, cmp;
};
#endif

template <int L>
__device__ __forceinline__ EnumEntry<L> load_entry(const EnumEntry<L> *p) {
  const uint2 v = *reinterpret_cast<const uint2 *>(p);
  EnumEntry<L> e;
  e.off = v.x;
  e.cmp = v.y;
  return e;
}
#ifdef PYNQS_WIDE_ENTRIES
template <>
__device__ __forceinline__ EnumEntry<1> load_entry<1>(const EnumEntry<1> *p) {
  // one LDS.128 (the compiler splits a plain 16-byte shared load into two LDS.64, which doubles
  // the shared-memory wavefronts of the stride-16 access pattern)
  uint4 v;
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  EnumEntry<1> e;
  e.mask = (u64)v.x | ((u64)v.y << 32);
  e.off = v.z;
  e.cmp = v.w;
  return e;
}
#endif

template <int L>
__device__ __forceinline__ void set_mask(EnumEntry<L> &, u32, u32) {}
#ifdef PYNQS_WIDE_ENTRIES
template <>
__device__ __forceinline__ void set_mask<1>(EnumEntry<1> &e, u32 a, u32 b) {
  e.mask = (1ull << a) | (1ull << b);
}
#endif

template <int L>
__device__ __forceinline__ Onv<L> entry_apply(const Onv<L> &x, const EnumEntry<L> &e) {
  Onv<L> y = x;
  flip_bit<L>(y, (int)(e.cmp & 0xffu));
  flip_bit<L>(y, (int)((e.cmp >> 16) & 0xffu));
  return y;
}
#ifdef PYNQS_WIDE_ENTRIES
template <>
__device__ __forceinline__ Onv<1> entry_apply<1>(const Onv<1> &x, const EnumEntry<1> &e) {
  Onv<1> y;
  y.w[0] = x.w[0] ^ e.mask;
  return y;
}
#endif

template <int L>
__device__ __forceinline__ void store_row_vec(u64 *dst, const Onv<L> &r) {
  if (L == 2) {
    *reinterpret_cast<ulonglong2 *>(dst) = make_ulonglong2(r.w[0], r.w[L - 1]);  // 16-byte rows: one vector store
  } else {
#pragma unroll
    for (int i = 0; i < L; ++i) dst[i] = r.w[i];
  }
}

constexpr int kRowsPerThread = 4;  // independent rows (and integral gathers) in flight per thread

// Rows [lo, hi) of one excitation class (CLS: 0/1 single a/b, 2/3 double aa/bb, 4 double ab);
// row m holds excitation r = m - 1.  A warp takes chunks of 32 * ROWS consecutive rows; lane l
// owns rows chunk + l + 32 j, so each store instruction of the warp covers 32 consecutive rows
// (256 contiguous bytes of comb at L = 1 and of Hmat): coalesced, every byte written once.
// The ROWS rows  c + lane + 32 j  (j < ROWS) of one excitation class (CLS: 0/1 single a/b, 2/3 double aa/bb,
// 4 double ab; row m holds excitation r = m - 1): determinant, |value| and sign word of each; rows >= hi are
// left as (x, 0, 0).
template <int L, typename T, bool WITH_H, int CLS, int ROWS>
__device__ __forceinline__ void class_rows(const Onv<L> &x, const EnumEntry<L> *__restrict__ tab, const TableOffsets &to,
                                           const ExcGeom &g, const OrbLists &lists, const T *__restrict__ h1e,
                                           const PrepView<T> &prep, int c, int hi, Onv<L> (&row)[ROWS], T (&val)[ROWS],
                                           u32 (&sgn)[ROWS]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < ROWS; ++j) {
    const int m = c + lane + 32 * j;
    row[j] = x;
    val[j] = (T)0.0;
    sgn[j] = 0;
    if (m < hi) {
      const u32 r = (u32)(m - 1);
      if (CLS <= 1) {
        const EnumEntry<L> e1 = load_entry<L>(tab + (CLS == 0 ? to.sa + (int)r : to.sb + (int)(r - g.d0)));
        row[j] = entry_apply<L>(x, e1);
        if (WITH_H) {
          // single h -> p: h1e(h,p) + sum over occupied k, in the reference's order, of <hk||pk>
          // SA packs hA | pA << 16, SB packs pB | hB << 16
          const u32 h = CLS == 0 ? (e1.cmp & 0xffu) : (e1.cmp >> 16), p = CLS == 0 ? (e1.cmp >> 16) : (e1.cmp & 0xffu);
          // (32-bit element offsets: the table has sorb * 2 * na^2 <= 3.6e6 entries; the occupied orbitals are read four
          //  at a time as one packed word of the order list; eight gathers in flight, added in order)
          const u32 na = (u32)prep.na;
          const u32 kstride = 2u * na * na;
          const int n_occ = lists.n_occ;
          const u32 *occ4 = reinterpret_cast<const u32 *>(lists.occ_order);
          T v = (T)0.0;
          v += __ldg(h1e + (size_t)p * g.sorb + h);
          const u32 base = ((h & 1u) * na + (p >> 1)) * na + (h >> 1);
          int q = 0;
          for (; q + 8 <= n_occ; q += 8) {
            const u32 w0 = occ4[q >> 2], w1 = occ4[(q >> 2) + 1];
            T t[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) t[i] = __ldg(prep.s + (base + kstride * (((i < 4 ? w0 : w1) >> (8 * (i & 3))) & 0xffu)));
#pragma unroll
            for (int i = 0; i < 8; ++i) v += t[i];
          }
          for (; q < n_occ; ++q) v += __ldg(prep.s + (base + kstride * (u32)lists.occ_order[q]));
          val[j] = v;
          sgn[j] = e1.off;  // bit 31 = the single's sign
        }
      } else {
        int t1, t2;
        if (CLS == 4) {
          const u32 q = r - (u32)g.d3;
          const u32 jb = fdiv(q, g.by_sA);
          t1 = to.sa + (int)(q - jb * g.sA);
          t2 = to.sb + (int)jb;
        } else if (CLS == 2) {
          t1 = to.hpa + (int)(r - fdiv(r, g.by_noAA) * g.noAA);  // r % noAA with the GLOBAL r (quirk Q1)
          t2 = to.ppa + (int)fdiv(r - (u32)g.d1, g.by_noAA);
        } else {
          t1 = to.hpb + (int)(r - fdiv(r, g.by_noBB) * g.noBB);
          t2 = to.ppb + (int)fdiv(r - (u32)g.d2, g.by_noBB);
        }
        const EnumEntry<L> e1 = load_entry<L>(tab + t1);
        const EnumEntry<L> e2 = load_entry<L>(tab + t2);
        row[j] = entry_apply<L>(entry_apply<L>(x, e1), e2);
        if (WITH_H) {
          const HitInfo i1 = {e1.off, e1.cmp}, i2 = {e2.off, e2.cmp};
          const T *tbl = CLS == 4 ? prep.ab : (CLS == 2 ? prep.aa : prep.bb);
          val[j] = __ldg(tbl + ((i1.off + i2.off) & 0x7fffffffu));
          sgn[j] = double_sign_word(CLS == 4, i1, i2);
        }
      }
    }
  }
}

}  // namespace pynqs
