// spin.cu -- Y = S^2 X over the sorted key table: Y[i, :] = sum over j of <bra_i|S^2|key_j> X[j, :].
//
// With orbital i's alpha at bit 2i and beta at bit 2i + 1, and the fermionic sign of get_hij_torch (an operator on bit b
// counts the occupied bits below b), S^2 = S-S+ + Sz(Sz + 1) has a closed form on a determinant x.  Let A be x's alpha-only
// orbitals, B its beta-only orbitals, Sz = (n_alpha - n_beta) / 2:
//   diagonal     <x|S^2|x> = |B| + Sz(Sz + 1);
//   off-diagonal x connects to the |A| |B| spin exchanges x_pq = x ^ (3 << 2p) ^ (3 << 2q), p in A, q in B (p and q keep
//                their occupation and swap their spins), each with the element +1.
// The kernel takes Sz from the row's own bits, so one call handles a table that mixes (n_alpha, n_beta) sectors.
//
// One thread per row.  A row has |A| |B| partners: at most 4 on the Fe2S2 CI space, at most 25 on a 15a15b sample of 20
// orbitals, against 7 876 connected determinants for H.  Each partner is one lookup in the beta-grouped table copy (hash of
// its beta string -> bucket -> binary search among the bucket's keys -> table row), the same lookup eloc_scan.cu's search route
// does.  So a warp's lanes stay busy on a few lookups each, and the row is summed in one thread in a fixed order: the
// diagonal, then the partners in ascending (p, q) -- p outer, q inner.  No atomics, no scratch, no host synchronisation: two
// calls give identical bits.
//
// Tables with duplicate keys (GroupHeader::has_dup) take the classic binary search over the sorted keys instead, so the
// column is the row that search lands on, as in lut.cu and hamiltonian.cu.
#include "gindex.cuh"
#include "lut.cuh"

namespace pynqs {

constexpr int kSpinThreads = 128;  // 8 CTAs per SM at least: the 64-register cap leaves every (L, K) variant free of spills
constexpr long long kSpinBlocksCap = 148LL * 16 * 8;  // a grid-stride loop past ~2.4 * 10^6 rows

template <int L, int K>
__global__ void __launch_bounds__(kSpinThreads, 8)
spin_square_kernel(const u64 *__restrict__ bra, long long n, const u64 *__restrict__ key, long long N, GroupView gv,
                   const double *__restrict__ X, long long ldx, double *__restrict__ Y, long long ldy) {
  const bool dup = __ldg(&gv.hdr->has_dup) != 0u;
  for (long long i = (long long)blockIdx.x * kSpinThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kSpinThreads) {
    const Onv<L> x = load_onv<L>(bra + i * L);
    u64 A[L], B[L];  // alpha-only / beta-only orbitals, both on the even (alpha) bit of the orbital
    int na = 0, nb = 0, nB = 0;
#pragma unroll
    for (int w = 0; w < L; ++w) {
      const u64 a = x.w[w] & kEven, b = (x.w[w] >> 1) & kEven;
      A[w] = a & ~b;
      B[w] = b & ~a;
      na += __popcll(a);
      nb += __popcll(b);
      nB += __popcll(B[w]);
    }
    const int sz2 = na - nb;  // 2 Sz; Sz(Sz + 1) = sz2 (sz2 + 2) / 4 is exact in double
    const double diag = (double)nB + 0.25 * (double)(sz2 * (sz2 + 2));
    double acc[K];
#pragma unroll
    for (int c = 0; c < K; ++c) acc[c] = 0.0;
    const long long self = spin_find<L>(key, N, gv, dup, x);
    if (self >= 0) {
#pragma unroll
      for (int c = 0; c < K; ++c) acc[c] = diag * __ldg(X + self * ldx + c);
    }
#pragma unroll
    for (int wp = 0; wp < L; ++wp) {
      for (u64 ap = A[wp]; ap; ap &= ap - 1) {
        const u64 fp = 3ull << (__ffsll((long long)ap) - 1);
#pragma unroll
        for (int wq = 0; wq < L; ++wq) {
          for (u64 bq = B[wq]; bq; bq &= bq - 1) {
            Onv<L> y = x;
            y.w[wp] ^= fp;
            y.w[wq] ^= 3ull << (__ffsll((long long)bq) - 1);
            const long long j = spin_find<L>(key, N, gv, dup, y);
            if (j >= 0) {
#pragma unroll
              for (int c = 0; c < K; ++c) acc[c] += __ldg(X + j * ldx + c);
            }
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < K; ++c) Y[i * ldy + c] = acc[c];
  }
}

template <int L, int K>
static void launch_lk(const u64 *bra, long long n, const u64 *key, long long N, const GroupView &gv, const double *X, long long ldx,
                      double *Y, long long ldy, cudaStream_t st) {
  const long long blocks = (n + kSpinThreads - 1) / kSpinThreads;
  spin_square_kernel<L, K><<<(unsigned)(blocks < kSpinBlocksCap ? blocks : kSpinBlocksCap), kSpinThreads, 0, st>>>(bra, n, key, N, gv, X,
                                                                                                                  ldx, Y, ldy);
}

template <int L>
static int launch_l(const u64 *bra, long long n, const u64 *key, long long N, const GroupView &gv, const double *X, long long ldx, int k,
                    double *Y, long long ldy, cudaStream_t st) {
  switch (k) {
    case 1: launch_lk<L, 1>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 2: launch_lk<L, 2>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 3: launch_lk<L, 3>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 4: launch_lk<L, 4>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 5: launch_lk<L, 5>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 6: launch_lk<L, 6>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 7: launch_lk<L, 7>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    case 8: launch_lk<L, 8>(bra, n, key, N, gv, X, ldx, Y, ldy, st); break;
    default: set_error("spin_square_apply: k = %d not in [1, 8]", k); return 1;
  }
  count_launch();
  return check_launch("spin_square_kernel");
}

// n > 0, N > 0; arguments checked by pynqs_spin_square_apply
int launch_spin_square(const u64 *bra, long long n, int L, const u64 *key, long long N, const void *group_ws, const double *X, long long ldx,
                       int k, double *Y, long long ldy, cudaStream_t st) {
  const GroupView gv = group_view(group_ws, N, L);
  switch (L) {
    case 1: return launch_l<1>(bra, n, key, N, gv, X, ldx, k, Y, ldy, st);
    case 2: return launch_l<2>(bra, n, key, N, gv, X, ldx, k, Y, ldy, st);
    case 3: return launch_l<3>(bra, n, key, N, gv, X, ldx, k, Y, ldy, st);
    default: set_error("spin_square_apply: unsupported ONV length L = %d", L); return 1;
  }
}

}  // namespace pynqs
