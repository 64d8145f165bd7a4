/*
 * pynqs_b200.h -- C ABI of the B200-native VMC local-energy library (libpynqs_b200.so).
 *
 * Drop-in boundary for the operator API of the reference's `libs/C_extension`
 * (stubs: libs/C_extension.pyi; pybind11 bindings: cpp_src/tensor/bind.cpp:317-391).
 * Every entry point takes plain pointers and sizes -- no torch / pybind types -- so the
 * reference-side binding is a ctypes stub (see INTEGRATION.md and pynqs_b200/C_extension.py).
 *
 * Conventions
 *  - All data pointers are DEVICE pointers on the current CUDA device unless stated otherwise;
 *    the caller sets the device (one process per GPU) and passes the stream to launch on.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - ONVs are `uint8[rows, 8*L]` contiguous, L = ceil(sorb/64), reinterpreted as little-endian
 *    `uint64[rows, L]`; spin orbital s = bit (s % 64) of word (s / 64); even = alpha, odd = beta
 *    (cpp_src/tensor/cpu_tensor.cpp:8-44, cpp_src/cpu/excitation.cpp:47-48).
 *  - `dtype`: PYNQS_F32 / PYNQS_F64 = element type of h1e, h2e and of the H output
 *    (the reference dispatches on h1e's dtype, cpp_src/tensor/cuda_tensor.cpp:186-199).
 *  - Every function returns 0 on success, a PYNQS_E* code otherwise; pynqs_last_error() gives
 *    the message of the calling thread's last failure.  Nothing is allocated for the caller;
 *    scratch comes from caller-provided workspaces whose sizes the *_bytes functions report.
 *  - Kernels are asynchronous w.r.t. the host; no call synchronises the device.
 */
#ifndef PYNQS_B200_H
#define PYNQS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYNQS_ABI_VERSION 1

enum { PYNQS_F32 = 0, PYNQS_F64 = 1 };

enum {
  PYNQS_OK = 0,
  PYNQS_EVALUE = 1,    /* bad argument  -> Python ValueError  (std::length_error in bind.cpp:282-291) */
  PYNQS_EOVERFLOW = 2, /* too many electrons/virtuals -> OverflowError (bind.cpp:292-301) */
  PYNQS_ECUDA = 3,     /* CUDA runtime / launch failure -> RuntimeError (cuda_handle_error.h:8-39) */
  PYNQS_EWORKSPACE = 4 /* workspace too small -> RuntimeError */
};

/* compile-time limits of this build; the reference exports the same three module attributes
 * (bind.cpp:382-384) but fixes L at compile time -- here L in {1,2,3} is dispatched at run time. */
#define PYNQS_MAX_SORB_LEN 3
#define PYNQS_MAX_SORB 192
#define PYNQS_MAX_NELE 120

int pynqs_abi_version(void);
const char *pynqs_last_error(void);

/* replaces check_sorb (bind.cpp:282-301): PYNQS_EVALUE if sorb not in (0, 192],
 * PYNQS_EOVERFLOW if nele > PYNQS_MAX_NELE.  The reference's per-L virtual-orbital cap
 * (MAX_NV = 40 L) is not needed by these kernels and is not enforced (SURVEY.md D3). */
int pynqs_check_sorb(int sorb, int nele);

/* replaces get_Num_SinglesDoubles (cpp_src/cpu/excitation.cpp:8-16); *nsd excludes the bra row. */
int pynqs_num_sd(int sorb, int noA, int noB, int64_t *nsd);

/* replaces tensor_to_onv (bind.cpp:9-22, cpu_tensor.cpp:8-44; kernel.cu:14-37):
 * states uint8[n, sorb] (value 1 = occupied) -> onv uint8[n, 8L]. */
int pynqs_tensor_to_onv(const uint8_t *states, int64_t n, int sorb, uint8_t *onv, void *stream);

/* replaces onv_to_tensor (bind.cpp:24-37, cpu_tensor.cpp:46-88; kernel.cu:39-64):
 * onv uint8[n, 8L] -> out dtype[n, sorb], +1 occupied / -1 empty. */
int pynqs_onv_to_tensor(const uint8_t *onv, int64_t n, int sorb, void *out, int dtype, void *stream);

/* replaces get_comb_tensor (bind.cpp:66-83, cuda_tensor.cpp:217-266; kernels K1+K2):
 * comb uint8[n, M, 8L], M = nsd + 1, row 0 = bra.  If states != NULL it receives the
 * flag_bit=True output double[n, M, sorb] of +-1 (cpu_tensor.cpp:186-190). */
int pynqs_comb(const uint8_t *bra, int64_t n, int sorb, int noA, int noB, uint8_t *comb, double *states,
               void *stream);

/* Gather-friendly internal copy of the packed h2e (same numbers, bit for bit), built once per
 * Hamiltonian into a caller-provided workspace of pynqs_prepared_bytes(sorb, dtype) bytes and
 * passed to pynqs_comb_hij_fused.  h2e is the packed array of cpp_src/cpu/hamiltonian.cpp:13-31. */
int pynqs_prepared_bytes(int sorb, int dtype, int64_t *bytes);
int pynqs_prepare_integrals(const void *h2e, int sorb, int dtype, void *prep_ws, int64_t prep_bytes, void *stream);

/* replaces get_comb_hij_fused (bind.cpp:239-250, cuda_tensor.cpp:162-215; kernels K1+K5):
 * comb uint8[n, M, 8L] and hmat dtype[n, M]; hmat[:,0] = <x|H|x> over the first `nele`
 * occupied orbitals (cpu_tensor.cpp:260-261).  prep_ws: workspace filled by
 * pynqs_prepare_integrals for the same (h2e, sorb, dtype), or NULL to read the packed arrays
 * directly (slower, identical results). */
int pynqs_comb_hij_fused(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n,
                         int sorb, int nele, int noA, int noB, uint8_t *comb, void *hmat, int dtype, void *stream);

/* replaces get_hij_torch (bind.cpp:39-64, cuda_tensor.cpp:97-141; kernels K3/K4):
 * ket3d != 0: ket uint8[n, m, 8L], out[i,j] = <bra_i|H|ket_ij>;
 * ket3d == 0: ket uint8[m, 8L],    out[i,j] = <bra_i|H|ket_j>.  More than a double excitation -> 0. */
int pynqs_hij(const uint8_t *bra, const uint8_t *ket, const void *h1e, const void *h2e, int64_t n, int64_t m,
              int ket3d, int sorb, int nele, void *out, int dtype, void *stream);

/* replaces wavefunction_lut (bind.cpp:220-237, cuda_tensor.cpp:436-487; kernel K6): classic
 * binary search (same probe sequence as cpu_tensor.cpp:589-640, so identical results even for
 * duplicate keys) of n queries in key uint8[N, 8L] sorted ascending as little-endian
 * multi-word integers.  idx int64[n] (-1 if absent), mask uint8/bool[n]. */
int pynqs_lut(const uint8_t *key, int64_t N, const uint8_t *onv, int64_t n, int L, int64_t *idx, uint8_t *mask,
              void *stream);

/* Hash index over a sorted UNIQUE key table -- an internal accelerator of pynqs_lut_hashed;
 * results are identical to pynqs_lut.  If the table holds duplicates the build records
 * it and the lookups fall back to the classic search on the device (no host round trip). */
int pynqs_hash_bytes(int64_t N, int L, int64_t *bytes);
int pynqs_hash_build(const uint8_t *key, int64_t N, int L, void *hash_ws, int64_t hash_bytes, void *stream);
int pynqs_lut_hashed(const uint8_t *key, int64_t N, const uint8_t *onv, int64_t n, int L, const void *hash_ws,
                     int64_t *idx, uint8_t *mask, void *stream);

/* String-grouped copies of a sorted key table (the keys bucketed by the hash of their beta string
 * and, a second time, of their alpha string) -- what pynqs_eloc_sample_space scans.  If the table
 * holds duplicates the build records it and the local-energy kernels take the classic search. */
int pynqs_group_bytes(int64_t N, int L, int64_t *bytes);
int pynqs_group_build(const uint8_t *key, int64_t N, int L, void *group_ws, int64_t group_bytes, void *stream);

/* ---- multi-GPU: pull collectives over NVLink peer memory (replace the all_gathers of vmc/sample.py:652-721) -----------
 * peer_ptrs: DEVICE array of `world` pointers, entry k = rank k's symmetric buffer as mapped into this process (e.g.
 * torch.distributed._symmetric_memory: handle.buffer_ptrs_dev).  The caller brackets the calls with barriers (data
 * published before, buffers free to overwrite after).
 *   pynqs_peer_gather     : out[k * bytes_per_rank + j] = peer k's byte src_offset + j, j < bytes_per_rank (multiples of 16);
 *   pynqs_peer_gather_rows: the peers' pieces (total elements split like split_length_idx: the first total % world pieces one
 *                           longer), piece k at src_offset of peer k; out[i] = element pos[i] of their concatenation.
 *                           elem_bytes 8 or 16. */
int pynqs_peer_gather(const void *const *peer_ptrs, int world, int64_t src_offset, int64_t bytes_per_rank, void *out, void *stream);
int pynqs_peer_gather_rows(const void *const *peer_ptrs, int world, int64_t src_offset, const uint32_t *pos, int64_t n, int64_t total,
                           int elem_bytes, void *out, void *stream);

/* Placement tier for integrals that do not stay in L2 on their own (reference: plain global loads,
 * cpp_src/cuda/hamiltonian.cu:9-34): set aside persisting L2 (up to the device maximum) and attach an access-policy window
 * over [ptr, ptr + bytes) to `stream`; kernels launched on it afterwards keep that range resident.  hit_ratio <= 0 picks
 * carve-out / window.  granted[0] = bytes set aside, granted[1] = window bytes (may be NULL).  ptr == NULL resets. */
int pynqs_l2_persist(const void *ptr, int64_t bytes, double hit_ratio, void *stream, int64_t *granted);

/* Where the pieces of a group workspace live (byte offsets), for callers that want to read the grouped copies -- e.g. to
 * hand each GPU the samples of a range of beta strings (pynqs_b200/distributed.py):
 * out[0] = log2(buckets); out[1 + g] = bucket starts uint32[2^log2 + 1]; out[3 + g] = keys uint64[N, L] in bucket order;
 * out[5 + g] = rows uint32[N] (row of the sorted table); out[7 + g] = folded other string uint32[N] (L = 1, else -1);
 * g = 0: bucketed by beta string, g = 1: by alpha string.  out[9] = position uint32[N] of every row of the sorted table in
 * the beta-grouped copy (the inverse of rows, g = 0).  out: int64[10]. */
int pynqs_group_layout(int64_t N, int L, int64_t *out);

/* Additive op: the whole sample-space local energy of vmc/energy/eloc.py:326-397 in one pass,
 * never materialising comb / Hmat:  for each sample x, psi0 = table value of x (0 if absent),
 *   eloc = sum over x' in {x} U SD(x) found in the table of (psi(x') / psi0) * <x|H|x'>.
 * psi: double[N] (psi_complex == 0) or interleaved complex128[N]; eloc / psi0 likewise [n].
 * scratch: pynqs_eloc_scratch_bytes(n, ...) bytes.  h1e/h2e are the packed float64 arrays.
 * group_ws must have been built by pynqs_group_build for exactly this key table. */
int pynqs_eloc_scratch_bytes(int64_t n, int sorb, int noA, int noB, int psi_complex, int64_t *bytes);
int pynqs_eloc_sample_space(const uint8_t *bra, int64_t n, const double *h1e, const double *h2e, int sorb,
                            int nele, int noA, int noB, const uint8_t *key, const void *psi, int psi_complex,
                            int64_t N, const void *group_ws, void *scratch, int64_t scratch_bytes, void *eloc,
                            void *psi0, void *stream);

/* Additive op: the sample-space Hamiltonian H[i, j] = <bra_i|H|key_j> (i < n, j < N) as a CSR matrix -- what the dense
 * get_hij_torch(bra, key) (pynqs_hij, ket3d == 0) gives, without its n x N array.  Row i holds exactly the table rows that
 * pynqs_eloc_sample_space sums over for bra_i: bra_i itself (if it is in the table) and its single and double excitations
 * that are in the table; entries are structural (an element equal to 0.0 is stored), the columns of a row strictly
 * ascending, the values bit-identical to pynqs_hij.  A table with duplicate keys gives the column the classic binary
 * search lands on.  Same count / emit protocol as pynqs_reduce_count / _emit:
 *   pynqs_hamiltonian_count: offsets int64[n + 1] = exclusive prefix of the row lengths, offsets[n] = nnz;
 *   pynqs_hamiltonian_emit : col int64[nnz] and val double[nnz] of every row at those offsets (nnz = offsets[n], read by
 *                            the caller).
 * key / group_ws as for pynqs_eloc_sample_space.  scratch: pynqs_hamiltonian_scratch_bytes(n, nnz, ...) bytes -- size it
 * for nnz = 0 before the count call and for the real nnz before the emit call. */
int pynqs_hamiltonian_scratch_bytes(int64_t n, int64_t nnz, int sorb, int noA, int noB, int64_t *bytes);
int pynqs_hamiltonian_count(const uint8_t *bra, int64_t n, int sorb, int noA, int noB, const uint8_t *key, int64_t N,
                            const void *group_ws, void *scratch, int64_t scratch_bytes, int64_t *offsets, void *stream);
int pynqs_hamiltonian_emit(const uint8_t *bra, int64_t n, const double *h1e, const double *h2e, int sorb, int nele, int noA,
                           int noB, const uint8_t *key, int64_t N, const void *group_ws, void *scratch, int64_t scratch_bytes,
                           const int64_t *offsets, int64_t nnz, int64_t *col, double *val, void *stream);

/* Additive op: Y = H X for a CSR matrix H laid out as pynqs_hamiltonian_emit writes it (crow int64[n + 1], col int64[nnz]
 * with columns < N, val double[nnz]; nnz = crow[n] is read on the device only) and row-major blocks X double[N, k] (row
 * stride ldx) and Y double[n, k] (row stride ldy), 1 <= k <= 8: Y[i, c] = sum over the entries p of row i of
 * val[p] * X[col[p], c].  Wider blocks go through in column slices (X + c0, Y + c0, same ld).  Deterministic: each Y[i, c]
 * is summed in an order fixed by the length of row i, so two calls give identical bits.  Empty rows give 0.  PYNQS_EVALUE,
 * before anything touches the device, for n < 0, N < 0, k outside [1, 8], ldx < k, ldy < k, or a NULL crow / Y (n > 0) or
 * col / val / X (n > 0 and N > 0).  n == 0 launches nothing. */
int pynqs_csr_spmm(const int64_t *crow, const int64_t *col, const double *val, int64_t n, int64_t N, const double *X, int64_t ldx, int k,
                   double *Y, int64_t ldy, void *stream);

/* Additive op: Y = S^2 X over the sorted key table, Y[i, c] = sum over j < N of <bra_i|S^2|key_j> X[j, c], for row-major
 * blocks X double[N, k] (row stride ldx) and Y double[n, k] (row stride ldy), 1 <= k <= 8; wider blocks go through in column
 * slices as for pynqs_csr_spmm.  Orbital i has alpha at bit 2i and beta at bit 2i + 1.  With A / B the alpha-only / beta-only
 * orbitals of x and Sz = (n_alpha - n_beta) / 2, taken from x's own bits:  <x|S^2|x> = |B| + Sz (Sz + 1), counted when x is
 * in the table;  <x|S^2|x ^ (3 << 2p) ^ (3 << 2q)> = +1 for p in A, q in B, counted when that spin exchange is in the table.
 * A table with duplicate keys gives the column the classic binary search lands on.  key / group_ws as for
 * pynqs_eloc_sample_space (N < 2^31).  Deterministic: row i is summed in one fixed order (the diagonal, then the partners in
 * ascending (p, q)); no scratch, no host synchronisation.  PYNQS_EVALUE, before anything touches the device, for an odd sorb
 * or one outside (0, PYNQS_MAX_SORB] (the ONV width is (sorb - 1) / 64 + 1 words), n < 0, N < 0 or >= 2^31, k outside
 * [1, 8], ldx < k, ldy < k, or a NULL bra / Y (n > 0) or key / group_ws / X (n > 0 and N > 0).  n == 0 does nothing;
 * N == 0 launches no kernel and clears Y. */
int pynqs_spin_square_apply(const uint8_t *bra, int64_t n, int sorb, const uint8_t *key, int64_t N, const void *group_ws,
                            const double *X, int64_t ldx, int k, double *Y, int64_t ldy, void *stream);

/* Additive op: the off-diagonal part of the one- and two-body reduced density matrices of c over the sorted key table
 * (N keys of (sorb - 1) / 64 + 1 words), summed over the entries (i, j != i) of a square CSR structure crow int64 [N + 1],
 * col int64 [nnz] -- the structure of pynqs_hamiltonian_emit with bra = key, whose entries are exactly the table pairs
 * connected by a single or double excitation.  c: N values, double (c_complex = 0) or interleaved (re, im) doubles
 * (c_complex = 1).  Orbital p has alpha at bit 2p and beta at bit 2p + 1, norb = sorb / 2; the sign counts the occupied
 * bits below each operator's bit.  Not normalised, and without the diagonal i == j, which the caller adds (|c_i|^2 times
 * occupation products).  Outputs, in c's element type, row-major, overwritten (zero where no off-diagonal pair lands):
 *   dm1 [2][norb][norb]            dm1[s][p][q] = sum conj(c_i) c_j <key_i| a+_{q s} a_{p s} |key_j>, s = alpha, beta;
 *   dm2 [3][norb][norb][norb][norb] (aa, ab, bb), or NULL for dm1 alone:
 *                                  dm2[st][p][q][r][s] = sum conj(c_i) c_j <key_i| a+_{p s} a+_{r t} a_{s t} a_{q s} |key_j>
 * (PySCF's make_rdm12s layout).  Entries that are not a single or double excitation, or change the spin, add nothing.
 * Deterministic (identical bits on every call, no float atomics): one record per CSR entry, a stable radix sort by output
 * bin, one warp per bin summing in the bin's order.  No host synchronisation.  scratch: pynqs_rdm_scratch_bytes(N, nnz,
 * sorb) = 24 nnz + 4 nnz (records, double-buffered, and run starts) + 2 nnz + 4 MiB (sort / run-length / scan
 * temporaries) + alignment; it does not depend on c's type or on dm2.  PYNQS_EVALUE, before anything touches the device,
 * for an odd sorb or one outside (0, PYNQS_MAX_SORB], N or nnz < 0 or >= 2^31, c_complex not 0 / 1, a NULL bytes / dm1,
 * crow / key / c (N > 0) or col / scratch (nnz > 0).  A table with duplicate keys is the caller's to refuse. */
int pynqs_rdm_scratch_bytes(int64_t N, int64_t nnz, int sorb, int64_t *bytes);
int pynqs_rdm_offdiag(const int64_t *crow, const int64_t *col, const uint8_t *key, int64_t N, int64_t nnz, int sorb, const double *c,
                      int c_complex, void *scratch, int64_t scratch_bytes, double *dm1, double *dm2, void *stream);

/* Additive op: the Epstein-Nesbet second-order correction of real states C over the sorted key table (N unique keys of one
 * (noA, noB) sector, (sorb - 1) / 64 + 1 words; group_ws built by pynqs_group_build for it):
 *   acc[r] += sum over the externals a of (sum over i of <key_i|H|a> C[i, r])^2 / (E[r] - <a|H|a>)
 * where the externals are the distinct single and double excitations of the table rows (the rows of get_comb_tensor) that
 * are not in the table, <key_i|H|a> has the bits of pynqs_comb_hij_fused and <a|H|a> those of pynqs_hij(a, a).  Not
 * normalised: the caller divides by sum_i C[i, r]^2.  The externals are split into 2^log2_parts partitions by a hash of the
 * determinant; one pass handles partition `part` completely, in four calls on one scratch buffer:
 *   pynqs_pt2_count : offsets int64[N + 1] = exclusive prefix of the rows' kept (row, external) pairs, offsets[N] = pairs;
 *   pynqs_pt2_emit  : per pair, the external and (<key_i|H|a>, i), rows ascending, each row's excitations ascending;
 *   pynqs_pt2_sort  : the pairs sorted by external, stable (pynqs_sort_table's sort);
 *   pynqs_pt2_reduce: acc[r] += the pass's sum (r < k <= 8; C double[N, k] with row stride ldc, E double[k]; wider blocks in
 *                     column slices), externals[0] += the pass's externals (externals may be NULL).
 * scratch: pynqs_pt2_scratch_bytes(N, pairs, sorb) bytes -- size it for pairs = 0 for the count call and for the pass's
 * pairs (offsets[N], read by the caller) for the other three.  Deterministic (no float atomics; each numerator summed in
 * ascending (row, excitation) order, the externals' terms in an order fixed by the sorted pairs and a fixed grid): two calls
 * give identical bits; adding the passes' sums in pass order makes the whole sum deterministic for a given log2_parts.  No
 * host synchronisation.  PYNQS_EVALUE, before anything touches the device, for an odd sorb or one outside
 * (0, PYNQS_MAX_SORB], N outside (0, 2^31), pairs outside [0, 2^31), a bad sector, part outside [0, 2^log2_parts),
 * log2_parts outside [0, 31], nele outside [0, sorb], k outside [1, 8], ldc < k, or a NULL pointer other than externals.
 * The table must not hold duplicate keys (the caller's to refuse).  pairs == 0 makes emit, sort and reduce do nothing. */
int pynqs_pt2_scratch_bytes(int64_t N, int64_t pairs, int sorb, int64_t *bytes);
int pynqs_pt2_count(const uint8_t *key, int64_t N, int sorb, int noA, int noB, const void *group_ws, int part, int log2_parts, void *scratch,
                    int64_t scratch_bytes, int64_t *offsets, void *stream);
int pynqs_pt2_emit(const uint8_t *key, int64_t N, const double *h1e, const void *prep_ws, int sorb, int noA, int noB, const void *group_ws,
                   int part, int log2_parts, const int64_t *offsets, int64_t pairs, void *scratch, int64_t scratch_bytes, void *stream);
int pynqs_pt2_sort(int64_t N, int64_t pairs, int sorb, void *scratch, int64_t scratch_bytes, void *stream);
int pynqs_pt2_reduce(int64_t N, int64_t pairs, const double *h1e, const double *h2e, int sorb, int nele, const double *C, int64_t ldc, int k,
                     const double *E, void *scratch, int64_t scratch_bytes, double *acc, int64_t *externals, void *stream);

/* ---- REDUCE method (vmc/energy/eloc.py:257-297, additive) -----------------------------------------
 * The reference materialises comb [n, M, 8L] and Hmat [n, M] and keeps torch.where(|Hmat| >= eps).  These
 * entry points return the kept rows only, in the same (ascending flat index s * M + m) order:
 *   pynqs_reduce_count: offsets int64[n + 1] = exclusive prefix of the per-sample counts, offsets[n] = K;
 *   pynqs_reduce_emit : x uint8[K, 8L] (determinants), hij T[K] (values, bit-identical to get_comb_hij_fused),
 *                       idx int64[K] (flat indices) written at those offsets.
 * prep_ws (pynqs_prepare_integrals) is required.  scratch: pynqs_reduce_scratch_bytes(n) bytes.
 *   pynqs_reduce_eloc : eloc[s] = sum over kept rows of sample s of (psi_k / psi0) * hij_k, psi0 = psi of row 0
 *                       (0 when row 0 was not kept); psi double[K] or interleaved complex128[K], hij double[K]. */
int64_t pynqs_reduce_scratch_bytes(int64_t n);
int pynqs_reduce_count(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb, int nele,
                       int noA, int noB, double eps, int dtype, void *scratch, int64_t scratch_bytes, int64_t *offsets,
                       void *stream);
int pynqs_reduce_emit(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb, int nele,
                      int noA, int noB, double eps, int dtype, void *scratch, int64_t scratch_bytes, const int64_t *offsets,
                      uint8_t *x, void *hij, int64_t *idx, void *stream);
int pynqs_reduce_eloc(const void *psi, int psi_complex, const double *hij, const int64_t *idx, const int64_t *offsets, int64_t n,
                      int64_t M, void *eloc, void *psi0, void *stream);

/* Stochastic / semi-stochastic branch of the REDUCE method (vmc/energy/eloc.py:257-283, eps_sample > 0; what every
 * shipped input selects, main.py:149-159): per sample, eps_sample draws from p(m) ~ |H_m| over the rows with |H_m| < eps
 * (all rows when eps == 0); a drawn row's element becomes (count / eps_sample) * H_m / p(m) = sign(H_m) * S * count /
 * eps_sample with S the sample's sum of sub-eps magnitudes; rows with |H_m| >= eps (eps > 0) are kept exactly.  eps is
 * compared in the integrals' dtype (as torch compares Hmat, and as pynqs_reduce_count does): under float32 the threshold
 * is (float)eps.  A sample with S = 0 (every row kept or exactly zero) has nothing drawn; the generator never draws a row
 * with H_m == 0.  Same count / emit protocol and outputs as pynqs_reduce_count / _emit; per sample the kept rows come
 * first (ascending m), then the drawn rows (ascending m).  No [n, M] array and no [n, eps_sample] array is materialised.
 * Draws: Philox4x32-10 keyed by `seed` (reproducible; not torch.multinomial's stream), or -- draws != NULL -- the caller's
 * row indices int64[n, eps_sample] (what torch.multinomial returned), which makes the result a deterministic function of
 * the inputs.  eps_sample <= 8192.  scratch: pynqs_reduce_sample_scratch_bytes(n) bytes, the same buffer for both calls. */
int64_t pynqs_reduce_sample_scratch_bytes(int64_t n);
int pynqs_reduce_sample_count(const uint8_t *bra, const void *h1e, const void *h2e, int64_t n, int sorb, int nele, int noA, int noB,
                              double eps, int eps_sample, uint64_t seed, const int64_t *draws, int dtype, void *scratch,
                              int64_t scratch_bytes, int64_t *offsets, void *stream);
int pynqs_reduce_sample_emit(const uint8_t *bra, const void *h1e, const void *h2e, int64_t n, int sorb, int nele, int noA, int noB,
                             double eps, int eps_sample, uint64_t seed, const int64_t *draws, int dtype, void *scratch,
                             int64_t scratch_bytes, const int64_t *offsets, uint8_t *x, void *hij, int64_t *idx, void *stream);

/* ---- unique-sample table: sort (utils/public_function.py:626-689, 754-788) ----------------------
 * Stable ascending sort of N keys (uint64[N, L] little-endian multi-word integers, the order of the
 * reference's torch_sort_onv) together with their psi values (psi_bytes = 8 or 16 per row; psi may
 * be NULL).  key_out / psi_out receive the sorted table, perm_out (int64[N], may be NULL) the source
 * row of every sorted row.  sorb > 0 promises that bits >= sorb of every key are zero (then only the
 * significant bits are sorted); sorb <= 0 sorts on all 64 L bits.  ws: pynqs_sort_bytes(N) bytes. */
int64_t pynqs_sort_bytes(int64_t N);
int pynqs_sort_table(const uint8_t *key, const void *psi, int64_t N, int L, int sorb, int psi_bytes, uint8_t *key_out,
                     void *psi_out, int64_t *perm_out, void *ws, int64_t ws_bytes, void *stream);

/* ---- index glue of the lookup (additive) ------------------------------------------------------------------------
 * WavefunctionLUT.lookup (utils/public_function.py:817-838) = wavefunction_lut + arange + two boolean-mask selections + a
 * gather; pynqs_lookup_count / _emit produce its three results from (idx, mask) in two passes:
 *   count: *n_hit (device, uint64) = number of set mask bytes;
 *   emit : hit_pos int64[n_hit] (ascending positions with mask set), miss_pos int64[n - n_hit] (ascending positions
 *          without), value[n_hit] = value_table[idx[hit_pos]] (value_bytes = 8 or 16 per element).
 * Func (vmc/energy/flip.py:44-61) = torch.unique(rows, dim=0, return_inverse=True) of the LUT misses;
 * pynqs_unique_count / _emit take the rows already sorted by pynqs_sort_table (sorted_key, perm):
 *   count: *n_unique (device, uint64);   emit: unique uint8[n_unique, 8L] (ascending), inverse int64[n] with
 *          unique[inverse[i]] == row i of the unsorted input.
 * scratch: pynqs_compact_scratch_bytes(n) bytes, the same buffer for the count and the emit call. */
int64_t pynqs_compact_scratch_bytes(int64_t n);
int pynqs_lookup_count(const uint8_t *mask, int64_t n, void *scratch, int64_t scratch_bytes, uint64_t *n_hit, void *stream);
int pynqs_lookup_emit(const uint8_t *mask, const int64_t *idx, int64_t n, const void *value_table, int value_bytes, void *scratch,
                      int64_t *hit_pos, int64_t *miss_pos, void *value, void *stream);
int pynqs_unique_count(const uint8_t *sorted_key, int64_t n, int L, void *scratch, int64_t scratch_bytes, uint64_t *n_unique, void *stream);
int pynqs_unique_emit(const uint8_t *sorted_key, const int64_t *perm, int64_t n, int L, void *scratch, uint8_t *unique, int64_t *inverse,
                      void *stream);

/* merge_rank_sample (libs/C_extension.pyi:256-279; cpu_tensor.cpp:537-556): out int64[length] = 0, then
 * out[idx[i]] += counts[i] for i < n (int64 atomics; indices outside [0, length) are ignored). */
int pynqs_merge_rank_sample(const int64_t *idx, const int64_t *counts, int64_t n, int64_t length, int64_t *out, void *stream);

/* ---- energy statistics (utils/stats/dist_stats.py:18-79) -----------------------------------------
 * out[7] = { sum w, sum w Re d, sum w Im d, sum w |d|^2, Re c, Im c, n } with d = eloc - c, c = eloc[0];
 * eloc: double[n] or interleaved complex128[n] (eloc_complex).  weight_kind 0: w = weight (double[n]);
 * 1: w = weight^2 (real amplitudes, double[n]); 2: w = |weight|^2 (complex128[n]).  Deterministic.
 * scratch: pynqs_moments_scratch_bytes() bytes, ZEROED once by the caller before its first use. */
int64_t pynqs_moments_scratch_bytes(void);
int pynqs_weighted_moments(const void *eloc, int eloc_complex, const void *weight, int weight_kind, int64_t n, void *scratch,
                           double *out, void *stream);

/* Test / experiment knobs of the one-pass local energy (process-wide, not thread-safe; production code never
 * calls this).  name: "scan_threads" (0 = automatic, 64, 128, 256), "search_factor" (bucket-size factor above which
 * a group is searched instead of walked, default 64), "full_keys" (1: one-word ONVs take the full-key route of
 * multi-word ONVs), "block_enable" (0: per-sample kernel only), "block_min_samples" (calls with fewer samples use the
 * per-sample kernel only, default 4096), "block_min_group" (samples sharing a beta string needed for a tile of the
 * block kernel, default 8), "eval_tiles" (evaluation kernel: 0 one warp per sample, 1 = default: 32 samples per warp for
 * large calls, 2: for every call), "block_parts" (block kernel: 0 = by the size of the call, 1 / 2 / 4: parts the groups
 * of a tile are split into), "lut_pipeline" (wavefunction_lut on one-word ONVs: 1 = default, four consecutive queries per
 * thread; 0: one query per thread), "sort_chunk" (pynqs_hamiltonian_emit: 0 = default, rows sorted in as few calls as
 * 31-bit offsets allow; else the calls take the rows starting in windows of this many entries).  name == NULL restores every default.  The scratch size of pynqs_eloc_scratch_bytes
 * depends on the knobs: set them before sizing the scratch. */
int pynqs_set_tuning(const char *name, int64_t value);

/* number of kernel launches issued by this library in this process (bench.py's gpu_launches). */
int64_t pynqs_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PYNQS_B200_H */
