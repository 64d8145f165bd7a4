// abi.cu -- extern "C" entry points of libpynqs_b200.so (declared in include/pynqs_b200.h).
// Argument validation mirrors the reference binding layer (cpp_src/tensor/bind.cpp) with its
// asserts / exit(1) turned into status codes.
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "../../include/pynqs_b200.h"
#include <cstring>

#include "eloc.cuh"

namespace pynqs {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
    return PYNQS_ECUDA;
  }
  return 0;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// launchers implemented in the other translation units
int launch_comb(const u64 *, u64 *, long long, const ExcGeom &, cudaStream_t);
int launch_comb_hij_f64(const u64 *, const double *, const double *, const void *, u64 *, double *, long long, const ExcGeom &,
                        cudaStream_t);
int launch_comb_hij_f32(const u64 *, const float *, const float *, const void *, u64 *, float *, long long, const ExcGeom &,
                        cudaStream_t);
long long prepared_bytes(int, int);
int launch_prepare(const void *, int, int, void *, long long, cudaStream_t);
int launch_states(const u64 *, double *, long long, int, cudaStream_t);
template <typename T>
int launch_hij(const u64 *, const u64 *, const T *, const T *, T *, long long, long long, int, int, int, cudaStream_t);
int launch_lut_classic(const u64 *, long long, const u64 *, long long, int, long long *, unsigned char *, cudaStream_t);
long long hash_workspace_bytes(long long);
int launch_hash_build(const u64 *, long long, int, void *, long long, cudaStream_t);
int launch_lut_hashed(const u64 *, long long, const u64 *, long long, int, const void *, long long *, unsigned char *, cudaStream_t);
long long eloc_scratch_bytes(long long, const ExcGeom &);
long long group_workspace_bytes(long long, int);
int launch_group_build(const u64 *, long long, int, void *, long long, cudaStream_t);
int launch_eloc(const u64 *, long long, const double *, const double *, const u64 *, const double *, int, long long,
                const void *, void *, long long, double *, double *, const ExcGeom &, cudaStream_t);
long long hamiltonian_scratch_bytes(long long, long long, const ExcGeom &);
int launch_hamiltonian(const u64 *, long long, const double *, const double *, const u64 *, long long, const void *, void *, long long,
                       long long *, long long, long long *, double *, const ExcGeom &, int, cudaStream_t);
long long sort_workspace_bytes(long long);
int launch_sort_table(const u64 *, const void *, long long, int, int, int, u64 *, void *, long long *, void *, long long, cudaStream_t);
long long moments_scratch_bytes();
int launch_moments(const double *, int, const double *, int, long long, void *, double *, cudaStream_t);
long long reduce_scratch_bytes(long long);
template <typename T>
int launch_reduce(const u64 *, const T *, const T *, const void *, long long, const ExcGeom &, double, int, void *, long long,
                  long long *, u64 *, T *, long long *, cudaStream_t);
int launch_reduce_eloc(const double *, int, const double *, const long long *, const long long *, long long, long long, double *,
                       double *, cudaStream_t);
long long reduce_sample_scratch_bytes(long long);
template <typename T>
int launch_reduce_sample(const u64 *, const T *, const T *, long long, const ExcGeom &, double, int, unsigned long long, const long long *, int,
                         void *, long long, long long *, u64 *, T *, long long *, cudaStream_t);
long long compact_scratch_bytes(long long);
int launch_lookup_count(const unsigned char *, long long, void *, long long, unsigned long long *, cudaStream_t);
int launch_lookup_emit(const unsigned char *, const long long *, long long, const void *, int, void *, long long *, long long *, void *,
                       cudaStream_t);
int launch_unique_count(const u64 *, long long, int, void *, long long, unsigned long long *, cudaStream_t);
int launch_unique_emit(const u64 *, const long long *, long long, int, void *, u64 *, long long *, cudaStream_t);
int launch_peer_gather(const void *const *, int, long long, long long, void *, cudaStream_t);
int launch_peer_gather_rows(const void *const *, long long, const u32 *, long long, long long, int, int, void *, cudaStream_t);
int launch_merge_counts(const long long *, const long long *, long long, long long, long long *, cudaStream_t);
int launch_onv_to_tensor(const u64 *, void *, int, long long, int, cudaStream_t);
int launch_tensor_to_onv(const unsigned char *, unsigned char *, long long, int, cudaStream_t);
int launch_csr_spmm(const long long *, const long long *, const double *, long long, const double *, long long, int, double *, long long,
                    cudaStream_t);
int launch_spin_square(const u64 *, long long, int, const u64 *, long long, const void *, const double *, long long, int, double *,
                       long long, cudaStream_t);
long long rdm_scratch_bytes(long long);
int launch_rdm(const long long *, const long long *, const u64 *, long long, long long, int, const double *, int, void *, long long, double *,
               double *, cudaStream_t);
long long pt2_scratch_bytes(long long, long long, int);
int launch_pt2_rows(const u64 *, long long, const double *, const void *, const void *, int, int, long long *, long long, void *, long long,
                    const ExcGeom &, int, cudaStream_t);
int launch_pt2_sort(long long, long long, int, void *, long long, cudaStream_t);
int launch_pt2_reduce(long long, long long, const double *, const double *, int, int, const double *, long long, int, const double *, void *,
                      long long, double *, long long *, cudaStream_t);

static int check_geometry(int sorb, int nele, int noA, int noB) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB) {
    set_error("sorb = %d not in (0, %d]", sorb, PYNQS_MAX_SORB);
    return PYNQS_EVALUE;
  }
  if (sorb & 1) {
    set_error("sorb = %d must be even (alpha/beta interleaved spin orbitals)", sorb);
    return PYNQS_EVALUE;
  }
  if (noA < 0 || noB < 0 || noA > sorb / 2 || noB > sorb / 2) {
    set_error("noA = %d, noB = %d outside [0, sorb/2 = %d]", noA, noB, sorb / 2);
    return PYNQS_EVALUE;
  }
  if (nele < 0 || nele > PYNQS_MAX_NELE) {
    set_error("nele = %d outside [0, %d]", nele, PYNQS_MAX_NELE);
    return PYNQS_EOVERFLOW;
  }
  return 0;
}

static int num_sd_checked(int sorb, int noA, int noB, long long *out) {
  const long long k = sorb / 2, nvA = k - noA, nvB = k - noB;
  const long long v = noA * nvA + noB * nvB + (long long)noA * (noA - 1) * nvA * (nvA - 1) / 4 +
                      (long long)noB * (noB - 1) * nvB * (nvB - 1) / 4 + (long long)noA * noB * nvA * nvB;
  *out = v;
  if (v >= (1LL << 31) - 2) {
    set_error("number of singles+doubles %lld does not fit the 31-bit row index", v);
    return PYNQS_EOVERFLOW;
  }
  return 0;
}

}  // namespace pynqs

using namespace pynqs;

extern "C" {

int pynqs_abi_version(void) { return PYNQS_ABI_VERSION; }

const char *pynqs_last_error(void) { return g_err; }

int64_t pynqs_launch_count(void) { return (int64_t)g_launches.load(); }

int pynqs_check_sorb(int sorb, int nele) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB) {
    set_error("Sorb error: sorb = %d not in (0, %d]", sorb, PYNQS_MAX_SORB);
    return PYNQS_EVALUE;
  }
  if (nele > PYNQS_MAX_NELE) {
    set_error("electron overflow: nele = %d > %d", nele, PYNQS_MAX_NELE);
    return PYNQS_EOVERFLOW;
  }
  return 0;
}

int pynqs_num_sd(int sorb, int noA, int noB, int64_t *nsd) {
  if (int rc = check_geometry(sorb, 0, noA, noB)) return rc;
  long long v;
  int rc = num_sd_checked(sorb, noA, noB, &v);
  *nsd = v;
  return rc;
}

int pynqs_tensor_to_onv(const uint8_t *states, int64_t n, int sorb, uint8_t *onv, void *stream) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB || n < 0) {
    set_error("tensor_to_onv: bad sorb = %d or n = %lld", sorb, (long long)n);
    return PYNQS_EVALUE;
  }
  return launch_tensor_to_onv(states, onv, n, sorb, (cudaStream_t)stream);
}

int pynqs_onv_to_tensor(const uint8_t *onv, int64_t n, int sorb, void *out, int dtype, void *stream) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB || n < 0 || (dtype != PYNQS_F32 && dtype != PYNQS_F64)) {
    set_error("onv_to_tensor: bad sorb = %d, n = %lld or dtype = %d", sorb, (long long)n, dtype);
    return PYNQS_EVALUE;
  }
  return launch_onv_to_tensor(reinterpret_cast<const u64 *>(onv), out, dtype, n, sorb, (cudaStream_t)stream);
}

int pynqs_comb(const uint8_t *bra, int64_t n, int sorb, int noA, int noB, uint8_t *comb, double *states, void *stream) {
  if (int rc = check_geometry(sorb, 0, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (n <= 0) return 0;
  const ExcGeom g = make_geom(sorb, noA + noB, noA, noB);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = launch_comb(reinterpret_cast<const u64 *>(bra), reinterpret_cast<u64 *>(comb), n, g, st)) return rc;
  if (states) return launch_states(reinterpret_cast<const u64 *>(comb), states, n * (nsd + 1), sorb, st);
  return 0;
}

int pynqs_prepared_bytes(int sorb, int dtype, int64_t *bytes) {
  if (int rc = check_geometry(sorb, 0, 0, 0)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("prepared_bytes: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  *bytes = prepared_bytes(sorb, dtype);
  return 0;
}

int pynqs_prepare_integrals(const void *h2e, int sorb, int dtype, void *prep_ws, int64_t prep_bytes, void *stream) {
  if (int rc = check_geometry(sorb, 0, 0, 0)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("prepare_integrals: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  return launch_prepare(h2e, sorb, dtype, prep_ws, prep_bytes, (cudaStream_t)stream);
}

int pynqs_comb_hij_fused(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb,
                         int nele, int noA, int noB, uint8_t *comb, void *hmat, int dtype, void *stream) {
  if (int rc = check_geometry(sorb, nele, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("comb_hij_fused: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  if (n <= 0) return 0;
  const ExcGeom g = make_geom(sorb, nele, noA, noB);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PYNQS_F64)
    return launch_comb_hij_f64(reinterpret_cast<const u64 *>(bra), (const double *)h1e, (const double *)h2e, prep_ws,
                               reinterpret_cast<u64 *>(comb), (double *)hmat, n, g, st);
  return launch_comb_hij_f32(reinterpret_cast<const u64 *>(bra), (const float *)h1e, (const float *)h2e, prep_ws,
                             reinterpret_cast<u64 *>(comb), (float *)hmat, n, g, st);
}

int pynqs_hij(const uint8_t *bra, const uint8_t *ket, const void *h1e, const void *h2e, int64_t n, int64_t m, int ket3d,
              int sorb, int nele, void *out, int dtype, void *stream) {
  if (int rc = check_geometry(sorb, nele, 0, 0)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("hij: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  if (n <= 0 || m <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PYNQS_F64)
    return launch_hij<double>(reinterpret_cast<const u64 *>(bra), reinterpret_cast<const u64 *>(ket), (const double *)h1e,
                              (const double *)h2e, (double *)out, n, m, ket3d, sorb, nele, st);
  return launch_hij<float>(reinterpret_cast<const u64 *>(bra), reinterpret_cast<const u64 *>(ket), (const float *)h1e,
                           (const float *)h2e, (float *)out, n, m, ket3d, sorb, nele, st);
}

static int check_L(int L) {
  if (L < 1 || L > PYNQS_MAX_SORB_LEN) {
    set_error("ONV width %d bytes unsupported (need 8, 16 or 24)", 8 * L);
    return PYNQS_EVALUE;
  }
  return 0;
}

int pynqs_lut(const uint8_t *key, int64_t N, const uint8_t *onv, int64_t n, int L, int64_t *idx, uint8_t *mask,
              void *stream) {
  if (int rc = check_L(L)) return rc;
  return launch_lut_classic(reinterpret_cast<const u64 *>(key), N, reinterpret_cast<const u64 *>(onv), n, L,
                            reinterpret_cast<long long *>(idx), mask, (cudaStream_t)stream);
}

int pynqs_hash_bytes(int64_t N, int L, int64_t *bytes) {
  if (int rc = check_L(L)) return rc;
  if (N < 0 || N >= (1LL << 32)) {
    set_error("hash index supports 0 <= N < 2^32 keys (got %lld)", (long long)N);
    return PYNQS_EVALUE;
  }
  *bytes = hash_workspace_bytes(N);
  return 0;
}

int pynqs_hash_build(const uint8_t *key, int64_t N, int L, void *hash_ws, int64_t hash_bytes, void *stream) {
  if (int rc = check_L(L)) return rc;
  return launch_hash_build(reinterpret_cast<const u64 *>(key), N, L, hash_ws, hash_bytes, (cudaStream_t)stream);
}

int pynqs_lut_hashed(const uint8_t *key, int64_t N, const uint8_t *onv, int64_t n, int L, const void *hash_ws,
                     int64_t *idx, uint8_t *mask, void *stream) {
  if (int rc = check_L(L)) return rc;
  return launch_lut_hashed(reinterpret_cast<const u64 *>(key), N, reinterpret_cast<const u64 *>(onv), n, L, hash_ws,
                           reinterpret_cast<long long *>(idx), mask, (cudaStream_t)stream);
}

int pynqs_group_bytes(int64_t N, int L, int64_t *bytes) {
  if (int rc = check_L(L)) return rc;
  if (N < 0 || N >= (1LL << 31)) {
    set_error("the grouped table supports 0 <= N < 2^31 keys (got %lld)", (long long)N);
    return PYNQS_EVALUE;
  }
  *bytes = group_workspace_bytes(N, L);
  return 0;
}

int pynqs_group_build(const uint8_t *key, int64_t N, int L, void *group_ws, int64_t group_bytes, void *stream) {
  if (int rc = check_L(L)) return rc;
  return launch_group_build(reinterpret_cast<const u64 *>(key), N, L, group_ws, group_bytes, (cudaStream_t)stream);
}

// h2e placement tier for Hamiltonians that neither fit shared memory nor stay in L2 on their own (north_star: "pinned in a
// persisting-L2 window"): carve persisting L2 out of the cache and mark [ptr, ptr + bytes) as persisting for the work
// launched on `stream` afterwards.  hit_ratio < 1 keeps a window larger than the carve-out from thrashing itself.
int pynqs_l2_persist(const void *ptr, int64_t bytes, double hit_ratio, void *stream, int64_t *granted) {
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return check_launch("l2_persist: device query");
  cudaStreamAttrValue attr;
  memset(&attr, 0, sizeof(attr));
  if (ptr == nullptr || bytes <= 0) {  // reset: no window, persisting lines back to normal
    attr.accessPolicyWindow.num_bytes = 0;
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &attr);
    cudaCtxResetPersistingL2Cache();
    if (granted) *granted = 0;
    return check_launch("l2_persist reset");
  }
  size_t carve = (size_t)prop.persistingL2CacheMaxSize;
  if ((size_t)bytes < carve) carve = (size_t)bytes;
  if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) != cudaSuccess) return check_launch("l2_persist: set-aside");
  size_t win = (size_t)bytes;
  if (win > (size_t)prop.accessPolicyMaxWindowSize) win = (size_t)prop.accessPolicyMaxWindowSize;
  attr.accessPolicyWindow.base_ptr = const_cast<void *>(ptr);
  attr.accessPolicyWindow.num_bytes = win;
  double ratio = hit_ratio > 0.0 ? hit_ratio : (double)carve / (double)win;
  if (ratio > 1.0) ratio = 1.0;
  attr.accessPolicyWindow.hitRatio = (float)ratio;
  attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  if (cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess)
    return check_launch("l2_persist: access policy window");
  if (granted) {
    granted[0] = (int64_t)carve;
    granted[1] = (int64_t)win;
  }
  return 0;
}

int pynqs_peer_gather(const void *const *peer_ptrs, int world, int64_t src_offset, int64_t bytes_per_rank, void *out, void *stream) {
  if (peer_ptrs == nullptr || world < 1 || bytes_per_rank < 0 || src_offset < 0) {
    set_error("peer_gather: bad arguments");
    return PYNQS_EVALUE;
  }
  return launch_peer_gather(peer_ptrs, world, src_offset, bytes_per_rank, out, (cudaStream_t)stream);
}

int pynqs_peer_gather_rows(const void *const *peer_ptrs, int world, int64_t src_offset, const uint32_t *pos, int64_t n, int64_t total,
                           int elem_bytes, void *out, void *stream) {
  if (peer_ptrs == nullptr || world < 1 || n < 0 || total < world || src_offset < 0) {
    set_error("peer_gather_rows: bad arguments");
    return PYNQS_EVALUE;
  }
  return launch_peer_gather_rows(peer_ptrs, src_offset, pos, n, total, world, elem_bytes, out, (cudaStream_t)stream);
}

int pynqs_group_layout(int64_t N, int L, int64_t *out) {
  if (N < 0 || L < 1 || L > PYNQS_MAX_SORB_LEN) {
    set_error("group_layout: bad N = %lld or L = %d", (long long)N, L);
    return PYNQS_EVALUE;
  }
  const GroupLayout l = group_layout(N, L);
  out[0] = (int64_t)l.log2_buckets;
  for (int g = 0; g < 2; ++g) {
    out[1 + g] = l.start_off[g];
    out[3 + g] = l.keys_off[g];
    out[5 + g] = l.rows_off[g];
    out[7 + g] = L == 1 ? l.half_off[g] : -1;
  }
  out[9] = l.pos_off;
  return 0;
}

int pynqs_set_tuning(const char *name, int64_t value) {
  ElocTuning &t = eloc_tuning();
  struct {
    const char *name;
    int *field;
    long long lo, hi;
  } knobs[] = {{"scan_threads", &t.scan_threads, 0, 256},        {"search_factor", &t.search_factor, 1, 4096},
               {"full_keys", &t.full_keys, 0, 1},                {"block_min_samples", &t.block_min_samples, 1, 1LL << 30},
               {"block_min_group", &t.block_min_group, 4, 32},   {"block_enable", &t.block_enable, 0, 1},
               {"eval_tiles", &t.eval_tiles, 0, 2},
               {"lut_pipeline", &t.lut_pipeline, 0, 1},          {"block_parts", &t.block_parts, 0, 4},
               {"sort_chunk", &t.sort_chunk, 0, 1LL << 30}};
  if (name == nullptr) {
    t = ElocTuning();  // back to the production values
    return 0;
  }
  for (auto &k : knobs) {
    if (strcmp(name, k.name) == 0) {
      if (value < k.lo || value > k.hi) {
        set_error("tuning knob %s: value %lld outside [%lld, %lld]", name, (long long)value, k.lo, k.hi);
        return PYNQS_EVALUE;
      }
      *k.field = (int)value;
      return 0;
    }
  }
  set_error("unknown tuning knob '%s'", name);
  return PYNQS_EVALUE;
}

int pynqs_eloc_scratch_bytes(int64_t n, int sorb, int noA, int noB, int psi_complex, int64_t *bytes) {
  if (int rc = check_geometry(sorb, 0, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  (void)psi_complex;
  *bytes = eloc_scratch_bytes(n, make_geom(sorb, noA + noB, noA, noB));
  return 0;
}

int pynqs_eloc_sample_space(const uint8_t *bra, int64_t n, const double *h1e, const double *h2e, int sorb, int nele,
                            int noA, int noB, const uint8_t *key, const void *psi, int psi_complex, int64_t N,
                            const void *group_ws, void *scratch, int64_t scratch_bytes, void *eloc, void *psi0,
                            void *stream) {
  if (int rc = check_geometry(sorb, nele, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  const ExcGeom g = make_geom(sorb, nele, noA, noB);
  return launch_eloc(reinterpret_cast<const u64 *>(bra), n, h1e, h2e, reinterpret_cast<const u64 *>(key),
                     (const double *)psi, psi_complex, N, group_ws, scratch, scratch_bytes, (double *)eloc, (double *)psi0, g,
                     (cudaStream_t)stream);
}

int pynqs_hamiltonian_scratch_bytes(int64_t n, int64_t nnz, int sorb, int noA, int noB, int64_t *bytes) {
  if (int rc = check_geometry(sorb, 0, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (n < 0 || nnz < 0) {
    set_error("hamiltonian_scratch_bytes: bad n = %lld or nnz = %lld", (long long)n, (long long)nnz);
    return PYNQS_EVALUE;
  }
  *bytes = hamiltonian_scratch_bytes(n, nnz, make_geom(sorb, noA + noB, noA, noB));
  return 0;
}

int pynqs_hamiltonian_count(const uint8_t *bra, int64_t n, int sorb, int noA, int noB, const uint8_t *key, int64_t N, const void *group_ws,
                            void *scratch, int64_t scratch_bytes, int64_t *offsets, void *stream) {
  if (int rc = check_geometry(sorb, noA + noB, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  return launch_hamiltonian(reinterpret_cast<const u64 *>(bra), n, nullptr, nullptr, reinterpret_cast<const u64 *>(key), N, group_ws, scratch,
                            scratch_bytes, reinterpret_cast<long long *>(offsets), 0, nullptr, nullptr, make_geom(sorb, noA + noB, noA, noB),
                            0, (cudaStream_t)stream);
}

int pynqs_hamiltonian_emit(const uint8_t *bra, int64_t n, const double *h1e, const double *h2e, int sorb, int nele, int noA, int noB,
                           const uint8_t *key, int64_t N, const void *group_ws, void *scratch, int64_t scratch_bytes, const int64_t *offsets,
                           int64_t nnz, int64_t *col, double *val, void *stream) {
  if (int rc = check_geometry(sorb, nele, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  return launch_hamiltonian(reinterpret_cast<const u64 *>(bra), n, h1e, h2e, reinterpret_cast<const u64 *>(key), N, group_ws, scratch,
                            scratch_bytes, const_cast<long long *>(reinterpret_cast<const long long *>(offsets)), nnz,
                            reinterpret_cast<long long *>(col), val, make_geom(sorb, nele, noA, noB), 1, (cudaStream_t)stream);
}

int pynqs_csr_spmm(const int64_t *crow, const int64_t *col, const double *val, int64_t n, int64_t N, const double *X, int64_t ldx, int k,
                   double *Y, int64_t ldy, void *stream) {
  if (n < 0 || N < 0 || k < 1 || k > 8 || ldx < k || ldy < k) {
    set_error("csr_spmm: bad n = %lld, N = %lld, k = %d, ldx = %lld or ldy = %lld (k in [1, 8], ld >= k)", (long long)n, (long long)N, k,
              (long long)ldx, (long long)ldy);
    return PYNQS_EVALUE;
  }
  if (n > 0 && (crow == nullptr || Y == nullptr || (N > 0 && (col == nullptr || val == nullptr || X == nullptr)))) {
    set_error("csr_spmm: null pointer (crow / Y for n > 0, col / val / X as well for N > 0)");
    return PYNQS_EVALUE;
  }
  if (n == 0) return 0;
  return launch_csr_spmm(reinterpret_cast<const long long *>(crow), reinterpret_cast<const long long *>(col), val, n, X, ldx, k, Y, ldy,
                         (cudaStream_t)stream);
}

int pynqs_spin_square_apply(const uint8_t *bra, int64_t n, int sorb, const uint8_t *key, int64_t N, const void *group_ws, const double *X,
                            int64_t ldx, int k, double *Y, int64_t ldy, void *stream) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB || (sorb & 1)) {
    set_error("spin_square_apply: sorb = %d must be even and in (0, %d]", sorb, PYNQS_MAX_SORB);
    return PYNQS_EVALUE;
  }
  if (n < 0 || N < 0 || N >= (1LL << 31) || k < 1 || k > 8 || ldx < k || ldy < k) {
    set_error("spin_square_apply: bad n = %lld, N = %lld, k = %d, ldx = %lld or ldy = %lld (N < 2^31, k in [1, 8], ld >= k)",
              (long long)n, (long long)N, k, (long long)ldx, (long long)ldy);
    return PYNQS_EVALUE;
  }
  if (n > 0 && (bra == nullptr || Y == nullptr || (N > 0 && (key == nullptr || group_ws == nullptr || X == nullptr)))) {
    set_error("spin_square_apply: null pointer (bra / Y for n > 0, key / group_ws / X as well for N > 0)");
    return PYNQS_EVALUE;
  }
  if (n == 0) return 0;
  if (N == 0) {  // no partner and no diagonal is in an empty table: Y = 0, without a kernel
    if (cudaMemset2DAsync(Y, 8 * (size_t)ldy, 0, 8 * (size_t)k, (size_t)n, (cudaStream_t)stream) != cudaSuccess)
      return check_launch("spin_square_apply: memset of Y");
    return 0;
  }
  return launch_spin_square(reinterpret_cast<const u64 *>(bra), n, (sorb - 1) / 64 + 1, reinterpret_cast<const u64 *>(key), N, group_ws, X,
                            ldx, k, Y, ldy, (cudaStream_t)stream);
}

static int rdm_check(const char *what, int64_t N, int64_t nnz, int sorb) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB || (sorb & 1)) {
    set_error("%s: sorb = %d must be even and in (0, %d]", what, sorb, PYNQS_MAX_SORB);
    return PYNQS_EVALUE;
  }
  if (N < 0 || N >= (1LL << 31) || nnz < 0 || nnz >= (1LL << 31)) {
    set_error("%s: bad N = %lld or nnz = %lld (both < 2^31)", what, (long long)N, (long long)nnz);
    return PYNQS_EVALUE;
  }
  return 0;
}

int pynqs_rdm_scratch_bytes(int64_t N, int64_t nnz, int sorb, int64_t *bytes) {
  if (int rc = rdm_check("rdm_scratch_bytes", N, nnz, sorb)) return rc;
  if (bytes == nullptr) {
    set_error("rdm_scratch_bytes: null bytes");
    return PYNQS_EVALUE;
  }
  *bytes = rdm_scratch_bytes(nnz);
  return 0;
}

int pynqs_rdm_offdiag(const int64_t *crow, const int64_t *col, const uint8_t *key, int64_t N, int64_t nnz, int sorb, const double *c,
                      int c_complex, void *scratch, int64_t scratch_bytes, double *dm1, double *dm2, void *stream) {
  if (int rc = rdm_check("rdm_offdiag", N, nnz, sorb)) return rc;
  if (c_complex != 0 && c_complex != 1) {
    set_error("rdm_offdiag: c_complex = %d must be 0 or 1", c_complex);
    return PYNQS_EVALUE;
  }
  if (dm1 == nullptr || (N > 0 && (crow == nullptr || key == nullptr || c == nullptr)) ||
      (nnz > 0 && (col == nullptr || scratch == nullptr))) {
    set_error("rdm_offdiag: null pointer (dm1; crow / key / c for N > 0; col / scratch for nnz > 0)");
    return PYNQS_EVALUE;
  }
  const size_t norb = (size_t)(sorb / 2), el = c_complex ? 16 : 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(dm1, 0, 2 * norb * norb * el, st) != cudaSuccess ||
      (dm2 != nullptr && cudaMemsetAsync(dm2, 0, 3 * norb * norb * norb * norb * el, st) != cudaSuccess))
    return check_launch("rdm_offdiag: memset of dm1 / dm2");
  if (N == 0 || nnz == 0) return 0;
  return launch_rdm(reinterpret_cast<const long long *>(crow), reinterpret_cast<const long long *>(col), reinterpret_cast<const u64 *>(key), N,
                    nnz, sorb, c, c_complex, scratch, scratch_bytes, dm1, dm2, st);
}

static int pt2_check(const char *what, int64_t N, int64_t pairs, int sorb) {
  if (sorb <= 0 || sorb > PYNQS_MAX_SORB || (sorb & 1)) {
    set_error("%s: sorb = %d must be even and in (0, %d]", what, sorb, PYNQS_MAX_SORB);
    return PYNQS_EVALUE;
  }
  if (N <= 0 || N >= (1LL << 31) || pairs < 0 || pairs >= (1LL << 31)) {
    set_error("%s: bad N = %lld or pairs = %lld (0 < N < 2^31, 0 <= pairs < 2^31)", what, (long long)N, (long long)pairs);
    return PYNQS_EVALUE;
  }
  return 0;
}

static int pt2_rows_common(const char *what, const uint8_t *key, int64_t N, const double *h1e, const void *prep_ws, int sorb, int noA, int noB,
                           const void *group_ws, int part, int log2_parts, int64_t *offsets, int64_t pairs, void *scratch,
                           int64_t scratch_bytes, int emit, void *stream) {
  if (int rc = check_geometry(sorb, noA + noB, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (int rc = pt2_check(what, N, pairs, sorb)) return rc;
  if (log2_parts < 0 || log2_parts > 31 || part < 0 || (long long)part >= (1LL << log2_parts)) {
    set_error("%s: bad part = %d of 2^%d partitions", what, part, log2_parts);
    return PYNQS_EVALUE;
  }
  if (key == nullptr || group_ws == nullptr || scratch == nullptr || offsets == nullptr || (emit && (h1e == nullptr || prep_ws == nullptr))) {
    set_error("%s: null pointer (key / group_ws / scratch / offsets, h1e / prep_ws for the emit call)", what);
    return PYNQS_EVALUE;
  }
  if (emit && pairs == 0) return 0;
  return launch_pt2_rows(reinterpret_cast<const u64 *>(key), N, h1e, prep_ws, group_ws, part, log2_parts, reinterpret_cast<long long *>(offsets),
                         pairs, scratch, scratch_bytes, make_geom(sorb, noA + noB, noA, noB), emit, (cudaStream_t)stream);
}

int pynqs_pt2_scratch_bytes(int64_t N, int64_t pairs, int sorb, int64_t *bytes) {
  if (int rc = pt2_check("pt2_scratch_bytes", N, pairs, sorb)) return rc;
  if (bytes == nullptr) {
    set_error("pt2_scratch_bytes: null bytes");
    return PYNQS_EVALUE;
  }
  *bytes = pt2_scratch_bytes(N, pairs, (sorb - 1) / 64 + 1);
  return 0;
}

int pynqs_pt2_count(const uint8_t *key, int64_t N, int sorb, int noA, int noB, const void *group_ws, int part, int log2_parts, void *scratch,
                    int64_t scratch_bytes, int64_t *offsets, void *stream) {
  return pt2_rows_common("pt2_count", key, N, nullptr, nullptr, sorb, noA, noB, group_ws, part, log2_parts, offsets, 0, scratch, scratch_bytes,
                         0, stream);
}

int pynqs_pt2_emit(const uint8_t *key, int64_t N, const double *h1e, const void *prep_ws, int sorb, int noA, int noB, const void *group_ws,
                   int part, int log2_parts, const int64_t *offsets, int64_t pairs, void *scratch, int64_t scratch_bytes, void *stream) {
  return pt2_rows_common("pt2_emit", key, N, h1e, prep_ws, sorb, noA, noB, group_ws, part, log2_parts, const_cast<int64_t *>(offsets), pairs,
                         scratch, scratch_bytes, 1, stream);
}

int pynqs_pt2_sort(int64_t N, int64_t pairs, int sorb, void *scratch, int64_t scratch_bytes, void *stream) {
  if (int rc = pt2_check("pt2_sort", N, pairs, sorb)) return rc;
  if (scratch == nullptr) {
    set_error("pt2_sort: null scratch");
    return PYNQS_EVALUE;
  }
  if (pairs == 0) return 0;
  return launch_pt2_sort(N, pairs, sorb, scratch, scratch_bytes, (cudaStream_t)stream);
}

int pynqs_pt2_reduce(int64_t N, int64_t pairs, const double *h1e, const double *h2e, int sorb, int nele, const double *C, int64_t ldc, int k,
                     const double *E, void *scratch, int64_t scratch_bytes, double *acc, int64_t *externals, void *stream) {
  if (int rc = pt2_check("pt2_reduce", N, pairs, sorb)) return rc;
  if (nele < 0 || nele > sorb || k < 1 || k > 8 || ldc < k) {
    set_error("pt2_reduce: bad nele = %d, k = %d or ldc = %lld (k in [1, 8], ldc >= k)", nele, k, (long long)ldc);
    return PYNQS_EVALUE;
  }
  if (h1e == nullptr || h2e == nullptr || C == nullptr || E == nullptr || scratch == nullptr || acc == nullptr) {
    set_error("pt2_reduce: null pointer (h1e / h2e / C / E / scratch / acc)");
    return PYNQS_EVALUE;
  }
  if (pairs == 0) return 0;
  return launch_pt2_reduce(N, pairs, h1e, h2e, sorb, nele, C, ldc, k, E, scratch, scratch_bytes, acc, reinterpret_cast<long long *>(externals),
                           (cudaStream_t)stream);
}

int64_t pynqs_reduce_scratch_bytes(int64_t n) { return reduce_scratch_bytes(n); }

static int reduce_common(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb, int nele,
                         int noA, int noB, double eps, int dtype, int emit, void *scratch, int64_t scratch_bytes, int64_t *offsets,
                         uint8_t *x, void *hij, int64_t *idx, void *stream) {
  if (int rc = check_geometry(sorb, nele, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("reduce: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  if (prep_ws == nullptr) {
    set_error("reduce: the prepared integrals (pynqs_prepare_integrals) are required");
    return PYNQS_EVALUE;
  }
  if (n < 0 || !(eps >= 0.0)) {
    set_error("reduce: bad n = %lld or eps = %g", (long long)n, eps);
    return PYNQS_EVALUE;
  }
  const ExcGeom g = make_geom(sorb, nele, noA, noB);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PYNQS_F64)
    return launch_reduce<double>(reinterpret_cast<const u64 *>(bra), (const double *)h1e, (const double *)h2e, prep_ws, n, g, eps, emit,
                                 scratch, scratch_bytes, reinterpret_cast<long long *>(offsets), reinterpret_cast<u64 *>(x),
                                 (double *)hij, reinterpret_cast<long long *>(idx), st);
  return launch_reduce<float>(reinterpret_cast<const u64 *>(bra), (const float *)h1e, (const float *)h2e, prep_ws, n, g, eps, emit,
                              scratch, scratch_bytes, reinterpret_cast<long long *>(offsets), reinterpret_cast<u64 *>(x), (float *)hij,
                              reinterpret_cast<long long *>(idx), st);
}

int pynqs_reduce_count(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb, int nele,
                       int noA, int noB, double eps, int dtype, void *scratch, int64_t scratch_bytes, int64_t *offsets,
                       void *stream) {
  return reduce_common(bra, h1e, h2e, prep_ws, n, sorb, nele, noA, noB, eps, dtype, 0, scratch, scratch_bytes, offsets, nullptr,
                       nullptr, nullptr, stream);
}

int pynqs_reduce_emit(const uint8_t *bra, const void *h1e, const void *h2e, const void *prep_ws, int64_t n, int sorb, int nele,
                      int noA, int noB, double eps, int dtype, void *scratch, int64_t scratch_bytes, const int64_t *offsets,
                      uint8_t *x, void *hij, int64_t *idx, void *stream) {
  return reduce_common(bra, h1e, h2e, prep_ws, n, sorb, nele, noA, noB, eps, dtype, 1, scratch, scratch_bytes,
                       const_cast<int64_t *>(offsets), x, hij, idx, stream);
}

int64_t pynqs_reduce_sample_scratch_bytes(int64_t n) { return reduce_sample_scratch_bytes(n); }

static int reduce_sample_common(const uint8_t *bra, const void *h1e, const void *h2e, int64_t n, int sorb, int nele, int noA, int noB,
                                double eps, int eps_sample, uint64_t seed, const int64_t *draws, int dtype, int emit, void *scratch,
                                int64_t scratch_bytes, int64_t *offsets, uint8_t *x, void *hij, int64_t *idx, void *stream) {
  if (int rc = check_geometry(sorb, nele, noA, noB)) return rc;
  long long nsd;
  if (int rc = num_sd_checked(sorb, noA, noB, &nsd)) return rc;
  if (dtype != PYNQS_F32 && dtype != PYNQS_F64) {
    set_error("reduce_sample: dtype %d is neither float32 nor float64", dtype);
    return PYNQS_EVALUE;
  }
  if (n < 0 || !(eps >= 0.0) || eps_sample < 1) {
    set_error("reduce_sample: bad n = %lld, eps = %g or eps_sample = %d", (long long)n, eps, eps_sample);
    return PYNQS_EVALUE;
  }
  const ExcGeom g = make_geom(sorb, nele, noA, noB);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PYNQS_F64)
    return launch_reduce_sample<double>(reinterpret_cast<const u64 *>(bra), (const double *)h1e, (const double *)h2e, n, g, eps, eps_sample,
                                        seed, reinterpret_cast<const long long *>(draws), emit, scratch, scratch_bytes,
                                        reinterpret_cast<long long *>(offsets), reinterpret_cast<u64 *>(x), (double *)hij,
                                        reinterpret_cast<long long *>(idx), st);
  return launch_reduce_sample<float>(reinterpret_cast<const u64 *>(bra), (const float *)h1e, (const float *)h2e, n, g, eps, eps_sample, seed,
                                     reinterpret_cast<const long long *>(draws), emit, scratch, scratch_bytes,
                                     reinterpret_cast<long long *>(offsets), reinterpret_cast<u64 *>(x), (float *)hij,
                                     reinterpret_cast<long long *>(idx), st);
}

int pynqs_reduce_sample_count(const uint8_t *bra, const void *h1e, const void *h2e, int64_t n, int sorb, int nele, int noA, int noB,
                              double eps, int eps_sample, uint64_t seed, const int64_t *draws, int dtype, void *scratch,
                              int64_t scratch_bytes, int64_t *offsets, void *stream) {
  return reduce_sample_common(bra, h1e, h2e, n, sorb, nele, noA, noB, eps, eps_sample, seed, draws, dtype, 0, scratch, scratch_bytes, offsets,
                              nullptr, nullptr, nullptr, stream);
}

int pynqs_reduce_sample_emit(const uint8_t *bra, const void *h1e, const void *h2e, int64_t n, int sorb, int nele, int noA, int noB,
                             double eps, int eps_sample, uint64_t seed, const int64_t *draws, int dtype, void *scratch,
                             int64_t scratch_bytes, const int64_t *offsets, uint8_t *x, void *hij, int64_t *idx, void *stream) {
  return reduce_sample_common(bra, h1e, h2e, n, sorb, nele, noA, noB, eps, eps_sample, seed, draws, dtype, 1, scratch, scratch_bytes,
                              const_cast<int64_t *>(offsets), x, hij, idx, stream);
}

int pynqs_reduce_eloc(const void *psi, int psi_complex, const double *hij, const int64_t *idx, const int64_t *offsets, int64_t n,
                      int64_t M, void *eloc, void *psi0, void *stream) {
  if (n < 0 || M <= 0) {
    set_error("reduce_eloc: bad n = %lld or M = %lld", (long long)n, (long long)M);
    return PYNQS_EVALUE;
  }
  return launch_reduce_eloc((const double *)psi, psi_complex, hij, reinterpret_cast<const long long *>(idx),
                            reinterpret_cast<const long long *>(offsets), n, M, (double *)eloc, (double *)psi0, (cudaStream_t)stream);
}

int64_t pynqs_compact_scratch_bytes(int64_t n) { return compact_scratch_bytes(n); }

int pynqs_lookup_count(const uint8_t *mask, int64_t n, void *scratch, int64_t scratch_bytes, uint64_t *n_hit, void *stream) {
  if (n < 0) {
    set_error("lookup_count: bad n = %lld", (long long)n);
    return PYNQS_EVALUE;
  }
  return launch_lookup_count(mask, n, scratch, scratch_bytes, reinterpret_cast<unsigned long long *>(n_hit), (cudaStream_t)stream);
}

int pynqs_lookup_emit(const uint8_t *mask, const int64_t *idx, int64_t n, const void *value_table, int value_bytes, void *scratch,
                      int64_t *hit_pos, int64_t *miss_pos, void *value, void *stream) {
  if (n < 0 || (value_bytes != 8 && value_bytes != 16)) {
    set_error("lookup_emit: bad n = %lld or value_bytes = %d", (long long)n, value_bytes);
    return PYNQS_EVALUE;
  }
  return launch_lookup_emit(mask, reinterpret_cast<const long long *>(idx), n, value_table, value_bytes, scratch,
                            reinterpret_cast<long long *>(hit_pos), reinterpret_cast<long long *>(miss_pos), value, (cudaStream_t)stream);
}

int pynqs_unique_count(const uint8_t *sorted_key, int64_t n, int L, void *scratch, int64_t scratch_bytes, uint64_t *n_unique, void *stream) {
  if (n < 0 || L < 1 || L > PYNQS_MAX_SORB_LEN) {
    set_error("unique_count: bad n = %lld or L = %d", (long long)n, L);
    return PYNQS_EVALUE;
  }
  return launch_unique_count(reinterpret_cast<const u64 *>(sorted_key), n, L, scratch, scratch_bytes,
                             reinterpret_cast<unsigned long long *>(n_unique), (cudaStream_t)stream);
}

int pynqs_unique_emit(const uint8_t *sorted_key, const int64_t *perm, int64_t n, int L, void *scratch, uint8_t *unique, int64_t *inverse,
                      void *stream) {
  if (n < 0 || L < 1 || L > PYNQS_MAX_SORB_LEN) {
    set_error("unique_emit: bad n = %lld or L = %d", (long long)n, L);
    return PYNQS_EVALUE;
  }
  return launch_unique_emit(reinterpret_cast<const u64 *>(sorted_key), reinterpret_cast<const long long *>(perm), n, L, scratch,
                            reinterpret_cast<u64 *>(unique), reinterpret_cast<long long *>(inverse), (cudaStream_t)stream);
}

int64_t pynqs_sort_bytes(int64_t N) { return sort_workspace_bytes(N < 0 ? 0 : N); }

int pynqs_sort_table(const uint8_t *key, const void *psi, int64_t N, int L, int sorb, int psi_bytes, uint8_t *key_out,
                     void *psi_out, int64_t *perm_out, void *ws, int64_t ws_bytes, void *stream) {
  if (N < 0 || L < 1 || L > PYNQS_MAX_SORB_LEN || (psi != nullptr && psi_bytes != 8 && psi_bytes != 16) || sorb > 64 * L) {
    set_error("sort_table: bad N = %lld, L = %d, sorb = %d or psi_bytes = %d", (long long)N, L, sorb, psi_bytes);
    return PYNQS_EVALUE;
  }
  return launch_sort_table(reinterpret_cast<const u64 *>(key), psi, N, L, sorb, psi_bytes, reinterpret_cast<u64 *>(key_out), psi_out,
                           reinterpret_cast<long long *>(perm_out), ws, ws_bytes, (cudaStream_t)stream);
}

int pynqs_merge_rank_sample(const int64_t *idx, const int64_t *counts, int64_t n, int64_t length, int64_t *out, void *stream) {
  if (n < 0 || length < 0) {
    set_error("merge_rank_sample: bad n = %lld or length = %lld", (long long)n, (long long)length);
    return PYNQS_EVALUE;
  }
  return launch_merge_counts(reinterpret_cast<const long long *>(idx), reinterpret_cast<const long long *>(counts), n, length,
                             reinterpret_cast<long long *>(out), (cudaStream_t)stream);
}

int64_t pynqs_moments_scratch_bytes(void) { return moments_scratch_bytes(); }

int pynqs_weighted_moments(const void *eloc, int eloc_complex, const void *weight, int weight_kind, int64_t n, void *scratch,
                           double *out, void *stream) {
  if (n < 0 || weight_kind < 0 || weight_kind > 2) {
    set_error("weighted_moments: bad n = %lld or weight_kind = %d", (long long)n, weight_kind);
    return PYNQS_EVALUE;
  }
  return launch_moments((const double *)eloc, eloc_complex, (const double *)weight, weight_kind, n, scratch, out, (cudaStream_t)stream);
}

}  // extern "C"
