"""Reduced density matrices over the sample space (energy.make_rdm1s / make_rdm12s) next to the H build they need and one
csr_matmul over it, on the benchmarked 10^6-sample Fe2S2 set, its Zipf-0.8 variant (each its own table, as the bench runs
them) and the 18 496-determinant Fe2S2 CI space.

    python profiles/micro/rdm.py [out.json]      # profiles/r07/rdm.json

Reports the GPU and its power limit; per table the CSR entries (nnz), the off-diagonal records the RDM kernel sorts
(nnz - N), the scratch bytes per CSR entry, and the times (CUDA events, median (min, max) of 10 calls after 3 warm-up
calls).  make_rdm1s / make_rdm12s include their argument checks (two host synchronisations: sum |c|^2 and duplicate keys,
then nnz), the occupation products and the normalisation."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200 import _lib  # noqa: E402
from pynqs_b200 import synthetic as S  # noqa: E402
from pynqs_b200.energy import make_rdm1s, make_rdm12s, sample_space_hamiltonian  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402
from sample_space_diag import gpu_name_and_power, timed  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE


def main():
    h1e_np, h2e_np, _ = bench.load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    out = {"gpu": gpu_name_and_power(), "config": "Fe2S2 40 sorb 15a15b, float64 c = the table's random psi",
           "timing": "CUDA events, median (min, max) of 10 calls after 3 warm-up calls; table, H and c resident between calls "
                     "(no cache flush)"}
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import fe2s2

    tables = {"uniform": lambda: bench.make_table("uniform", 1_000_000), "zipf0.8": lambda: bench.make_table("zipf0.8", 1_000_000),
              "fe2s2_ci": lambda: fe2s2()["ci"]}
    for name, make in tables.items():
        keys = make()
        lut = WavefunctionLUT(torch.from_numpy(keys).to(dev), torch.from_numpy(S.random_psi(keys.shape[0], seed=1235)).to(dev), SORB, dev,
                              rank=0, world_size=1)
        x, N, c = lut.bra_key, lut.bra_key.size(0), lut.wf_value

        def build():
            return sample_space_hamiltonian(x, h1e, h2e, lut, SORB, NELE, NOA, NOB)

        H = build()
        crow, col, val = H.crow_indices(), H.col_indices(), H.values()
        nnz = col.numel()
        nb = _lib.ctypes.c_int64()
        _lib.check(_lib.load().pynqs_rdm_scratch_bytes(_lib.i64(N), _lib.i64(nnz), SORB, _lib.ctypes.byref(nb)))
        res = {"n": N, "nnz": nnz, "records_off_diagonal": nnz - N, "scratch_bytes_per_csr_entry": nb.value / nnz}
        res["hamiltonian_build_ms"] = timed(build, reps=10)
        res["csr_matmul_k1_ms"] = timed(lambda: ops.csr_matmul(crow, col, val, c, N), reps=10)
        res["make_rdm1s_ms"] = timed(lambda: make_rdm1s(lut, c, SORB, H), reps=10)
        res["make_rdm12s_ms"] = timed(lambda: make_rdm12s(lut, c, SORB, H), reps=10)
        res["make_rdm12s_over_build"] = res["make_rdm12s_ms"][0] / res["hamiltonian_build_ms"][0]
        out[name] = res
        print(name, json.dumps(res), flush=True)
        del lut, x, H, crow, col, val
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
