"""The CSR x block product (C_extension.csr_matmul) and the Davidson solve (energy.sample_space_ground_state) on the
benchmarked 10^6-sample Fe2S2 set and its Zipf-0.8 variant, each its own table (built as hamiltonian_build.py builds them).

    python profiles/micro/sample_space_diag.py [out.json]      # profiles/r03/sample_space_diag.json

Reports the GPU and its power limit; per table nnz, csr_matmul and torch.sparse.mm on the same CSR for k = 1, 4, 8 (CUDA
events, medians after warm-up) with the rate of the col + val stream (16 B per entry), the largest difference between the
two products; and Davidson iterations, products and wall time (host clock around a device synchronise) for nroots = 1, 4."""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200 import synthetic as S  # noqa: E402
from pynqs_b200.energy import sample_space_ground_state, sample_space_hamiltonian  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE


def timed(fn, reps=20):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts), max(ts)


def gpu_name_and_power():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(dev)


def main():
    h1e_np, h2e_np, _ = bench.load_integrals()
    h1e, h2e = torch.from_numpy(h1e_np).to(dev), torch.from_numpy(h2e_np).to(dev)
    out = {"gpu": gpu_name_and_power(), "config": "Fe2S2 40 sorb 15a15b, 10^6 samples = the table (bench.make_table)",
           "timing": "csr_matmul / torch.sparse.mm: CUDA events, median (min, max) of 20 calls after 3 warm-up calls, CSR and X "
                     "resident (X of 8-64 MB stays in L2, col + val do not); Davidson: host clock around the whole call, "
                     "ending in a device synchronise"}
    for table in ("uniform", "zipf0.8"):
        keys = bench.make_table(table, 1_000_000)
        lut = WavefunctionLUT(torch.from_numpy(keys).to(dev), torch.from_numpy(S.random_psi(keys.shape[0], seed=1235)).to(dev), SORB, dev,
                              rank=0, world_size=1)
        H = sample_space_hamiltonian(lut.bra_key, h1e, h2e, lut, SORB, NELE, NOA, NOB)
        crow, col, val = H.crow_indices(), H.col_indices(), H.values()
        n, nnz = crow.numel() - 1, col.numel()
        res = {"n": n, "nnz": nnz, "entries_per_row": nnz / n, "max_row": int((crow[1:] - crow[:-1]).max())}
        g = torch.Generator(device=dev).manual_seed(5)
        for k in (1, 4, 8):
            X = torch.randn(n, k, dtype=torch.float64, device=dev, generator=g)
            t_own = timed(lambda: ops.csr_matmul(crow, col, val, X, n))
            t_ref = timed(lambda: torch.sparse.mm(H, X))
            a, b = ops.csr_matmul(crow, col, val, X, n), torch.sparse.mm(H, X)
            res[f"k{k}"] = {
                "csr_matmul_ms": t_own, "torch_sparse_mm_ms": t_ref, "speedup_vs_torch_sparse_mm": t_ref[0] / t_own[0],
                "col_val_gb_per_s": 16 * nnz / (t_own[0] * 1e-3) / 1e9,
                "max_rel_diff_vs_torch_sparse_mm": float(((a - b).abs().max() / b.abs().max())),
            }
            del X, a, b
        for nroots in (1, 4):
            sample_space_ground_state(lut, h1e, h2e, SORB, NELE, NOA, NOB, nroots, H=H, max_iter=2)  # warm-up of the shapes
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e, C, info = sample_space_ground_state(lut, h1e, h2e, SORB, NELE, NOA, NOB, nroots, H=H)
            torch.cuda.synchronize()
            res[f"davidson_nroots{nroots}"] = {"solve_s": time.perf_counter() - t0, "energies": e.tolist(), **info}
        out[table] = res
        del H, crow, col, val, lut
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
