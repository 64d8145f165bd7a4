"""Time of the sample-space Hamiltonian (count + emit, pynqs_hamiltonian_count / _emit) on the benchmarked 10^6-sample
Fe2S2 set and its Zipf-0.8 variant, next to the one-pass E_loc call on the same inputs.

    python profiles/micro/hamiltonian_build.py [out.json]      # profiles/r03/hamiltonian_build.json

Reports the GPU and its power limit, nnz, count / emit / E_loc times (CUDA events, medians after warm-up), the bytes of
the output (crow + col + val) and their rate, and the identity (H psi)[i] = eloc[i] * psi0[i] over all rows."""
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from pynqs_b200 import C_extension as ops  # noqa: E402
from pynqs_b200 import _lib  # noqa: E402
from pynqs_b200 import synthetic as S  # noqa: E402
from pynqs_b200.lut import WavefunctionLUT  # noqa: E402

dev = torch.device("cuda", 0)
SORB, NOA, NOB, NELE = bench.SORB, bench.NOA, bench.NOB, bench.NELE


def timed(fn, reps=7):
    for _ in range(2):
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
    out = {"gpu": gpu_name_and_power(), "config": "Fe2S2 40 sorb 15a15b, 10^6 samples = the table (bench.make_table)"}
    for table in ("uniform", "zipf0.8"):
        keys = bench.make_table(table, 1_000_000)
        psi = S.random_psi(keys.shape[0], seed=1235)
        lut = WavefunctionLUT(torch.from_numpy(keys).to(dev), torch.from_numpy(psi).to(dev), SORB, dev, rank=0, world_size=1)
        x, key, gi = lut.bra_key, lut.bra_key, lut.group_index
        n, N = x.size(0), key.size(0)
        lib = _lib.load()
        stream = _lib.vp(torch.cuda.current_stream(dev).cuda_stream)
        crow = torch.empty(n + 1, dtype=torch.int64, device=dev)

        def nbytes(nnz):
            b = _lib.ctypes.c_int64()
            _lib.check(lib.pynqs_hamiltonian_scratch_bytes(_lib.i64(n), _lib.i64(nnz), SORB, NOA, NOB, _lib.ctypes.byref(b)))
            return b.value

        table_args = (_lib.vp(key.data_ptr()), _lib.i64(N), _lib.vp(gi.workspace.data_ptr()))
        scratch0 = torch.empty(nbytes(0), dtype=torch.uint8, device=dev)

        def count():
            _lib.check(lib.pynqs_hamiltonian_count(_lib.vp(x.data_ptr()), _lib.i64(n), SORB, NOA, NOB, *table_args,
                                                   _lib.vp(scratch0.data_ptr()), _lib.i64(scratch0.numel()), _lib.vp(crow.data_ptr()), stream))

        count()
        nnz = int(crow[n].item())
        scratch = torch.empty(nbytes(nnz), dtype=torch.uint8, device=dev)
        col = torch.empty(nnz, dtype=torch.int64, device=dev)
        val = torch.empty(nnz, dtype=torch.float64, device=dev)

        def emit():
            _lib.check(lib.pynqs_hamiltonian_emit(_lib.vp(x.data_ptr()), _lib.i64(n), _lib.vp(h1e.data_ptr()), _lib.vp(h2e.data_ptr()), SORB,
                                                  NELE, NOA, NOB, *table_args, _lib.vp(scratch.data_ptr()), _lib.i64(scratch.numel()),
                                                  _lib.vp(crow.data_ptr()), _lib.i64(nnz), _lib.vp(col.data_ptr()), _lib.vp(val.data_ptr()),
                                                  stream))

        def eloc():
            return ops.eloc_sample_space(x, h1e, h2e, SORB, NELE, NOA, NOB, key, lut.wf_value, gi)

        t_count, t_emit, t_eloc = timed(count), timed(emit), timed(eloc)
        e, p0 = eloc()
        Hpsi = torch.sparse.mm(torch.sparse_csr_tensor(crow, col, val, size=(n, N)), lut.wf_value.view(-1, 1)).view(-1)
        want = e * p0
        out_bytes = 8 * (n + 1) + 16 * nnz
        t_build = t_count[0] + t_emit[0]
        out[table] = {
            "n": n, "N": N, "nnz": nnz, "entries_per_row": nnz / n,
            "count_ms": t_count, "emit_ms": t_emit, "eloc_sample_space_ms": t_eloc, "count_plus_emit_over_eloc": t_build / t_eloc[0],
            "output_bytes": out_bytes, "output_gb_per_s": out_bytes / (t_build * 1e-3) / 1e9,
            "scratch_bytes_emit": scratch.numel(),
            "hpsi_identity_max_rel_err": float(((Hpsi - want).abs() / want.abs()).max()),
            "timing": "CUDA events, median (min, max) of 7 calls after 2 warm-up calls; inputs stay resident between calls",
        }
        del scratch, scratch0, col, val, Hpsi
        torch.cuda.empty_cache()
    txt = json.dumps(out, indent=1)
    print(txt)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
