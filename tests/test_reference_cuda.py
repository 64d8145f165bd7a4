"""GPU-vs-GPU: this library against the UNMODIFIED reference CUDA extension (cpp_src/compile.sh -s GPU recipe,
cross-compiled for sm_100a by oracle/build_ref.py into the git-ignored oracle/_ref/C_extension_cuda_L{1,2}.so)
on the same device tensors -- SURVEY.md section 8(c) calls it the literal parity target.  Bit-exact for
determinant lists, lookup indices, masks and conversions; H_ij bit-exact (same order of additions).

The expected outputs are stored as SHA-256 digests in tests/golden/reference_cuda.npz, so the test runs without the
reference; where its build is present, every output is also compared with a live call of it.  The digests come from the
CPU oracle (oracle/pynqs_oracle.c, pinned bit for bit to the reference extension by test_oracle_golden.py), never from
this library: `PYTHONPATH=. python tests/test_reference_cuda.py tests/golden/reference_cuda.npz` from the repository root."""
import sys

import numpy as np
import pytest
import torch

from pynqs_b200 import C_extension as ops
from pynqs_b200 import synthetic as S

from util import fe2s2, load, sha

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OPERATOR_CASES = [(1, 40, 15, 15, 512), (1, 52, 5, 5, 256), (1, 12, 3, 3, 300), (2, 100, 25, 25, 3), (2, 100, 4, 3, 200)]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def ref_cuda(L):
    """the reference CUDA build, or None where it was not built"""
    from oracle import build_ref

    from pynqs_b200 import _lib

    _lib.load()
    assert torch.cuda.is_available()
    return build_ref.load_ref(L, cuda=True) if build_ref.cuda_available(L) else None


def rejected_by_reference(L, sorb, nele):
    """The reference's check_sorb limits (cpp_src/common/default.h: MAX_NELE = MAX_NV = 40 L, SURVEY.md D3)."""
    return nele > 40 * L or sorb - nele > 40 * L


def fe2s2_inputs():
    f = fe2s2()
    return f, dev(f["ci"][:2048].copy()), dev(f["h1e"]), dev(f["h2e"])


def operator_inputs(sorb, noA, noB, n, dtype):
    bra = S.random_onvs(n, sorb, noA, noB, seed=91)
    h1e, h2e = S.random_packed_integrals(sorb, seed=92, symmetric=False, dtype=dtype)
    return dev(bra), dev(h1e), dev(h2e)


def operator_outputs(mod, x, d1, d2, sorb, noA, noB):
    """Every output the operator test compares, from `mod` (this library or the reference extension).  The lookup
    table is sorted by this library in both cases, and the queries are the connected determinants of the first samples."""
    nele = noA + noB
    comb, hmat = mod.get_comb_hij_fused(x, d1, d2, sorb, nele, noA, noB)
    m = min(x.size(0), 128)
    st = mod.onv_to_tensor(x, sorb)
    occ = ((st + 1) / 2).to(torch.uint8)
    order = ops.sort_table(x, None, sorb)[0]
    q = comb[: min(x.size(0), 64)].reshape(-1, comb.size(2)).contiguous()
    idx, mask = mod.wavefunction_lut(order, q, sorb)
    return {"comb": comb, "hmat": hmat, "comb_tensor": mod.get_comb_tensor(x, sorb, nele, noA, noB, False)[0],
            "hij_3d": mod.get_hij_torch(x, comb, d1, d2, sorb, nele), "hij_2d": mod.get_hij_torch(x[:m], x[:m].contiguous(), d1, d2, sorb, nele),
            "onv_to_tensor": st, "tensor_to_onv": mod.tensor_to_onv(occ, sorb), "lut_idx": idx, "lut_mask": mask}


def digests(outs, prefix):
    return {f"{prefix}/{k}": sha(v.cpu().numpy()) for k, v in outs.items()}


def case_name(L, sorb, noA, noB, n, dtype):
    return f"L{L}_{sorb}sorb_{noA}a{noB}b_n{n}_{np.dtype(dtype).name}"


def assert_same(got, want):
    """bit-exact (floating-point outputs compared as raw bytes, NaN-proof)"""
    assert got.dtype == want.dtype and got.shape == want.shape
    assert torch.equal(got.view(torch.uint8), want.view(torch.uint8)) if got.is_floating_point() else torch.equal(got, want)


def test_fe2s2_fused_bit_identical_to_reference_cuda():
    """get_comb_hij_fused on 2048 determinants of the reference's Fe2S2 ci_space, real integrals (config 2)."""
    ref = ref_cuda(1)
    g = load("reference_cuda")
    f, x, h1e, h2e = fe2s2_inputs()
    want = ref.get_comb_hij_fused(x, h1e, h2e, f["sorb"], f["nele"], f["noA"], f["noB"]) if ref is not None else None
    for prepared in (None, False):
        comb, hmat = ops.get_comb_hij_fused(x, h1e, h2e, f["sorb"], f["nele"], f["noA"], f["noB"], prepared=prepared)
        assert digests({"comb": comb, "hmat": hmat}, "fe2s2") == {k: str(g[k]) for k in ("fe2s2/comb", "fe2s2/hmat")}
        if want is not None:
            assert_same(comb, want[0])
            assert_same(hmat, want[1])


@pytest.mark.parametrize("L,sorb,noA,noB,n", OPERATOR_CASES)
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_operators_bit_identical_to_reference_cuda(L, sorb, noA, noB, n, dtype):
    ref = ref_cuda(L)
    if rejected_by_reference(L, sorb, noA + noB):
        pytest.skip("the reference rejects this geometry (its check_sorb limits)")
    name = case_name(L, sorb, noA, noB, n, dtype)
    g = load("reference_cuda")
    x, d1, d2 = operator_inputs(sorb, noA, noB, n, dtype)
    got = operator_outputs(ops, x, d1, d2, sorb, noA, noB)
    want = {k: str(g[k]) for k in g.files if k.startswith(name + "/")}
    assert len(want) == len(got)
    assert digests(got, name) == want
    if ref is not None:
        for k, v in operator_outputs(ref, x, d1, d2, sorb, noA, noB).items():
            assert_same(got[k], v)


def record(path):
    """Write the expected digests of every case to `path`, computed on the CPU by the oracle (oracle/pynqs_oracle.c)."""
    from oracle import oracle as O

    out = {}
    f = fe2s2()
    comb, hmat = O.comb_hij_fused(f["ci"][:2048], f["h1e"], f["h2e"], f["sorb"], f["nele"], f["noA"], f["noB"])
    out.update({"fe2s2/comb": sha(comb), "fe2s2/hmat": sha(hmat)})
    for L, sorb, noA, noB, n in OPERATOR_CASES:
        if rejected_by_reference(L, sorb, noA + noB):
            continue
        nele = noA + noB
        for dtype in (np.float64, np.float32):
            bra = S.random_onvs(n, sorb, noA, noB, seed=91)
            h1e, h2e = S.random_packed_integrals(sorb, seed=92, symmetric=False, dtype=dtype)
            comb, hmat = O.comb_hij_fused(bra, h1e, h2e, sorb, nele, noA, noB)
            m = min(n, 128)
            st = O.onv_to_tensor(bra, sorb, dtype=np.float32)  # torch's default dtype, which onv_to_tensor follows
            idx, mask = O.lut(bra[O.sort_onv(bra)], comb[: min(n, 64)].reshape(-1, comb.shape[2]))
            outs = {"comb": comb, "hmat": hmat, "comb_tensor": O.comb(bra, sorb, noA, noB), "hij_3d": O.hij(bra, comb, h1e, h2e, sorb, nele),
                    "hij_2d": O.hij(bra[:m], bra[:m], h1e, h2e, sorb, nele), "onv_to_tensor": st,
                    "tensor_to_onv": O.tensor_to_onv(((st + 1) / 2).astype(np.uint8), sorb), "lut_idx": idx, "lut_mask": mask}
            out.update({f"{case_name(L, sorb, noA, noB, n, dtype)}/{k}": sha(v) for k, v in outs.items()})
    np.savez_compressed(path, **{k: np.array(v) for k, v in out.items()})
    print(f"{path}: {len(out)} digests")


if __name__ == "__main__":
    record(sys.argv[1])
