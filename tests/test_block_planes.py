"""The block kernel's key test over the bit-transposed alpha strings (one bit-sliced count per 32 keys and lane), on
geometries that take each of its forms: 5 virtual alpha orbitals (Fe2S2 sizes), 5 / 8 occupied ones, 6 of either,
4 occupied ones (the loop over any number of orbitals) and a fully occupied alpha shell (no orbital to count).

The tables hold groups of a few keys, groups that straddle 32-key chunks and groups longer than a fill of the
kernel's stage (1 024 keys), next to a random share of the samples' connected determinants, so that every group has
hits.  E_loc must match the oracle, and the Hamiltonian built on the block route must equal, entry for entry, the
one built by the per-sample kernel."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import local_energy_sample_space
from pynqs_b200.lut import WavefunctionLUT

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (spin orbitals, alpha electrons, beta electrons)
GEOMETRIES = [(40, 15, 15), (40, 5, 5), (24, 6, 6), (64, 8, 8), (28, 4, 4), (24, 12, 4)]


@pytest.fixture(scope="module", autouse=True)
def _library_loaded():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    _lib.load()


@pytest.fixture(autouse=True)
def _default_tuning():
    _lib.set_tuning()
    yield
    _lib.set_tuning()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def spin_string(orbs, spin):
    return sum(1 << (2 * int(k) + spin) for k in orbs)


def random_strings(rng, n, norb, nocc, spin):
    """up to n distinct strings of nocc of norb orbitals on the even (spin 0) or odd (spin 1) bits"""
    out = {spin_string(np.sort(rng.choice(norb, nocc, replace=False)), spin) for _ in range(3 * n)}
    return sorted(out)[:n]


def beta_singles(b, norb):
    occ = [k for k in range(norb) if b >> (2 * k + 1) & 1]
    vir = [k for k in range(norb) if not b >> (2 * k + 1) & 1]
    return [b ^ (1 << (2 * i + 1)) ^ (1 << (2 * a + 1)) for i in occ for a in vir]


def to_u8(words):
    return np.array(words, dtype=np.uint64).view(np.uint8).reshape(-1, 8)


def make_case(sorb, noA, noB, seed=2024):
    """samples: 40 on one beta string, 12 on a second, 6 on random ones (repeated when the alpha shell is full);
    table: the samples, a third of their connected determinants, and groups of 3 ... 1 100 keys on the first beta
    string and on some of its single excitations"""
    rng = np.random.default_rng(seed)
    norb = sorb // 2
    betas = random_strings(rng, 8, norb, noB, 1)
    samples = []
    for b, n in zip(betas, (40, 12, 1, 1, 1, 1, 1, 1)):
        alphas = random_strings(rng, n, norb, noA, 0)
        samples += [a | b for a in alphas] * (n // len(alphas))
    x = to_u8(samples)
    comb = O.comb(np.unique(x, axis=0), sorb, noA, noB).reshape(-1, 8)
    extra = []
    sizes = (3, 17, 45, 70, 300, 1100)
    for b, n in zip([betas[0]] + beta_singles(betas[0], norb)[:: max(1, noB * (norb - noB) // 8)], sizes * 2):
        extra += [a | b for a in random_strings(rng, n, norb, noA, 0)]
    keys = np.unique(np.concatenate([x, comb[rng.permutation(comb.shape[0])[: comb.shape[0] // 3]], to_u8(extra)]), axis=0)
    return x, keys


@pytest.mark.parametrize("parts", [1, 4], ids=["whole_tiles", "4_parts"])
@pytest.mark.parametrize("sorb,noA,noB", GEOMETRIES)
def test_block_route_against_oracle_and_per_sample_kernel(sorb, noA, noB, parts):
    x, keys = make_case(sorb, noA, noB)
    nele = noA + noB
    psi = S.random_psi(keys.shape[0], seed=sorb + noA)
    h1e, h2e = S.random_packed_integrals(sorb, seed=17, symmetric=True)
    lut = WavefunctionLUT(dev(keys), dev(psi), sorb, DEV, rank=0, world_size=1)
    xd, h1d, h2d = dev(x), dev(h1e), dev(h2e)

    def block_route():
        _lib.set_tuning()
        _lib.set_tuning("block_min_samples", 1)
        _lib.set_tuning("block_min_group", 4)
        _lib.set_tuning("eval_tiles", 2)
        _lib.set_tuning("block_parts", parts)

    block_route()
    eloc, _, _ = local_energy_sample_space(xd, h1d, h2d, lut, sorb, nele, noA, noB)
    order = O.sort_onv(keys)
    first = np.unique(x, axis=0, return_index=True)[1]
    want = O.eloc_sample_space(x[first], h1e, h2e, keys[order], psi[order], sorb, nele, noA, noB)
    np.testing.assert_allclose(eloc.cpu().numpy()[first], want, rtol=1e-12, atol=0)

    got = ops.sample_space_hamiltonian(xd, h1d, h2d, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    _lib.set_tuning()
    _lib.set_tuning("block_enable", 0)
    ref = ops.sample_space_hamiltonian(xd, h1d, h2d, sorb, nele, noA, noB, lut.bra_key, lut.group_index)
    for a, b in zip(got, ref):
        assert torch.equal(a, b)
    assert ref[1].numel() > x.shape[0]  # rows hold more than the diagonal
