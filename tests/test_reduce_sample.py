"""The stochastic / semi-stochastic REDUCE (get_comb_hij_sampled, csrc/reduce_sample.cu) element for element against a host
reference: one-, two- and three-word ONVs, float64 and float32 integrals, rows per sample below one 256-row chunk of the
kernel, on a chunk edge, one past it and the 571 876 rows of an H50 sample; eps from 0 to above max |H|; eps_sample from 1
to 8192; the caller's draws, and the seeded Philox stream replayed draw by draw; E_loc through reduce_eloc.

Host reference of one call, per sample, from the oracle's Hmat in the integrals' dtype T:
  kept rows: eps > 0 and |H| >= T(eps) (torch compares in the tensor's dtype, as O.reduced and get_comb_hij_reduced do);
  w = |H| (as float64) on the other rows, S = fsum(w), the inclusive prefix of w in long double;
  output: kept rows (ascending m), then drawn rows (ascending m), flat index s * M + m; a kept value is H (bit for bit), a
  drawn value sign(H) * S * count / eps_sample.
Seeded draws: Philox4x32-10 with key (seed & 0xffffffff, seed >> 32) and counter (j >> 1, s & 0xffffffff, s >> 32, 0x5eed)
for draw j of the call's sample s; words (x, y) for even j, (z, w) for odd j; u = ((hi >> 5) 2^26 + (lo >> 6) + 0.5) 2^-53;
the target t = u S lands on the row with before <= t < before + w."""
import math

import numpy as np
import pytest
import torch

from oracle import oracle as O
from pynqs_b200 import C_extension as ops
from pynqs_b200 import _lib
from pynqs_b200 import synthetic as S
from pynqs_b200.energy import local_energy_reduced

from util import fe2s2, ops_inputs, toy_amplitude

DEV = "cuda:0"
gpu = pytest.mark.gpu
CHUNK = 256  # kRsThreads: the kernel scans a sample's rows in chunks of this many
U32 = np.uint64(0xFFFFFFFF)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (run with -m gpu on the B200 box)")
    _lib.load()  # fails loudly if libpynqs_b200.so is missing: there is no fallback


# ---- host replay of the generator -----------------------------------------------------------------------------------
def philox4x32_10(key, ctr):
    """Philox4x32-10 (Salmon et al., SC'11) on uint64 arrays that hold 32-bit words: key (k0, k1) and counter (c0, c1, c2, c3)
    broadcast against each other; returns the four output words"""
    k0, k1 = (np.asarray(k, dtype=np.uint64) for k in key)
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) for c in ctr)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & U32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & U32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & U32, (k1 + np.uint64(0xBB67AE85)) & U32
    return c0, c1, c2, c3


def uniforms(seed, samples, n_draw):
    """the kernel's uniforms in (0, 1) of the given call-local sample indices: float64 [len(samples), n_draw]"""
    seed = int(seed) & (2**64 - 1)
    j = np.arange(n_draw, dtype=np.uint64)[None, :]
    s = np.asarray(samples, dtype=np.uint64)[:, None]
    x, y, z, w = philox4x32_10((seed & 0xFFFFFFFF, seed >> 32), (j >> np.uint64(1), s & U32, s >> np.uint64(32), 0x5EED))
    odd = (j & np.uint64(1)) == 1
    hi, lo = np.where(odd, z, x), np.where(odd, w, y)
    return ((hi >> np.uint64(5)).astype(np.float64) * 67108864.0 + (lo >> np.uint64(6)).astype(np.float64) + 0.5) * 2.0**-53


# ---- host reference ---------------------------------------------------------------------------------------------------
def keep_mask(hmat, eps):
    return np.abs(hmat) >= hmat.dtype.type(eps) if eps > 0 else np.zeros(hmat.shape, dtype=bool)


def sub_eps_weights(hmat, eps):
    return np.where(keep_mask(hmat, eps), 0.0, np.abs(hmat).astype(np.float64))


class Reference:
    """What one get_comb_hij_sampled call must return, from the oracle's comb / Hmat of its samples (module docstring).
    `draws` [n, eps_sample]: the caller's row indices; otherwise `seed` is replayed.  `near` lists the seeded draws whose
    target lies within 2 scan_rtol(M) S of an interval boundary (sample, row, neighbouring row or -1): the device's target
    and running sums each differ from the exact ones by up to scan_rtol(M) S, so such a draw may land on either neighbour."""

    def __init__(self, comb, hmat, eps, n_draw, *, seed=None, draws=None):
        n, M = hmat.shape
        self.comb, self.hmat, self.n_draw, self.M = comb, hmat, n_draw, M
        self.keep = keep_mask(hmat, eps)
        w = sub_eps_weights(hmat, eps)
        self.S = np.array([math.fsum(r) for r in w])
        self.counts = np.zeros((n, M), dtype=np.int64)
        self.near = []
        if draws is not None:
            draws = np.asarray(draws)
            for s in range(n):
                self.counts[s] = np.bincount(draws[s], minlength=M)
            assert not ((self.counts > 0) & (w == 0)).any(), "draws on a kept or zero row: not what torch.multinomial returns"
            return
        u = uniforms(seed, np.arange(n), n_draw)
        for s in range(n):
            if self.S[s] == 0:
                continue  # nothing to draw from
            pre = np.cumsum(w[s].astype(np.longdouble))
            t = u[s].astype(np.longdouble) * np.longdouble(self.S[s])
            rows = np.minimum(np.searchsorted(pre, t, side="right"), M - 1)
            self.counts[s] = np.bincount(rows, minlength=M)
            tol = 2 * scan_rtol(M) * self.S[s]
            lower = np.where(rows > 0, pre[rows - 1], 0)
            nz = np.nonzero(w[s])[0]  # the rows a draw can land on; k: the position of each draw's row among them
            k = np.searchsorted(nz, rows)
            for i in np.nonzero((t - lower < tol) & (lower > 0))[0]:
                self.near.append((s, int(rows[i]), int(nz[k[i] - 1])))
            for i in np.nonzero(pre[rows] - t < tol)[0]:
                self.near.append((s, int(rows[i]), int(nz[k[i] + 1]) if k[i] + 1 < nz.size else -1))

    def rows(self, s):
        return np.nonzero(self.keep[s])[0], np.nonzero(self.counts[s])[0]

    def drawn_values(self, s, rows, counts):
        """sign(H) * S * count / eps_sample, exactly (long double)"""
        h = self.hmat[s, rows].astype(np.float64)
        return np.where(h < 0, -1, 1) * (np.longdouble(self.S[s]) * counts.astype(np.longdouble) / self.n_draw)


def scan_rtol(M):
    """bound on the relative error (to S) of the device's S, running sums, targets and drawn float64 values: a 32-lane shuffle
    scan per warp, then each 256-row chunk's eight warp sums added to the running total one after another (8 ceil(M / 256) + 5
    additions of positive terms), and a few roundings more forming u S and S / eps_sample * count"""
    return (8 * -(-M // CHUNK) + 16) * 2.0**-53


def check_call(out, ref):
    """one get_comb_hij_sampled call against its host reference, sample by sample"""
    x, hij, idx, off = (t.cpu().numpy() for t in out)
    n, M = ref.hmat.shape
    dtype = ref.hmat.dtype
    near = {}  # sample -> (rows a boundary draw may land on, number of such draws)
    for s, r, r2 in ref.near:
        rows, k = near.get(s, (set(), 0))
        near[s] = (rows | {r, r2}, k + 1)
    assert off[0] == 0 and np.all(np.diff(off) >= 0) and off[n] == idx.size == hij.size == x.shape[0]
    assert hij.dtype == dtype
    for s in range(n):
        kept, drawn = ref.rows(s)
        k = slice(off[s], off[s + 1])
        gi, gx, gh = idx[k] - s * M, x[k], hij[k]
        nk = kept.size
        # kept rows first: determinants, flat indices, values bit for bit
        np.testing.assert_array_equal(gi[:nk], kept, err_msg=f"sample {s}: kept rows")
        np.testing.assert_array_equal(gx[:nk], ref.comb[s, kept])
        np.testing.assert_array_equal(gh[:nk].view(np.uint8), ref.hmat[s, kept].view(np.uint8))
        # then the drawn rows, ascending, with their counts recovered from the values
        dr, dh = gi[nk:], gh[nk:]
        assert np.all(np.diff(dr) > 0) and not ref.keep[s, dr].any() and np.all(ref.hmat[s, dr] != 0), f"sample {s}"
        np.testing.assert_array_equal(gx[nk:], ref.comb[s, dr])
        if ref.S[s] == 0:
            assert dr.size == 0, f"sample {s}: S = 0, yet {dr.size} rows drawn"
            continue
        cnt = np.rint(np.abs(dh.astype(np.float64)) * ref.n_draw / ref.S[s]).astype(np.int64)
        assert np.all(cnt >= 1)
        assert cnt.sum() == ref.n_draw, f"sample {s}: {cnt.sum()} draws counted, {ref.n_draw} made"
        if s in near:  # a draw on an interval boundary may have gone to either neighbour
            got = np.zeros(M, dtype=np.int64)
            got[dr] = cnt
            moved = np.nonzero(got != ref.counts[s])[0]
            assert set(moved.tolist()) <= near[s][0], f"sample {s}: counts differ at rows {moved} away from the boundaries {near[s]}"
            assert np.abs(got - ref.counts[s]).sum() <= 2 * near[s][1]
        else:
            np.testing.assert_array_equal(dr, drawn, err_msg=f"sample {s}: drawn rows")
            np.testing.assert_array_equal(cnt, ref.counts[s, drawn], err_msg=f"sample {s}: counts")
        exact = ref.drawn_values(s, dr, cnt)
        err = np.abs(dh.astype(np.longdouble) - exact)
        if dtype == np.float64:
            bound = scan_rtol(M) * np.abs(exact)
        else:  # the device rounds its double once to float32
            bound = np.spacing(np.abs(exact).astype(np.float32)).astype(np.longdouble)
        assert np.all(err <= bound), f"sample {s}: drawn values off by up to {float(np.max(err / np.abs(exact))):.3g} relative"
    if not near:
        kept_sizes = ref.keep.sum(1)
        want = np.concatenate([[0], np.cumsum(kept_sizes + (ref.counts > 0).sum(1))])
        np.testing.assert_array_equal(off, want)


def check_kept_equals_reduced(c, out, ref, eps):
    """the kept rows are get_comb_hij_reduced's at the same eps: determinants, values and flat indices"""
    x, hij, idx, off = (t.cpu().numpy() for t in out)
    sel = np.concatenate([np.arange(off[s], off[s] + ref.keep[s].sum()) for s in range(off.size - 1)]).astype(np.int64)
    rx, rh, ri, ro = (t.cpu().numpy() for t in ops.get_comb_hij_reduced(c["d_bra"], c["d_h1e"], c["d_h2e"], c["sorb"], c["nele"],
                                                                       c["noA"], c["noB"], eps))
    np.testing.assert_array_equal(np.diff(ro), ref.keep.sum(1))
    np.testing.assert_array_equal(idx[sel], ri)
    np.testing.assert_array_equal(x[sel], rx)
    np.testing.assert_array_equal(hij[sel].view(np.uint8), rh.view(np.uint8))


# ---- geometries ---------------------------------------------------------------------------------------------------------
def _synthetic(sorb, noA, noB, n, dtype, seed):
    bra = S.random_onvs(n, sorb, noA, noB, seed=seed)
    h1e, h2e = S.random_packed_integrals(sorb, seed=seed + 1, symmetric=True, dtype=dtype)
    return dict(bra=bra, h1e=h1e, h2e=h2e, sorb=sorb, noA=noA, noB=noB)


def _fe2s2(dtype):
    f = fe2s2()
    return dict(bra=f["ci"][::1153][:16], h1e=f["h1e"].astype(dtype), h2e=f["h2e"].astype(dtype), sorb=f["sorb"], noA=f["noA"],
                noB=f["noB"])


def _golden(name, n, dtype):
    c = ops_inputs(name)
    return dict(bra=c["bra"][:n], h1e=c["h1e"].astype(dtype), h2e=c["h2e"].astype(dtype), sorb=c["sorb"], noA=c["noA"], noB=c["noB"])


# name: (inputs, L, M); M = rows per sample, the kernel scans them in chunks of 256
GEOMETRIES = {
    "8so_2a1b": (lambda: _synthetic(8, 2, 1, 20, np.float64, 801), 1, 21),  # fewer rows than one chunk
    "36so_6a1b": (lambda: _synthetic(36, 6, 1, 12, np.float64, 3601), 1, 2304),  # exactly 9 chunks
    "42so_5a5b_f32": (lambda: _synthetic(42, 5, 5, 8, np.float32, 4201), 1, 8961),  # 35 chunks + 1 row
    "fe2s2": (lambda: _fe2s2(np.float64), 1, 7876),  # production integrals
    "fe2s2_f32": (lambda: _fe2s2(np.float32), 1, 7876),
    "74so_5a0b_f32": (lambda: _synthetic(74, 5, 0, 8, np.float32, 7401), 2, 5121),  # 20 chunks + 1 row, one spin sector
    "h50": (lambda: _golden("ops_c4_h50_100sorb", 1, np.float64), 2, 571876),  # long rows
    "l3_132": (lambda: _golden("ops_l3_132sorb_3a2b", 3, np.float64), 3, 32385),  # three-word ONVs
    "l3_132_f32": (lambda: _golden("ops_l3_132sorb_3a2b", 3, np.float32), 3, 32385),
}
_cases = {}


def case(name, device=True):
    """inputs, the oracle's comb / Hmat and (device=True) the inputs on the GPU, made once per module"""
    if name not in _cases:
        make, L, M = GEOMETRIES[name]
        c = make()
        c["nele"] = c["noA"] + c["noB"]
        assert c["bra"].shape[1] == 8 * L
        c["comb"], c["hmat"] = O.comb_hij_fused(c["bra"], c["h1e"], c["h2e"], c["sorb"], c["nele"], c["noA"], c["noB"])
        assert c["hmat"].shape[1] == M and c["hmat"].dtype == c["h1e"].dtype
        nz = np.sort(np.abs(c["hmat"][c["hmat"] != 0]))
        c["nz"] = nz  # the nonzero |H| of the call, ascending, in the integrals' dtype
        _cases[name] = c
    c = _cases[name]
    if device and "d_bra" not in c:
        c["d_bra"], c["d_h1e"], c["d_h2e"] = dev(c["bra"]), dev(c["h1e"]), dev(c["h2e"])
    return c


def quantile_eps(c, q):
    """an element of the call's nonzero |H| (float64), or 0 for q = 0"""
    return 0.0 if q == 0 else float(c["nz"][int(q * (c["nz"].size - 1))])


def sampled(c, eps, n_draw, *, seed=None, draws=None, rows=None):
    bra = c["d_bra"] if rows is None else c["d_bra"][rows]
    return ops.get_comb_hij_sampled(bra, c["d_h1e"], c["d_h2e"], c["sorb"], c["nele"], c["noA"], c["noB"], eps, n_draw, seed=seed,
                                    draws=draws)


def multinomial_draws(hmat, eps, n_draw, gen_seed):
    """what the reference's torch.multinomial returns for p = sub-eps |H| / S (host generator)"""
    w = torch.from_numpy(sub_eps_weights(hmat, eps))
    return torch.multinomial(w / w.sum(1, keepdim=True), n_draw, replacement=True, generator=torch.Generator().manual_seed(gen_seed))


def run_checked(c, eps, n_draw, mode, *, seed=0x5A17_0000_0000_0001, gen_seed=5):
    """one call in `draws` or `seeded` mode, checked element for element; returns (outputs, reference)"""
    if mode == "draws":
        d = multinomial_draws(c["hmat"], eps, n_draw, gen_seed)
        out = sampled(c, eps, n_draw, draws=dev(d.numpy()))
        ref = Reference(c["comb"], c["hmat"], eps, n_draw, draws=d.numpy())
    else:
        out = sampled(c, eps, n_draw, seed=seed)
        ref = Reference(c["comb"], c["hmat"], eps, n_draw, seed=seed)
    check_call(out, ref)
    if eps > 0:
        check_kept_equals_reduced(c, out, ref, eps)
    return out, ref


def assert_same_bytes(a, b):
    """equal tensors, byte for byte (NaN included)"""

    def raw(t):
        t = torch.view_as_real(t) if t.is_complex() else t
        return t.view(torch.uint8) if t.dtype.is_floating_point else t

    for u, v in zip(a, b):
        assert u.dtype == v.dtype and u.shape == v.shape
        assert torch.equal(raw(u), raw(v))


# ---- host-only: the replay and the reference ----------------------------------------------------------------------------
def test_philox_known_answers():
    """Random123's known-answer vectors for Philox4x32-10: pins the host replay independently of the kernel"""
    f = 0xFFFFFFFF
    vectors = [
        ((0, 0), (0, 0, 0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((f, f), (f, f, f, f), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0xA4093822, 0x299F31D0), (0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for key, ctr, want in vectors:
        assert tuple(int(v) for v in philox4x32_10(key, ctr)) == want
    # broadcasting over counters gives the same words as one call per counter
    ks = (0x12345678, 0x9ABCDEF0)
    batch = philox4x32_10(ks, (np.arange(4, dtype=np.uint64), 7, 0, 0x5EED))
    for i in range(4):
        assert tuple(int(v[i]) for v in batch) == tuple(int(v) for v in philox4x32_10(ks, (i, 7, 0, 0x5EED)))


def test_uniforms_layout():
    """draw j of sample s: words (x, y) of counter (j >> 1, s lo, s hi, 0x5eed) for even j, (z, w) for odd j; u in (0, 1),
    ((hi >> 5) 2^26 + (lo >> 6) + 1/2) 2^-53 rounded to double; every sample its own stream"""
    seed = (0xDEADBEEF << 32) | 0x01234567
    u = uniforms(seed, [(1 << 32) + 5], 6)[0]  # a sample index with a high word
    for j in range(6):
        x, y, z, w = (int(v) for v in philox4x32_10((0x01234567, 0xDEADBEEF), (j >> 1, 5, 1, 0x5EED)))
        hi, lo = (z, w) if j & 1 else (x, y)
        assert u[j] == (float((hi >> 5) * 2**26 + (lo >> 6)) + 0.5) / 2**53 and 0.0 < u[j] < 1.0
    all_u = uniforms(seed, np.arange(64), 4096)
    assert np.all((all_u > 0) & (all_u < 1))
    assert len({r.tobytes() for r in all_u}) == 64  # every sample its own stream
    assert abs(all_u.mean() - 0.5) < 5 * np.sqrt(1 / 12 / all_u.size)


@pytest.mark.parametrize("name", ["8so_2a1b", "fe2s2", "fe2s2_f32"])
def test_reference_kept_set_is_the_oracles(name):
    """the reference's kept rows are O.reduced's at the same eps, including eps = nextafter(v, inf) for an |H| value v,
    which float32 keeps and float64 samples"""
    c = case(name, device=False)
    nz = c["nz"]
    v = nz[nz.size // 2]
    for eps in (quantile_eps(c, 0.9), float(nz[-1]) * 2, float(nz[0]) / 2, float(np.nextafter(np.float64(v), np.inf))):
        ref = Reference(c["comb"], c["hmat"], eps, 64, seed=3)
        x, h, idx, off = O.reduced(c["bra"], c["h1e"], c["h2e"], c["sorb"], c["nele"], c["noA"], c["noB"], eps)
        np.testing.assert_array_equal(idx, np.nonzero(ref.keep.reshape(-1))[0])
        np.testing.assert_array_equal(off, np.concatenate([[0], np.cumsum(ref.keep.sum(1))]))
        np.testing.assert_array_equal(h, c["hmat"].reshape(-1)[idx])
        np.testing.assert_array_equal(x, c["comb"].reshape(c["hmat"].size, -1)[idx])
    at_v = np.abs(c["hmat"]) == v
    assert ref.keep[at_v].all() == (c["hmat"].dtype == np.float32)


def test_reference_draws():
    """seeded: every sample with S > 0 gets exactly eps_sample draws, none on a kept or zero row, and the draws follow
    p = w / S; S = 0 (eps below the smallest nonzero |H|): nothing drawn"""
    c = case("fe2s2", device=False)
    eps, n_draw = quantile_eps(c, 0.9), 8192
    ref = Reference(c["comb"], c["hmat"], eps, n_draw, seed=99)
    w = sub_eps_weights(c["hmat"], eps)
    assert np.all(ref.S > 0) and np.all(ref.counts.sum(1) == n_draw)
    assert not ((ref.counts > 0) & (w == 0)).any() and not ref.near
    p = w / ref.S[:, None]
    # the most likely rows of each sample: frequency within 5 standard errors of p
    for s in range(w.shape[0]):
        top = np.argsort(p[s])[-5:]
        se = np.sqrt(p[s, top] * (1 - p[s, top]) / n_draw)
        assert np.all(np.abs(ref.counts[s, top] / n_draw - p[s, top]) <= 5 * se)
    none = Reference(c["comb"], c["hmat"], float(c["nz"][0]) / 2, n_draw, seed=99)
    assert np.all(none.S == 0) and not none.counts.any() and none.keep.all() == (c["nz"].size == c["hmat"].size)


# ---- A. every geometry, the caller's draws and the seeded stream -------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["draws", "seeded"])
@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_geometries_against_the_host_reference(cuda, name, mode):
    c = case(name)
    run_checked(c, quantile_eps(c, 0.9), 1000, mode)


# ---- B. eps ---------------------------------------------------------------------------------------------------------------
EPS_GEOMETRIES = ["fe2s2", "fe2s2_f32", "42so_5a5b_f32", "74so_5a0b_f32", "l3_132"]


@gpu
@pytest.mark.parametrize("q", [0.0, 0.5, 0.99])
@pytest.mark.parametrize("name", EPS_GEOMETRIES)
def test_eps_zero_and_quantiles(cuda, name, q):
    c = case(name)
    for mode in ("draws", "seeded"):
        run_checked(c, quantile_eps(c, q), 500, mode)


@gpu
@pytest.mark.parametrize("name", EPS_GEOMETRIES)
def test_eps_above_every_element_is_eps_zero(cuda, name):
    """nothing reaches eps: the same bits as the purely stochastic call, for the same seed and for the same draws"""
    c = case(name)
    big = float(c["nz"][-1]) * 2
    zero_seeded, _ = run_checked(c, 0.0, 700, "seeded", seed=41)
    big_seeded, ref = run_checked(c, big, 700, "seeded", seed=41)
    assert not ref.keep.any()
    assert_same_bytes(zero_seeded, big_seeded)
    d = dev(multinomial_draws(c["hmat"], 0.0, 700, 8).numpy())
    assert_same_bytes(sampled(c, 0.0, 700, draws=d), sampled(c, big, 700, draws=d))


@gpu
@pytest.mark.parametrize("name", EPS_GEOMETRIES)
def test_eps_below_every_element_draws_nothing(cuda, name):
    """S = 0 (every row kept or exactly zero): the kept rows only, nothing drawn, no NaN; the reference would fail inside
    torch.multinomial here, so this pins the library's own behaviour"""
    c = case(name)
    eps = float(c["nz"][0]) / 2
    out, ref = run_checked(c, eps, 1000, "seeded", seed=17)
    assert np.all(ref.S == 0)
    assert int(out[3][-1]) == int(ref.keep.sum()) and torch.isfinite(out[1]).all()


@gpu
@pytest.mark.parametrize("name", ["fe2s2_f32", "42so_5a5b_f32", "74so_5a0b_f32", "l3_132_f32", "fe2s2"])
def test_eps_is_compared_in_the_integrals_dtype(cuda, name):
    """eps = nextafter(v, +inf) for an element's |H| = v: float32 rounds eps to v and keeps that row, as torch.where, O.reduced
    and get_comb_hij_reduced do; float64 samples it"""
    c = case(name)
    v = c["nz"][c["nz"].size // 2]
    eps = float(np.nextafter(np.float64(v), np.inf))
    at_v = np.abs(c["hmat"]) == v
    for mode in ("draws", "seeded"):
        _, ref = run_checked(c, eps, 1000, mode)
        assert ref.keep[at_v].all() == (c["hmat"].dtype == np.float32)


# ---- C. eps_sample ----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["draws", "seeded"])
@pytest.mark.parametrize("n_draw", [1, 2, 3, 64, 1000, 4096, 4097, 8192])  # from 4097 on the sorted draws need > 48 KB of shared memory
def test_eps_sample(cuda, n_draw, mode):
    c = case("fe2s2")
    run_checked(c, quantile_eps(c, 0.9), n_draw, mode, seed=n_draw * 1_000_003)


@gpu
def test_eps_sample_above_8192_is_refused_before_any_launch(cuda):
    c = case("fe2s2")
    l0 = _lib.launch_count()
    with pytest.raises(ValueError, match="8192"):
        sampled(c, 1e-3, 8193, seed=1)
    with pytest.raises(ValueError, match="8192"):
        sampled(c, 1e-3, 8193, draws=torch.zeros((c["bra"].shape[0], 8193), dtype=torch.int64, device=DEV))
    assert _lib.launch_count() == l0


# ---- D. the seeded stream -----------------------------------------------------------------------------------------------------
@gpu
def test_seeded_stream_depends_on_seed_and_sample_only(cuda):
    """same seed: the same bytes; the first 5 samples of a call are those of a call on the first 5 alone (the stream does not
    depend on the launch geometry); two copies of one determinant in a call draw differently"""
    c = case("fe2s2")
    eps, n_draw, seed = quantile_eps(c, 0.9), 1000, 0x0BAD_5EED_0000_0007
    a = sampled(c, eps, n_draw, seed=seed)
    assert_same_bytes(a, sampled(c, eps, n_draw, seed=seed))
    head = sampled(c, eps, n_draw, seed=seed, rows=slice(0, 5))
    k = int(a[3][5])
    assert_same_bytes(head, (a[0][:k], a[1][:k], a[2][:k], a[3][:6]))
    twin = sampled(c, eps, n_draw, seed=seed, rows=[3, 3])
    ref = Reference(c["comb"][[3, 3]], c["hmat"][[3, 3]], eps, n_draw, seed=seed)
    check_call(twin, ref)
    assert not np.array_equal(ref.counts[0], ref.counts[1])
    other = sampled(c, eps, n_draw, seed=seed ^ (1 << 40))  # the key's high word matters
    assert not torch.equal(other[2], a[2])


# ---- E. E_loc through reduce_eloc / local_energy_reduced --------------------------------------------------------------------
class PsiTable:
    """toy_amplitude of every determinant the samples connect to, evaluated once: psi as a function of the determinant
    alone, whatever batch it is asked for in"""

    def __init__(self, comb, sorb, cplx):
        assert comb.shape[2] == 8  # one-word ONVs: a determinant is its uint64 key
        self.keys = np.unique(np.ascontiguousarray(comb).view(np.uint64).reshape(-1))
        self.vals = toy_amplitude(torch.from_numpy(O.onv_to_tensor(self.keys.view(np.uint8).reshape(-1, 8), sorb)), sorb, cplx).numpy()

    def host(self, x):
        q = np.ascontiguousarray(x).view(np.uint64).reshape(-1)
        pos = np.minimum(np.searchsorted(self.keys, q), self.keys.size - 1)
        assert np.array_equal(self.keys[pos], q)
        return self.vals[pos]

    def __call__(self, xk):
        return torch.from_numpy(self.host(xk.cpu().numpy())).to(xk.device)


def eloc_reference(ref, psi):
    """E_loc[s] = sum over the kept and drawn rows of (psi_k / psi_0) h_k with the reference's h (psi_0 = 0 when row 0 is
    neither kept nor drawn, as the reference's scatter into zeros gives), and psi_0"""
    n = ref.hmat.shape[0]
    cplx = np.iscomplexobj(psi.vals)
    eloc = np.empty(n, dtype=complex if cplx else float)
    psi0 = np.zeros(n, dtype=eloc.dtype)
    for s in range(n):
        kept, drawn = ref.rows(s)
        h = np.concatenate([ref.hmat[s, kept].astype(np.float64), ref.drawn_values(s, drawn, ref.counts[s, drawn]).astype(np.float64)])
        rows = np.concatenate([kept, drawn])
        p = psi.host(ref.comb[s, rows])
        if 0 in rows:
            psi0[s] = p[np.nonzero(rows == 0)[0][0]]
        with np.errstate(divide="ignore", invalid="ignore"):
            q = p / psi0[s]
            terms = [q.real * h] + ([q.imag * h] if cplx else [])
            parts = [math.fsum(t) if np.all(np.isfinite(t)) else np.sum(t) for t in terms]
        eloc[s] = complex(parts[0], parts[1]) if cplx else parts[0]
    return eloc, psi0


def assert_eloc(got, want):
    """rtol 1e-12 where the reference is finite; where it is not, the same inf (with its sign) or NaN in each part"""
    fin = np.isfinite(want)
    np.testing.assert_array_equal(np.isfinite(got), fin)
    np.testing.assert_array_equal(got[~fin].real, want[~fin].real)
    np.testing.assert_array_equal(got[~fin].imag, want[~fin].imag)
    assert np.all(np.abs(got[fin] - want[fin]) <= 1e-12 * np.abs(want[fin])), np.max(np.abs(got[fin] - want[fin]) / np.abs(want[fin]))


@gpu
@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("mode", ["draws", "seeded"])
@pytest.mark.parametrize("diag", ["kept", "sampled"])
def test_local_energy_against_a_host_sum(cuda, diag, mode, cplx):
    """E_loc of local_energy_reduced in batches of 7 (the seed of each batch offset by its start, its samples counted from 0)
    against a host fsum over the reference's kept and drawn rows.  The diagonal is kept (eps below |H_00|), or sub-eps with
    one draw per sample (eps above every |H|), drawn in some samples and not in others; there psi_0 = 0 and E_loc is inf / NaN
    exactly where the reference's division gives it.  With the caller's draws, batches of 7 give the bits of one batch."""
    f = fe2s2()
    n, batch = 24, 7
    c = dict(bra=f["ci"][5::701][:n], h1e=f["h1e"], h2e=f["h2e"], sorb=f["sorb"], noA=f["noA"], noB=f["noB"], nele=f["nele"])
    comb, hmat = O.comb_hij_fused(c["bra"], c["h1e"], c["h2e"], c["sorb"], c["nele"], c["noA"], c["noB"])
    psi = PsiTable(comb, c["sorb"], cplx)
    nz = np.sort(np.abs(hmat[hmat != 0]))
    eps, n_draw = (float(nz[int(0.9 * nz.size)]), 64) if diag == "kept" else (float(nz[-1]) * 2, 1)
    batches = range(0, n, batch)
    if mode == "draws":
        d = multinomial_draws(hmat, eps, n_draw, 13)
        if diag == "sampled":  # every third sample draws from the off-diagonal rows only
            d[::3] = multinomial_draws(hmat[::3, 1:], eps, n_draw, 14) + 1
        refs = [Reference(comb[b : b + batch], hmat[b : b + batch], eps, n_draw, draws=d[b : b + batch].numpy()) for b in batches]
        kw = dict(draws=dev(d.numpy()))
    else:
        for seed in range(1000, 1100):  # the first seed whose draws cover both cases of the diagonal
            refs = [Reference(comb[b : b + batch], hmat[b : b + batch], eps, n_draw, seed=seed + b) for b in batches]
            diag_drawn = np.concatenate([r.counts[:, 0] > 0 for r in refs])
            if diag == "kept" or (diag_drawn.any() and not diag_drawn.all()):
                break
        kw = dict(seed=seed)
    keep0 = np.concatenate([r.keep[:, 0] for r in refs])
    drawn0 = np.concatenate([r.counts[:, 0] > 0 for r in refs])
    if diag == "kept":
        assert keep0.all()
    else:
        assert not keep0.any() and drawn0.any() and not drawn0.all()
    assert not any(r.near for r in refs)
    want = [eloc_reference(r, psi) for r in refs]
    want_eloc, want_psi0 = np.concatenate([w[0] for w in want]), np.concatenate([w[1] for w in want])
    dtype = torch.complex128 if cplx else torch.double
    args = (dev(c["bra"]), dev(c["h1e"]), dev(c["h2e"]), psi, c["sorb"], c["nele"], c["noA"], c["noB"])
    eloc, _, psi_x = local_energy_reduced(*args, dtype=dtype, eps=eps, eps_sample=n_draw, batch=batch, **kw)
    assert_eloc(eloc.cpu().numpy(), want_eloc)
    np.testing.assert_array_equal(psi_x.cpu().numpy(), want_psi0)
    assert np.isfinite(want_eloc).sum() == (keep0 | drawn0).sum()
    if mode == "draws":
        one, _, psi_one = local_energy_reduced(*args, dtype=dtype, eps=eps, eps_sample=n_draw, batch=n, **kw)
        assert_same_bytes((eloc, psi_x), (one, psi_one))
