"""Every NTT plan, both twiddle-factor paths and the witness map against the C++ oracle (oracle/c/oracle.cpp, 64-bit limbs,
textbook iterative radix-2: no code in common with the kernels), compared on raw Montgomery limbs.

* b2s_ntt at every log_n in 0..27 on both curves (BN254's two-adicity is 28; the backend stops at 2^27): all four modes
  up to 2^22 -- one pass up to 2^10, two up to 2^18, three beyond -- and one or two modes per size from 2^23, rotated
  so that each mode meets a radix-9 plan (2^25 = 9+8+8, 2^26 = 9+9+8, 2^27 = 9+9+9) on each curve.  The host-buffer
  path must give what the device path gives.
* The composed factors (B2S_NTT_FULL=0: two-level power tables, what runs when the full-size tables do not fit) must
  give, bit for bit, what the full-size tables give, at every size 1..27 in every mode and in witness_map, where they
  also switch the merged scalings (alpha = 1, beta = Zinv / N) for Zinv / Zinv.
* witness_map with dense random assignments that satisfy nothing, on both curves, up to BN254's radix-9 plan 2^25.
* The distributed schedule (witness_map_sim) at every cut dist_supported accepts, and the first cut beyond it refused.

Every input carries the edge values 0, 1, -1 (Montgomery forms) and the largest canonical limb value r - 1 at index 0,
at N - 1, on both sides of tile boundaries (multiples of 1024) and inside a run of zeros."""
import numpy as np
import pytest

from oracle import cnative
from oracle.params import BLS12_381, BN254
from tests.util import pack_u32, random_fr_limbs

pytestmark = pytest.mark.gpu
CURVES = [BLS12_381, BN254]
CURVE_IDS = ["bls12_381", "bn254"]
MODES = {"fwd": (False, False), "inv": (True, False), "coset": (False, True), "coset_inv": (True, True)}
TILE = 1024
ALL_MODES_MAX = 22
# 2^23..2^27: the modes compared with the oracle, per curve (a 2^27 oracle transform takes tens of seconds on the host)
LARGE_MODES = {
    0: {23: ["fwd"], 24: ["inv"], 25: ["coset", "coset_inv"], 26: ["fwd"], 27: ["inv"]},
    1: {23: ["coset_inv"], 24: ["coset"], 25: ["fwd", "inv"], 26: ["coset"], 27: ["coset_inv"]},
}


@pytest.fixture(autouse=True)
def _full_tables_default(monkeypatch):
    """Every test starts on the default (full-size table) path; the composed path is opted into inside a test."""
    monkeypatch.delenv("B2S_NTT_FULL", raising=False)


@pytest.fixture(scope="module", params=[0, 1], ids=CURVE_IDS)
def be(request):
    """One context per curve for the sizes up to 2^ALL_MODES_MAX (their plans and tables: about 1 GiB together)."""
    from snark_b200 import Backend

    b = Backend(curve=request.param)
    yield b
    b.close()


# ---- inputs ---------------------------------------------------------------------------------------------------------
def _bits(curve):
    return curve.r.bit_length() - 1


def _limb_rows(values):
    return pack_u32(values, 8).reshape(-1, 8)


def edge_rows(curve):
    """0, 1, -1 in Montgomery form, and r - 1 as raw limbs (the largest representative a reduction must keep)."""
    R, r = 1 << 256, curve.r
    return _limb_rows([0, R % r, (r - 1) * R % r, r - 1])


def edge_index(n):
    """Index 0, N - 1 and both sides of tile boundaries (all of them up to 8 tiles, a spread beyond)."""
    idx = {0, n - 1}
    bounds = range(TILE, n, TILE) if n <= 8 * TILE else (TILE, 2 * TILE, n // 2, n - TILE)
    for m in bounds:
        idx |= {m - 1, m}
    return np.array(sorted(idx), dtype=np.int64)


def plant_edges(x, curve):
    """x: (n, 8) uint32 numpy array or int32 torch tensor of raw limbs, changed in place: a run of zeros with one edge
    value in its middle, and the edge values cycled over edge_index(n)."""
    n = x.shape[0]
    rows = edge_rows(curve)
    idx = edge_index(n)
    if n >= 16:
        lo = n // 4 + 3
        run = min(n // 8, 300)
        idx = np.union1d(idx, [lo + run // 2])
    vals = rows[np.arange(len(idx)) % len(rows)]
    if isinstance(x, np.ndarray):
        if n >= 16:
            x[lo : lo + run] = 0
        x[idx] = vals
    else:
        import torch

        if n >= 16:
            x[lo : lo + run] = 0
        x[torch.from_numpy(idx).to(x.device)] = torch.from_numpy(vals.view(np.int32)).to(x.device)
    return x


def host_input(curve, n, seed):
    """(n, 8) uint32 random field elements (Montgomery limbs) with the edge values planted; filled in chunks so that
    2^27 elements need no 8 GiB temporary."""
    rng = np.random.default_rng(seed)
    out = np.empty((n, 8), dtype=np.uint32)
    step = 1 << 22
    for s in range(0, n, step):
        k = min(step, n - s)
        out[s : s + k] = random_fr_limbs(rng, k, bits=_bits(curve)).reshape(k, 8)
    return plant_edges(out, curve)


def device_input(curve, n, seed):
    """The same kind of input generated on the device (int32 view of the limbs)."""
    import torch

    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    t = torch.randint(-(1 << 31), (1 << 31) - 1, (n, 8), dtype=torch.int32, device="cuda", generator=gen)
    t[:, 7] &= (1 << (_bits(curve) - 224)) - 1
    return plant_edges(t, curve)


def to_device(a):
    import torch

    return torch.from_numpy(a.view(np.int32)).cuda()


def to_host(t):
    return t.cpu().numpy().view(np.uint32)


def oracle_ntt(curve_id, x, log_n, mode):
    inverse, coset = MODES[mode]
    return cnative.ntt(curve_id, x.copy(), log_n, inverse=inverse, coset=coset)


def gpu_ntt(be, x_dev, log_n, mode):
    inverse, coset = MODES[mode]
    y = x_dev.clone()
    be.ntt(y, log_n, inverse=inverse, coset=coset)
    be.sync()
    return y


# ---- 1. b2s_ntt against the oracle, every plan ---------------------------------------------------------------------
def test_mode_rotation_covers_radix9_plans():
    for modes in LARGE_MODES.values():
        assert sorted(modes) == list(range(ALL_MODES_MAX + 1, 28))
        assert {m for lg in (25, 26, 27) for m in modes[lg]} == set(MODES)


@pytest.mark.parametrize("log_n", range(0, ALL_MODES_MAX + 1))
def test_ntt_matches_oracle(be, log_n):
    curve = CURVES[be.curve]
    x = host_input(curve, 1 << log_n, 1000 + log_n)
    x_dev = to_device(x)
    for mode in MODES:
        got = to_host(gpu_ntt(be, x_dev, log_n, mode))
        assert np.array_equal(got, oracle_ntt(be.curve, x, log_n, mode)), f"2^{log_n} {mode}"


@pytest.mark.parametrize("log_n", range(ALL_MODES_MAX + 1, 28))
@pytest.mark.parametrize("curve_id", [0, 1], ids=CURVE_IDS)
def test_ntt_matches_oracle_large(curve_id, log_n):
    """One context per size (2^27: 16 GiB of tables), closed before the next."""
    from snark_b200 import Backend

    curve = CURVES[curve_id]
    x = host_input(curve, 1 << log_n, 2000 + log_n)
    b = Backend(curve=curve_id)
    try:
        x_dev = to_device(x)
        for mode in LARGE_MODES[curve_id][log_n]:
            got = to_host(gpu_ntt(b, x_dev, log_n, mode))
            assert np.array_equal(got, oracle_ntt(curve_id, x, log_n, mode)), f"2^{log_n} {mode}"
            del got
    finally:
        b.close()


@pytest.mark.parametrize("log_n", [0, 11, 19])
def test_ntt_host_buffer_matches_device(be, log_n):
    curve = CURVES[be.curve]
    x = host_input(curve, 1 << log_n, 3000 + log_n)
    x_dev = to_device(x)
    for mode, (inverse, coset) in MODES.items():
        y = x.copy()
        be.ntt(y.reshape(-1), log_n, inverse=inverse, coset=coset)
        assert np.array_equal(y, to_host(gpu_ntt(be, x_dev, log_n, mode))), f"2^{log_n} {mode}"


# ---- 2. composed factors == full-size tables ------------------------------------------------------------------------
def check_composed_equals_full(full, curve_id, log_n, monkeypatch):
    import torch

    from snark_b200 import Backend

    x = device_input(CURVES[curve_id], 1 << log_n, 4000 + 32 * curve_id + log_n)
    # the first transform builds this size's plan and full-size tables in `full` while B2S_NTT_FULL is unset; the choice
    # is made once per plan and context, so later transforms of `full` keep the tables whatever the variable says
    want = gpu_ntt(full, x, log_n, "fwd")
    monkeypatch.setenv("B2S_NTT_FULL", "0")
    comp = Backend(curve=curve_id)        # every plan of this context is built with the variable set
    try:
        for mode in MODES:
            if mode != "fwd":
                want = gpu_ntt(full, x, log_n, mode)
            got = gpu_ntt(comp, x, log_n, mode)
            assert torch.equal(got, want), f"2^{log_n} {mode}: composed factors differ from the full-size tables"
            del got
    finally:
        comp.close()


@pytest.mark.parametrize("log_n", range(1, ALL_MODES_MAX + 1))
def test_ntt_composed_equals_full(be, log_n, monkeypatch):
    check_composed_equals_full(be, be.curve, log_n, monkeypatch)


@pytest.mark.parametrize("log_n", range(ALL_MODES_MAX + 1, 28))
@pytest.mark.parametrize("curve_id", [0, 1], ids=CURVE_IDS)
def test_ntt_composed_equals_full_large(curve_id, log_n, monkeypatch):
    from snark_b200 import Backend

    full = Backend(curve=curve_id)
    try:
        check_composed_equals_full(full, curve_id, log_n, monkeypatch)
    finally:
        full.close()


# ---- 3. witness map with dense random assignments --------------------------------------------------------------------
def coeff_pool(curve, rng, n_random=300):
    """1 (interned as id 0, no multiplication), 0, -1, 2, r - 1 as raw limbs, and random values."""
    R, r = 1 << 256, curve.r
    head = _limb_rows([R % r, 0, (r - 1) * R % r, 2 * R % r, r - 1])
    return np.concatenate([head, random_fr_limbs(rng, n_random, bits=_bits(curve)).reshape(-1, 8)])


def draw_coeffs(pool, rng, nnz):
    """Half the entries one, the rest uniform over the pool."""
    pick = rng.integers(0, len(pool), nnz)
    pick[rng.random(nnz) < 0.5] = 0
    return pool[pick].reshape(-1)


def bench_system(curve, log_n, seed):
    """BenchCircuit-shaped rows (tools/spmv_probe.py) with pool coefficients; the domain is 2^log_n with padding rows."""
    from tools.spmv_probe import bench_shaped_csr

    rng = np.random.default_rng(seed)
    n_rows = (1 << log_n) - 1 - min(1500, 1 << (log_n - 2))
    mats, n_wit = bench_shaped_csr(n_rows, seed=seed)
    pool = coeff_pool(curve, rng)
    csr = [(rp, col, draw_coeffs(pool, rng, len(col))) for rp, col in mats]
    return csr, n_rows, 1, n_wit


def perm_system(curve, log_n, seed, n_inst=2):
    """One nonzero per row whose columns are a random permutation of the variables (with the DummyCircuit's fixed
    columns a, b and c would be constant vectors), pool coefficients; a few padding rows."""
    rng = np.random.default_rng(seed)
    n_rows = (1 << log_n) - n_inst - min(700, 1 << (log_n - 3))
    n_wit = n_rows + 11
    pool = coeff_pool(curve, rng)
    row_ptr = np.arange(n_rows + 1, dtype=np.uint64)
    csr = []
    for _ in range(3):
        col = rng.permutation(n_inst + n_wit)[:n_rows].astype(np.uint32)
        csr.append((row_ptr, col, draw_coeffs(pool, rng, n_rows)))
    return csr, n_rows, n_inst, n_wit


def assignment(curve, n_vars, seed):
    """Random z (satisfies nothing) with z[0] = 1 and the edge values planted."""
    z = host_input(curve, n_vars, seed)
    z[0] = edge_rows(curve)[1]
    return z.reshape(-1)


def gpu_witness_map(curve_id, csr, n_rows, n_inst, n_wit, z):
    """h from a fresh context, closed afterwards."""
    from snark_b200 import Backend

    b = Backend(curve=curve_id)
    try:
        m = b.r1cs_upload(n_rows, n_inst, n_wit, csr)
        h = b.witness_map(m, z)
        b.r1cs_free(m)
    finally:
        b.close()
    return h


@pytest.mark.parametrize(
    "curve_id,log_n,shape",
    [(1, 19, "bench"), (1, 22, "bench"), (1, 25, "perm"), (0, 22, "bench")],
    ids=["bn254-19-bench", "bn254-22-bench", "bn254-25-perm", "bls12_381-22-bench"],
)
def test_witness_map_dense_matches_oracle(curve_id, log_n, shape, monkeypatch):
    curve = CURVES[curve_id]
    csr, n_rows, n_inst, n_wit = (bench_system if shape == "bench" else perm_system)(curve, log_n, 5000 + log_n)
    z = assignment(curve, n_inst + n_wit, 6000 + log_n)
    h = gpu_witness_map(curve_id, csr, n_rows, n_inst, n_wit, z)
    assert len(h) == 8 << log_n
    assert np.array_equal(h, cnative.witness_map(curve_id, csr, n_rows, n_inst, z)), "witness_map differs from the CPU oracle"
    # composed factors: unmerged scalings (alpha = beta = Zinv) after three 1/N-scaled inverse transforms
    monkeypatch.setenv("B2S_NTT_FULL", "0")
    h_comp = gpu_witness_map(curve_id, csr, n_rows, n_inst, n_wit, z)
    assert np.array_equal(h_comp, h), "witness_map with composed factors differs from the full-size tables"


# ---- 4. distributed schedule at every cut ----------------------------------------------------------------------------
def max_log_ranks(log_n):
    """The largest cut dist_supported accepts for an even log_n: 2^lg ranks with lg <= floor(log_n / 4)."""
    return (log_n // 2) // 2


@pytest.mark.parametrize(
    "curve_id,log_n",
    [(c, lg) for lg in range(8, 25, 2) for c in (0, 1)] + [(1, 26)],
    ids=[f"{CURVE_IDS[c]}-{lg}" for lg in range(8, 25, 2) for c in (0, 1)] + ["bn254-26"],
)
def test_dist_sim_every_cut(curve_id, log_n):
    from snark_b200 import B2SError, Backend

    curve = CURVES[curve_id]
    top = max_log_ranks(log_n)
    cuts = list(range(1, top + 1)) if log_n <= 24 else [1, top]
    csr, n_rows, n_inst, n_wit = perm_system(curve, log_n, 7000 + log_n)
    z = assignment(curve, n_inst + n_wit, 8000 + log_n)
    b = Backend(curve=curve_id)
    try:
        m = b.r1cs_upload(n_rows, n_inst, n_wit, csr)
        h = b.witness_map(m, z)
        for lg in cuts:
            assert np.array_equal(b.witness_map_sim(m, z, lg), h), f"2^{log_n} over 2^{lg} ranks"
        with pytest.raises(B2SError) as e:
            b.witness_map_sim(m, z, top + 1)
        assert e.value.code == 16
        b.r1cs_free(m)
    finally:
        b.close()
