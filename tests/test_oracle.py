"""CPU tests: the oracle (oracle/admm_oracle.py, oracle/packed_layout_model.py) against the golden
fixtures produced by the unmodified reference (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from conftest import golden, golden_names
from oracle import admm_oracle as O
from oracle import packed_layout_model as M

FWD = golden_names(exclude=("module", "grad"))
GRAD = golden_names(prefix="grad")


@pytest.mark.parametrize("name", FWD)
def test_spectral_form_matches_reference_fp64(name):
    d = golden(name)
    out = O.admm_tv_spectral_form(d["x"].astype(np.float64), d["lam"], d["rho"], d["kern"], bool(d["iso"]), int(d["maxit"]))
    assert O.rel_err(out, d["out64"]) < 1e-11


@pytest.mark.parametrize("name", [n for n in FWD if "cfg" not in n])
def test_stencil_form_matches_reference_fp64(name):
    d = golden(name)
    out = O.admm_tv_stencil_form(d["x"].astype(np.float64), d["lam"], d["rho"], d["kern"], bool(d["iso"]), int(d["maxit"]))
    assert O.rel_err(out, d["out64"]) < 1e-11


@pytest.mark.parametrize("name", FWD)
def test_spectral_form_fp32_within_tolerance(name):
    """fp32 oracle vs the reference in fp32 AND fp64: the 1e-4 bar of BASELINE.json."""
    d = golden(name)
    out = O.admm_tv_spectral_form(d["x"], d["lam"], d["rho"], d["kern"], bool(d["iso"]), int(d["maxit"]))
    assert out.dtype == np.float32
    assert O.rel_err(out, d["out64"]) < 1e-4
    assert O.rel_err(out, d["out32"]) < 1e-4


@pytest.mark.parametrize("name", [n for n in FWD if not n.startswith("iso")])
def test_packed_layout_model_matches_reference(name):
    d = golden(name)
    k = d["kern"]
    k2 = None if k.size == 0 else k[0, 0].astype(np.float64)
    out = M.admm_tv_packed(d["x"], float(d["lam"]), float(d["rho"]), k2, int(d["maxit"]))
    assert O.rel_err(out, d["out64"]) < 1e-11


@pytest.mark.parametrize("name", GRAD)
def test_adjoint_matches_reference_autograd(name):
    d = golden(name)
    gx, gl, gr, gk = O.admm_tv_backward(d["x"], d["lam"], d["rho"], d["kern"], d["gout"], bool(d["iso"]), int(d["maxit"]))
    assert O.rel_err(gx, d["gx"]) < 1e-11
    assert abs(gl - d["glam"][0]) <= 1e-10 * max(1.0, abs(d["glam"][0]))
    assert abs(gr - d["grho"][0]) <= 1e-10 * max(1.0, abs(d["grho"][0]))
    if d["kern"].size:
        assert O.rel_err(gk, d["gkern"]) < 1e-11


def test_known_answers():
    """SURVEY.md section 4: maxit=0 -> zeros; constant image is a fixed point; delta kernel == denoise."""
    rng = np.random.default_rng(3)
    x = rng.random((1, 2, 16, 16))
    k = rng.random((3, 3)); k /= k.sum()
    assert np.all(O.admm_tv_spectral_form(x, 0.02, 0.04, k[None, None], False, 0) == 0)
    c = np.full((1, 1, 16, 16), 0.37)
    assert O.rel_err(O.admm_tv_spectral_form(c, 0.02, 0.04, k[None, None], False, 5), c) < 1e-12
    delta = np.zeros((3, 3)); delta[1, 1] = 1.0
    a = O.admm_tv_spectral_form(x, 0.05, 0.1, delta[None, None], False, 7)
    b = O.admm_tv_spectral_form(x, 0.05, 0.1, np.zeros((0,)), False, 7)
    assert O.rel_err(a, b) < 1e-12
    # circular shift equivariance
    r = O.admm_tv_spectral_form(np.roll(x, (3, 5), (-2, -1)), 0.02, 0.04, k[None, None], False, 6)
    assert O.rel_err(r, np.roll(O.admm_tv_spectral_form(x, 0.02, 0.04, k[None, None], False, 6), (3, 5), (-2, -1))) < 1e-12


# ---------------------------------------------------------------------------- one-step replay (the GPU route gate)
# tests/test_gpu_routes.py gates every saved state of a GPU training forward against one fp64 iteration replayed from the
# state before it (admm_tv_replay), at max|a-b| / max(max|q|, max|x_N|) <= 5e-6 (pair_err with the output as floor).
# These tests show that the replay is exact for the fp64 oracle, that an fp32 implementation passes it by a wide margin
# where whole trajectories do not (tau < 0), and that the gate catches a small change of one element.
REPLAY_GATE = 5e-6
REPLAY_CASES = [(iso, lam, k, maxit) for iso in (False, True) for lam in (0.02, -0.02) for k in (0, 5) for maxit in (1, 2, 12)]


def _replay_run(shape, lam, k, iso, maxit, dtype, seed=3, rho=0.04):
    psf = O.make_psf("gauss", k, 1.5) if k else None
    kern = psf[None, None] if k else np.zeros((0,), np.float32)
    x = O.make_blurred(shape, psf, seed=seed, noise=0.02).astype(dtype)
    out, hist = O.admm_tv_spectral_form(x, lam, rho, kern, iso, maxit, return_state=True)
    return x, kern, out, hist[:-1]


@pytest.mark.parametrize("iso,lam,k,maxit", REPLAY_CASES)
def test_replay_reproduces_fp64_history(iso, lam, k, maxit):
    x, kern, out, states = _replay_run((2, 2, 30, 45), lam, k, iso, maxit, np.float64)
    preds, norms, x_out = O.admm_tv_replay(x, lam, 0.04, kern, states, iso)
    assert len(preds) == maxit - 1
    assert O.pair_err(states, preds, np.abs(x_out).max()) <= 1e-12
    assert O.rel_err(x_out, out) <= 1e-12
    if iso:
        assert O.pair_err([(O.pixelnorm(a), O.pixelnorm(b)) for a, b in states], norms) == 0.0


@pytest.mark.parametrize("iso,lam,k,maxit", REPLAY_CASES)
def test_replay_of_fp32_run_is_one_step_sharp(iso, lam, k, maxit):
    x, kern, out, states = _replay_run((2, 2, 30, 45), lam, k, iso, maxit, np.float32)
    tau32 = float(np.float32(lam) / np.float32(0.04))
    nmaps = [(O.pixelnorm(a), O.pixelnorm(b)) for a, b in states] if iso else None       # fp32 maps, as a GPU saves them
    preds, norms, x_out = O.admm_tv_replay(x, lam, 0.04, kern, states, iso, tau32, nmaps)
    e_q, e_x = O.pair_err(states, preds, np.abs(x_out).max()), O.rel_err(out, x_out)
    e_n = O.pair_err(nmaps, norms) if iso else 0.0
    print("iso=%s lam=%g k=%d N=%d: one-step q %.1e  norms %.1e  x %.1e" % (iso, lam, k, maxit, e_q, e_n, e_x))
    assert e_q <= 1e-6 and e_n <= 1e-6 and e_x <= 1e-6


def test_replay_gate_holds_where_the_trajectory_separates():
    """iso=True, tau < 0: the fp32 trajectory ends 4e-4 from the fp64 one (over the 1e-4 end-to-end bound) although
    every iteration is computed correctly; one step from the fp32 state stays at fp32 rounding."""
    x, kern, out, states = _replay_run((1, 2, 128, 256), -0.02, 0, True, 20, np.float32)
    ref = O.admm_tv_spectral_form(x.astype(np.float64), -0.02, 0.04, kern, True, 20)
    preds, _, x_out = O.admm_tv_replay(x, -0.02, 0.04, kern, states, True, float(np.float32(-0.02) / np.float32(0.04)))
    e_traj, e_q, e_x = O.rel_err(out, ref), O.pair_err(states, preds, np.abs(x_out).max()), O.rel_err(out, x_out)
    print("trajectory %.1e  one-step q %.1e  x %.1e" % (e_traj, e_q, e_x))
    assert e_traj > 1e-4
    assert e_q <= 1e-6 and e_x <= 1e-6


@pytest.mark.parametrize("iso", [False, True])
@pytest.mark.parametrize("which", [0, 2, 4])
def test_replay_gate_catches_one_perturbed_element(iso, which):
    x, kern, out, states = _replay_run((1, 2, 32, 48), 0.02, 5, iso, 6, np.float32)
    tau32 = float(np.float32(0.02) / np.float32(0.04))
    preds, _, x_out = O.admm_tv_replay(x, 0.02, 0.04, kern, states, iso, tau32)
    assert O.pair_err(states, preds, np.abs(x_out).max()) <= 1e-6
    qmax = max(float(np.abs(q).max()) for s in states for q in s)
    bad = [(a.copy(), b.copy()) for a, b in states]
    bad[which][1][0, 1, 17, 23] += np.float32(1e-4 * qmax)
    preds, _, x_out = O.admm_tv_replay(x, 0.02, 0.04, kern, bad, iso, tau32)
    e = O.pair_err(bad, preds, np.abs(x_out).max())
    print("state %d perturbed by 1e-4 max|q|: replay error %.1e" % (which + 1, e))
    assert e > REPLAY_GATE


@pytest.mark.parametrize("lam", [0.02, -0.02])
def test_backward_nmaps_override_with_own_maps_changes_nothing(lam):
    x, kern, out, states = _replay_run((2, 2, 24, 30), lam, 5, True, 6, np.float32)
    gout = np.random.default_rng(4).standard_normal(x.shape)
    tau32 = float(np.float32(lam) / np.float32(0.04))
    s64 = [(a.astype(np.float64), b.astype(np.float64)) for a, b in states]
    nm = [(O.pixelnorm(a), O.pixelnorm(b)) for a, b in s64]
    a = O.admm_tv_backward(x, lam, 0.04, kern, gout, True, 6, qs_override=states, tau_override=tau32)
    b = O.admm_tv_backward(x, lam, 0.04, kern, gout, True, 6, qs_override=states, tau_override=tau32, nmaps_override=nm)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2] == b[2] and np.array_equal(a[3], b[3])
    # the fp64 oracle's own state given in full reproduces the plain adjoint (which re-runs the forward itself)
    _, _, _, h64 = _replay_run((2, 2, 24, 30), lam, 5, True, 6, np.float64)
    c = O.admm_tv_backward(x, lam, 0.04, kern, gout, True, 6)
    d = O.admm_tv_backward(x, lam, 0.04, kern, gout, True, 6, qs_override=h64,
                           nmaps_override=[(O.pixelnorm(p), O.pixelnorm(q)) for p, q in h64])
    assert O.rel_err(d[0], c[0]) < 1e-12 and O.rel_err(d[3], c[3]) < 1e-12
    assert abs(d[1] - c[1]) <= 1e-10 * max(1.0, abs(c[1])) and abs(d[2] - c[2]) <= 1e-10 * max(1.0, abs(c[2]))


def test_non_square_kernel_raises_like_reference():
    with pytest.raises(RuntimeError):
        O.admm_tv_spectral_form(np.zeros((1, 1, 8, 8)), 0.02, 0.04, np.zeros((1, 1, 3, 5)), False, 2)


@pytest.mark.parametrize("n", [2, 3, 4, 5, 6, 7, 8, 9, 12, 15, 16, 31, 45, 60, 64, 90, 135, 256])
def test_stockham_index_model(n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    r = M.factorize(n)
    assert np.abs(M.stockham_fft(x, r, -1) - np.fft.fft(x)).max() < 1e-11 * n
    assert np.abs(M.stockham_fft(x, r, +1) - np.fft.ifft(x) * n).max() < 1e-11 * n


@pytest.mark.parametrize("W", [4, 7, 8, 9, 16, 33])
def test_pair_trick(W):
    rng = np.random.default_rng(W)
    a, b = rng.standard_normal(W), rng.standard_normal(W)
    Pa, Pb = M.pair_r2c(a, b)
    assert np.abs(Pa - M.rows_r2c(a)).max() < 1e-12 and np.abs(Pb - M.rows_r2c(b)).max() < 1e-12
    ra, rb = M.pair_c2r(Pa, Pb, W)
    assert np.abs(ra - a * W).max() < 1e-11 and np.abs(rb - b * W).max() < 1e-11


def test_tile_major_spectrum_layout_model():
    """The tile-major layout between the two large-frame kernels: a bijection of the H x Wc entries in which (a) the two
    rows the row kernel transforms together are adjacent complex slots (one 16-byte access), (b) the 8 columns of a tile
    for one row pair are one 128-byte run, (c) a column tile is one contiguous block."""
    from oracle import packed_layout_model as M
    H, Wc = 12, 16
    for kind in ("v", "x"):
        idx = np.array([[M.tile_major_index(u, c, H, kind) for c in range(Wc)] for u in range(H)])
        assert sorted(idx.ravel().tolist()) == list(range(H * Wc))
        for k in range(H // 2):
            ra, rb = (2 * k, 2 * k + 1) if kind == "v" else ((2 * k - 1) % H, 2 * k)
            assert np.all(idx[rb] == idx[ra] + 1)                                   # (a)
            assert np.all(np.diff(idx[ra, :8]) == 2) and idx[ra, 0] % 16 == 0       # (b): 8 columns x 2 rows x 8 bytes
        assert idx[:, :8].max() < H * 8 and idx[:, 8:].min() >= H * 8               # (c)
    P = np.arange(H * Wc).reshape(H, Wc).astype(np.complex64)
    assert np.array_equal(np.sort(M.to_tile_major(P, "x").real), np.arange(H * Wc))


def test_cfg3_full_size_fixture_pins_oracle_to_reference():
    """BASELINE configs[2] at its real shape and length (1 x 3 x 2160 x 3840, 63 x 63 PSF, 200 iterations): the fixture of
    tests/golden/make_golden_cfg3.py holds summaries of the fp64 oracle AND of the unmodified reference (fp32: its fp64
    run needs 263 GB) on the same input; they must agree within the reference's own fp32 noise."""
    d = golden("cfg3_2160x3840_gauss63_n200")
    amax = float(d["ref32_absmax"])
    assert tuple(d["shape"]) == (1, 3, 2160, 3840) and int(d["maxit"]) == 200 and int(d["k"]) == 63
    assert float(np.abs(d["oracle64_crops"] - d["ref32_crops"]).max()) / amax < 1e-4
    assert float(np.abs(d["oracle64_rowmean"] - d["ref32_rowmean"]).max()) / amax < 1e-4
    assert float(np.abs(d["oracle64_colmean"] - d["ref32_colmean"]).max()) / amax < 1e-4
    assert abs(float(d["oracle64_sum"]) - float(d["ref32_sum"])) / abs(float(d["ref32_sum"])) < 1e-5
    assert float(d["oracle_vs_ref32"]) < 1e-4
