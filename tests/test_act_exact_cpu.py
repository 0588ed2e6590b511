"""CPU: the exact fp32 model of the action sampling (``tests/act_exact.py``) against the float64 transcription of the
noise (``tests/action_noise_ref.py``) and the oracle (``oracle/policy.py::gaussian_act``), on Philox words random
counters never reach, and with planted defects: each must change an output bit on the fixture the GPU tests use.  The
tolerance comparisons the sampling had before (4 ulp on the noise, rtol 1e-4 on the log-prob, one launch against
forward + ``gaussian_act`` of the previewed noise) are run on the same mutants to record which ones they let through."""
import math
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import act_exact as X  # noqa: E402
from action_noise_ref import normal2_f64  # noqa: E402
from oracle import policy as OP  # noqa: E402
from scan_exact import fma32, mul_add32  # noqa: E402

F = np.float32
F64 = X.Float64Math()


def _f64_words(w0, w1):
    """``normal2_f64``'s formula on explicit words."""
    u1 = ((np.asarray(w0, np.uint32) >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24
    u2 = (np.asarray(w1, np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    r = np.sqrt(-2.0 * np.log(u1))
    return np.stack([r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)], axis=-1)


def _within_4ulp(z, ref):
    tol = 4.0 * np.spacing(np.abs(ref).astype(F)).astype(np.float64) + 1e-12  # (+: cos(pi/2) is 6e-17 in float64)
    with np.errstate(invalid="ignore"):
        return bool((np.abs(z.astype(np.float64) - ref) <= tol).all())


def _oracle(mean, ls, eps):
    a, lp = OP.gaussian_act(torch.from_numpy(mean), torch.from_numpy(ls), torch.from_numpy(eps))
    return a.numpy(), lp.numpy().reshape(-1)


# ------------------------------------------------------------------------------------------------ ties to the references
def test_model_noise_against_float64():
    seed, step, n, off = 2024, 17, 200_000, 99
    assert _within_4ulp(X.normal2(seed, step, n, F64, env_offset=off), normal2_f64(seed, step, n, off))
    w0, w1 = X.crafted_words()
    assert _within_4ulp(X.box_muller(w0, w1, F64), _f64_words(w0, w1))


def test_crafted_words_hit_the_edges_exactly():
    """``w >> 8`` = 2^24 - 1 gives u1 = 1 and r = 0; ``w >> 8`` = 0 gives the largest radius sqrt(-2 ln 2^-24); the
    quadrant points of ``w1 >> 8`` (0, 2^22, 2^23, 3 2^22) give exact axes: sincospif(0, 1/2, 1, 3/2)."""
    r_max = F(np.sqrt(F(-2) * F64.log(F(2.0 ** -24))))
    assert abs(float(r_max) - math.sqrt(-2 * math.log(2.0 ** -24))) < 1e-6
    q = [(0, (r_max, 0)), (1 << 22, (0, r_max)), (1 << 23, (-r_max, 0)), (3 << 22, (0, -r_max))]
    for hi1, want in q:
        for lo in (0, 0xFF):
            z = X.box_muller(np.uint32(0 | lo), np.uint32((hi1 << 8) | lo), F64)
            assert np.array_equal(z, F(want)), (hi1, z)
    z = X.box_muller(np.uint32(0xFFFFFFFF), np.uint32(0x12345678), F64)
    assert np.array_equal(np.abs(z), F([0, 0]))
    assert np.isfinite(X.box_muller(*X.crafted_words(), F64)).all()


def test_model_against_the_oracle():
    """With float64 math and mul + add in place of the fma, the model is the oracle's arithmetic, bit for bit (where
    torch's fp32 exp is float64's rounded); with the fma, the two agree on every NaN and bit for bit wherever the fma
    and mul + add round alike."""
    cases = X.gaussian_fixture(F64)
    for ls, mean, eps in cases:
        a, lp = X.gaussian_sample(mean, ls, eps, F64)
        a_mul, lp_mul = X.gaussian_sample(mean, ls, eps, F64, mut={"mul_add"})
        oa, olp = _oracle(mean, ls, eps)
        assert np.array_equal(np.isnan(a), np.isnan(oa)) and np.array_equal(np.isnan(lp), np.isnan(olp)), ls
        if np.isnan(ls).any():
            assert np.isnan(a[:, np.isnan(ls)]).all() and np.isnan(lp).all()
        sd = F64.exp(X.clamp(ls, -20, 2))
        if not X.bits_equal(torch.exp(torch.from_numpy(X.clamp(ls, -20, 2))).numpy(), sd).all():
            continue
        assert X.bits_equal(a_mul, oa).all() and X.bits_equal(lp_mul, olp).all(), ls
        with np.errstate(invalid="ignore"):
            same = (fma32(sd, eps, mean) == mul_add32(sd, eps, mean)) | np.isnan(mean)
        rows = same.all(axis=1)
        assert X.bits_equal(a[same], oa[same]).all() and X.bits_equal(lp[rows], olp[rows]).all(), ls


def test_nan_means_and_log_std_stay_nan():
    """torch.clamp keeps NaN; so does the model (the kernel after the fix), the old fminf / fmaxf clip did not."""
    mean = F([[np.nan, 0.2], [np.nan, np.nan], [0.1, -0.3]])
    eps = F([[0.5, -1.0], [0.0, 0.0], [0.2, 0.2]])
    a, lp = X.gaussian_sample(mean, F([0.0, 0.0]), eps, F64)
    assert np.isnan(a[0, 0]) and a[0, 1] == F(0.2) + F(-1.0) and np.isnan(a[1]).all() and np.isnan(lp[:2]).all()
    assert np.isfinite(a[2]).all() and np.isfinite(lp[2])
    old, old_lp = X.gaussian_sample(mean, F([0.0, 0.0]), eps, F64, mut={"nan_drop"})
    assert old[0, 0] == -1 and (old[1] == -1).all() and np.isnan(old_lp[:2]).all()
    a, lp = X.gaussian_sample(F([[0.1, 0.2]]), F([np.nan, 0.0]), F([[0.3, 0.3]]), F64)
    assert np.isnan(a[0, 0]) and np.isfinite(a[0, 1]) and np.isnan(lp).all()
    oa, olp = _oracle(F([[0.1, 0.2]]), F([np.nan, 0.0]), F([[0.3, 0.3]]))
    assert np.isnan(oa[0, 0]) and np.isnan(olp).all()


# ------------------------------------------------------------------------------------------------ mutants
def _fixture(math_):
    """What the GPU tests compare, with ``math_`` for the three functions: noise of crafted, recorded-logf and random
    words; ``gaussian_sample`` on the constructed cases; one sampling epilogue (noise into gaussian_sample)."""
    w0, w1 = X.crafted_words()
    lw = X.log_words()
    rnd = X.philox_words(2024, 17, 20_000, 99)
    W0 = np.concatenate([w0, lw, rnd[:, 0]])
    W1 = np.concatenate([w1, np.full_like(lw, 0x00ABCDEF), rnd[:, 1]])
    W2 = np.concatenate([w1 ^ np.uint32(0x5555), lw ^ np.uint32(0xFFFF), rnd[:, 2]])
    words = np.stack([W0, W1, W2, W2], axis=1)
    mean = np.tanh(np.random.default_rng(3).standard_normal((len(words), 2)) * 2).astype(F)
    mean[::53] = np.nan
    return words, X.gaussian_fixture(math_), mean


def _run(fix, math_, mut):
    words, cases, mean = fix
    noise = X.box_muller(words[:, 0], words[:, 1], math_, mut, words[:, 2])
    gauss = [X.gaussian_sample(m, ls, e, math_, mut) for ls, m, e in cases]
    fused = X.sample_from_words(words, mean, F([-0.5, 0.7]), math_, mut)
    return noise, gauss, fused


def _differs(base, out):
    (n0, g0, f0), (n1, g1, f1) = base, out
    d = not X.bits_equal(n0, n1).all()
    d |= any(not X.bits_equal(x, y).all() for (a, b), (c, e) in zip(g0, g1) for x, y in ((a, c), (b, e)))
    d |= any(not X.bits_equal(x, y).all() for x, y in zip(f0, f1))
    return d


def _old_tolerances_accept(fix, out, math_, mut=frozenset()):
    """Would the sampling's earlier comparisons accept these outputs?  (i) the previewed noise within 4 ulp of the
    float64 transcription; (ii) gaussian_act against the oracle, actions rtol / atol 1e-6, log_prob rtol / atol 1e-4, on
    what those tests fed it (finite means and log_std); (iii) a sampling launch equal, bit for bit, to gaussian_act of
    the previewed noise and the launch's mean."""
    words, cases, mean = fix
    noise, gauss, fused = out
    ok = _within_4ulp(noise, _f64_words(words[:, 0], words[:, 1]))
    for (ls, m, e), (a, lp) in zip(cases, gauss):
        if not np.isfinite(ls).all():
            continue
        rows = np.isfinite(m).all(axis=1)
        oa, olp = _oracle(m[rows], ls, e[rows])
        ok &= np.allclose(a[rows], oa, rtol=1e-6, atol=1e-6) and np.allclose(lp[rows], olp, rtol=1e-4, atol=1e-4)
    eps, fa, flp = fused
    ga, glp = X.gaussian_sample(mean, F([-0.5, 0.7]), eps, math_, mut - {"rc_fused"})
    ok &= bool(X.bits_equal(fa, ga).all() and X.bits_equal(flp, glp).all())
    return bool(ok)


# Mutants that every earlier comparison accepts on this fixture: only the bit-exact model sees them.  The others change
# the noise by more than 4 ulp (u1 without +1 sends w0 >> 8 = 0 to log 0, r = inf), move a clipped log-prob far, or make
# the one-launch form differ from gaussian_act of the preview.
LET_THROUGH_BY_TOLERANCES = {"log_f64", "mul_add", "neg_log_exp", "ls_bound_ulp", "nan_drop"}


@pytest.fixture(scope="module")
def mutant_base():
    rm = X.RecordedMath()
    fix = _fixture(rm)
    return rm, fix, _run(fix, rm, frozenset())


@pytest.mark.parametrize("mut", sorted(X.MUTANTS))
def test_mutant_changes_an_output_bit(mutant_base, mut):
    rm, fix, base = mutant_base
    out = _run(fix, rm, frozenset([mut]))
    assert _differs(base, out), f"mutant {mut!r} ({X.MUTANTS[mut]}) changes no bit"
    tolerated = _old_tolerances_accept(fix, out, rm, frozenset([mut]))
    assert tolerated == (mut in LET_THROUGH_BY_TOLERANCES), (mut, tolerated)


def test_unmutated_model_passes_the_old_tolerances(mutant_base):
    rm, fix, base = mutant_base
    assert _old_tolerances_accept(fix, base, rm)


def test_recorded_logf_points_differ_from_the_correctly_rounded_log():
    z = np.load(X.GOLDEN_MATH)
    assert len(z["log_x"]) and not X.bits_equal(z["log_y"], F64.log(z["log_x"])).any()
    assert (np.abs(z["log_y"].astype(np.float64) - np.log(z["log_x"].astype(np.float64)))
            <= np.spacing(np.abs(z["log_y"])).astype(np.float64)).all()  # within logf's 1 ulp
    k = np.round(z["log_x"].astype(np.float64) * 2.0 ** 24)
    assert (k >= 1).all() and (k <= 2 ** 24).all() and np.array_equal(k * 2.0 ** -24, z["log_x"])  # on the u1 grid


# ------------------------------------------------------------------------------------------------ equivalences
def test_dropped_mutant_two_sd_sd():
    """2 (sd sd) against (2 sd) sd: sd = expf(ls) lies in [e^-20, e^2], where doubling is exact, so both are the one
    rounding of 2 sd^2 -- the candidate cannot change a bit and is dropped.  torch's 2 * var is the first form."""
    ls = np.concatenate([np.random.default_rng(0).uniform(-20, 2, 1 << 20).astype(F), F([-20, 2, 0])])
    sd = F64.exp(ls)
    assert np.array_equal((F(2) * (sd * sd).astype(F)).astype(F), ((F(2) * sd).astype(F) * sd).astype(F))


def test_dropped_mutant_log_prob_sum_from_zero():
    """fl(0 + t0) + t1 against t0 + t1 (torch's sum of two): 0 + t is t unless t = -0, and a term is never -0 -- its last
    operation subtracts the nonzero 0.9189385f, and x - y = 0 gives +0 in round-to-nearest."""
    t = np.concatenate([np.random.default_rng(1).standard_normal(1 << 16).astype(F), F([0.0, X.LOG_SQRT_2PI])])
    terms = (t - X.LOG_SQRT_2PI).astype(F)
    assert not (np.signbit(terms) & (terms == 0)).any()
    assert np.array_equal((F(0) + terms).astype(F).view(np.uint32), terms.view(np.uint32))


def test_dropped_mutant_negation_placement():
    """-(d d) / q against -((d d) / q): division is sign-symmetric, so the two are the same number."""
    g = np.random.default_rng(2)
    d = g.standard_normal(1 << 16).astype(F)
    q = np.abs(g.standard_normal(1 << 16)).astype(F) + F(1e-3)
    dd = (d * d).astype(F)
    assert np.array_equal(((-dd) / q).astype(F).view(np.uint32), (-(dd / q)).astype(F).view(np.uint32))


def test_uniforms_and_constant_are_exact():
    """fl(k + 1) 2^-24 and fl(2 u2) are exact, and 0.9189385f is torch's log(sqrt(2 pi)) as an fp32 scalar."""
    k = np.arange(1 << 24, dtype=np.int64)
    assert np.array_equal(((k + 1).astype(F) * X.TWO_M24).astype(np.float64), (k + 1) * 2.0 ** -24)
    u2 = (k.astype(F) * X.TWO_M24).astype(F)
    assert np.array_equal((F(2) * u2).astype(np.float64), 2.0 * (k * 2.0 ** -24))
    assert F(math.log(math.sqrt(2 * math.pi))) == X.LOG_SQRT_2PI
