"""Weighted sampling on the host: the specification (oracle/sampler_oracle.py) against a brute-force sampler and against
today's uniform stream, the planner classes' weighted draws in all four regimes of integers(0, T), and the argument checks,
which all raise before any device is used.  No GPU needed."""
import copy

import numpy as np
import pytest

from oracle import sampler_oracle as S
from rrtplanner_b200 import RRTDubins, RRTStandard, RRTStar, RRTStarInformed, _lib, batch


def _case(seed, W=23, H=37, p=0.3):
    rng = np.random.default_rng(seed)
    og = (rng.random((W, H)) < p).astype(np.uint8)
    w = rng.integers(0, 256, size=(W, H)).astype(np.uint8)
    return og, w


@pytest.mark.parametrize("seed", range(4))
def test_oracle_against_brute_force(seed):
    og, w = _case(seed)
    w[w < 128] = 0                                   # many zero-weight free cells among the occupied ones
    got, _, _ = S.weighted_stream(w, og == 0, 300, seed=seed)
    assert np.array_equal(got, S.brute_force_stream(w, og == 0, 300, seed=seed))
    e = S.effective_weights(w, og == 0)
    assert (e[got[:, 0], got[:, 1]] > 0).all()


@pytest.mark.parametrize("seed", range(4))
def test_all_ones_is_the_uniform_stream(seed):
    og, _ = _case(seed)
    free = np.argwhere(og == 0)
    got, words, carry = S.weighted_stream(np.ones_like(og), og == 0, 500, seed=seed)
    rng = np.random.default_rng(seed)
    assert np.array_equal(got, free[rng.integers(0, free.shape[0], 500)])
    assert rng.bit_generator.state == S.generator(state=words, carry=carry).bit_generator.state


def test_oracle_resumes_a_carried_generator():
    og, w = _case(7)
    rng = np.random.default_rng(11)
    rng.integers(0, 1000, size=3)                    # leaves a buffered 32-bit half
    assert rng.bit_generator.state["has_uint32"] == 1
    words, carry = S.generator_words(rng)
    got, w2, c2 = S.weighted_stream(w, og == 0, 100, state=words, carry=carry)
    cum = np.cumsum(S.effective_weights(w, og == 0).ravel())
    k = np.searchsorted(cum, rng.integers(0, int(cum[-1]), size=100), side="right")
    assert np.array_equal(got, np.stack(np.divmod(k, og.shape[1]), axis=1))
    assert (np.array_equal(w2, S.generator_words(rng)[0]) and np.array_equal(c2, S.generator_words(rng)[1]))


def weights_with_total(shape, total):
    """uint8 map of ``shape`` whose entries sum to ``total`` (255 almost everywhere)."""
    w = np.full(shape, 255, dtype=np.uint8).ravel()
    excess = 255 * w.size - total
    assert 0 <= excess
    full, part = divmod(excess, 255)
    w[:full] = 0
    w[full] -= np.uint8(part)
    return w.reshape(shape)


# T = 1, a 32-bit total, 2^32 - 1, 2^32 (raw halves), 2^32 + 1 (64-bit Lemire)
REGIMES = {"one": (8, 9, 1), "small": (23, 37, None), "2^32-1": (4160, 4096, 2 ** 32 - 1), "2^32": (4160, 4096, 2 ** 32),
           "2^32+1": (4160, 4096, 2 ** 32 + 1)}


@pytest.mark.parametrize("regime", list(REGIMES))
def test_class_draws_equal_repeated_sample_all_free(regime):
    W, H, T = REGIMES[regime]
    og = np.zeros((W, H), dtype=np.uint8)
    if T is None:
        og, w = _case(3, W, H)
    elif T == 1:
        w = np.zeros((W, H), dtype=np.uint8)
        w[5, 2] = 1
        og[0, :] = 1
    else:
        w = weights_with_total((W, H), T)
    a = RRTStandard(og, 50, pbar=False, seed=5, sample_weights=w)
    b = RRTStandard(og, 50, pbar=False, seed=5, sample_weights=w)
    a.rand_gen.integers(0, 7, size=1)                # start both from a generator with a buffered half
    b.rand_gen.integers(0, 7, size=1)
    words, carry = S.generator_words(a.rand_gen)
    got = a._draw_samples(40)
    one_by_one = np.array([b.sample_all_free() for _ in range(40)])
    assert np.array_equal(got, one_by_one)
    assert a.rand_gen.bit_generator.state == b.rand_gen.bit_generator.state
    want, w2, c2 = S.weighted_stream(w, og == 0, 40, state=words, carry=carry)
    assert np.array_equal(got, want)
    assert np.array_equal(S.generator_words(a.rand_gen)[0], w2) and np.array_equal(S.generator_words(a.rand_gen)[1], c2)
    if T == 1:
        assert (got == [5, 2]).all() and a.rand_gen.bit_generator.state == S.generator(state=words, carry=carry).bit_generator.state


def test_all_ones_classes_draw_todays_stream():
    og, _ = _case(2)
    ones = np.ones_like(og)
    for make in (lambda **k: RRTStandard(og, 80, pbar=False, seed=9, **k), lambda **k: RRTStar(og, 80, 5.0, pbar=False, seed=9, **k),
                 lambda **k: RRTDubins(og, 80, 3.0, 8, pbar=False, seed=9, **k)):
        a, b = make(), make(sample_weights=ones)
        assert np.array_equal(a._draw_samples(80), b._draw_samples(80))
        assert np.array_equal(a.sample_all_free(), b.sample_all_free())
        assert a.rand_gen.bit_generator.state == b.rand_gen.bit_generator.state


def test_informed_probe_generator_is_weighted():
    og, w = _case(4)
    p = RRTStarInformed(og, 60, 5.0, 3.0, pbar=False, seed=2, sample_weights=w)
    g = copy.deepcopy(p.rand_gen)
    want, _, _ = S.weighted_stream(w, og == 0, 60, state=S.generator_words(g)[0], carry=S.generator_words(g)[1])
    assert np.array_equal(p._draw_free(g, 60), want)


class _OwnSampler(RRTStandard):
    def sample_all_free(self):
        return np.array([0, 0])


def test_argument_checks_raise_before_any_device_use():
    og, w = _case(1)
    for bad in (w.astype(np.float64), w.astype(np.int16), w.astype(np.int64) + 300):
        with pytest.raises(TypeError):
            RRTStandard(og, 10, pbar=False, sample_weights=bad)
    with pytest.raises(ValueError):
        RRTStar(og, 10, 5.0, pbar=False, sample_weights=w[:, :-1])
    zero = np.where(og == 0, 0, 255).astype(np.uint8)          # weight on occupied cells only: masked away, T = 0
    with pytest.raises(ValueError):
        RRTStandard(og, 10, pbar=False, sample_weights=zero)
    with pytest.raises(TypeError):
        _OwnSampler(og, 10, pbar=False, sample_weights=w)
    p = RRTStandard(og, 10, pbar=False, sample_weights=w)
    with pytest.raises(ValueError):
        p.set_og(np.zeros((og.shape[0] + 1, og.shape[1])))
    p.set_og(np.zeros_like(og))                                  # re-masked: every cell free now
    assert int(p._wcum[-1]) == int(w.astype(np.int64).sum())
    # plan_batch: refused before a context (which needs a device) exists
    ogs = np.stack([og, og])
    st, gl = np.zeros((2, 2), int), np.ones((2, 2), int)
    with pytest.raises(ValueError):
        batch.plan_batch("informed", ogs, 10, st, gl, r_rewire=5.0, r_goal=2.0, seeds=[0, 1], balls="seed", sample_weights=w)
    with pytest.raises(ValueError):
        batch.plan_batch("standard", ogs, 10, st, gl, samples=np.zeros((2, 10, 2)), sample_weights=w)
    with pytest.raises(ValueError):
        batch.plan_batch("standard", ogs, 10, st, gl, seeds=[0, 1], sample_weights=np.stack([w, w, w]))
    with pytest.raises(TypeError):
        batch.plan_batch("star", ogs, 10, st, gl, r_rewire=3.0, seeds=[0, 1], sample_weights=w.astype(np.float32))
    assert _lib.sample_weights_array(w, (3, *w.shape)).shape == (3, *w.shape)
