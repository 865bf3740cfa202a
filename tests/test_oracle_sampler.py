"""WeightedSampler restatement (oracle/vg_oracle.c vgo_sampler_*) pinned against the REFERENCE's own
code: golden vectors generated from voxgraph::WeightedSampler compiled out of the reference sources
(tests/golden/make_sampler_golden.py), and - where oracle/_ref is present - the compiled reference
itself."""
import json
import os

import numpy as np
import pytest

from oracle import oracle as o

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "weighted_sampler.json")
REF_DRAWS = os.path.join(os.path.dirname(__file__), "golden", "weighted_sampler_draws.npz")


def _cases():
    return json.load(open(GOLDEN))["cases"]


def test_mt19937_standard_check_value():
    # [rand.predef]: the 10000th consecutive invocation of a default-constructed mt19937 is 4123659995
    s = o.WeightedSampler(np.ones(4, np.float32))
    v = [s.next_u32() for _ in range(10000)]
    assert v[0] == 3499211612 and v[-1] == 4123659995


def test_canonical_in_unit_interval_and_two_draws_per_number():
    s = o.WeightedSampler(np.ones(4, np.float32))
    t = o.WeightedSampler(np.ones(4, np.float32))
    for _ in range(1000):
        g1, g2 = t.next_u32(), t.next_u32()
        r = s.canonical()
        assert 0.0 <= r < 1.0
        assert r == (g1 + g2 * 4294967296.0) / 18446744073709551616.0


@pytest.mark.parametrize("case", _cases(), ids=lambda c: c["name"])
def test_draws_match_reference_golden(case):
    w = np.array(case["weights"], np.float32)
    s = o.WeightedSampler(w)
    assert s.draw(64).tolist() == case["draw_0_64"]
    assert s.draw(64).tolist() == case["draw_64_128"]     # the generator state carries over


def test_draws_match_compiled_reference():
    """2000 draws from each of five weight vectors (1 to 20000 items) as the compiled reference made
    them (tests/golden/weighted_sampler_draws.npz); where oracle/_ref is built, also the live one."""
    z = np.load(REF_DRAWS)
    live = o.ref_sampler_lib() is not None
    for n in z["sizes"]:
        w, want = z["weights_%d" % n], z["draws_%d" % n]
        assert np.array_equal(o.WeightedSampler(w).draw(len(want)), want)
        if live:
            assert np.array_equal(o.RefWeightedSampler(w).draw(len(want)), want)


def test_zero_weight_items_are_never_drawn_and_frequencies_follow_weights():
    w = np.array([0.0, 1.0, 0.0, 3.0, 0.0], np.float32)
    idx = o.WeightedSampler(w).draw(20000)
    cnt = np.bincount(idx, minlength=5)
    assert cnt[0] == cnt[2] == cnt[4] == 0
    assert abs(cnt[3] / cnt[1] - 3.0) < 0.2


def test_sampled_num_residuals_is_float_product_truncated():
    # registration_cost_function.cpp:45-55
    assert o.sampled_num_residuals(-1, 10000) == 10000
    assert o.sampled_num_residuals(0.05, 10000) == 500
    assert o.sampled_num_residuals(0.2, 1001) == int(np.float32(0.2) * np.float32(1001))
    assert o.sampled_num_residuals(0.05, 19) == 0
