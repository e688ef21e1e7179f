"""Fill-up loops (SURVEY.md §8 f1) on the CPU: the oracle restatement (oracle/fillup_np.py) driven by the
REFERENCE's own Rejector / IndependenceSampler classes and by the pinned oracle samplers must agree row for row, and
the loop quirks of nsgan/GAN.py:311-339 / synthetic/main.py:149-169 are what the restatement says they are."""
import numpy as np
import pytest

from oracle import fillup_np as F
from oracle import ref_cases, ref_shims


def _stream(seed, dim=3):
    rng = np.random.RandomState(seed)

    def propose(n):
        x = rng.randn(n, dim).astype(np.float32)
        s = rng.beta(2, 5, size=(n, 1)).astype(np.float32)
        return x, s
    return propose


@pytest.mark.parametrize("kind", ["rejection", "hastings"])
def test_oracle_loop_with_reference_samplers_equals_oracle_samplers(kind):
    exp = ref_cases.expected("fillup_%s" % kind)       # the loop over the reference's own sampler classes
    if exp is None:
        pytest.skip(ref_shims.SKIP_REASON + " and no recorded outputs (python -m oracle.make_golden)")
    b = ref_cases.fillup_run(kind, F.OracleRejector, F.OracleIndependenceSampler)
    assert int(exp["cnt"]) == b["cnt"] and int(exp["cnt_propose"]) == b["cnt_propose"]
    assert int(exp["n_backfilled"]) == b["n_backfilled"]
    assert np.array_equal(exp["samples"], b["samples"]) and b["cnt"] >= 200


def test_backfill_starts_at_the_efficiency_cap_and_efficiency_may_overshoot():
    propose = _stream(5)
    base_x, base_s = propose(64)
    np.random.seed(1)
    mh = F.OracleIndependenceSampler(T=20)                 # at most 1/21 efficiency < MIN_EFFICIENCY (App. C8)
    mh.set_score_curr(np.float32(0.3))
    r = F.fill_up_nsgan(base_x, base_s, propose, mh.sampling, 64, 16)
    # filtering stops once cnt_propose >= eval_size / 0.2 = 320: (320 - 64) / 16 = 16 filtered batches, then back-fill
    assert r["n_backfilled"] > 0 and r["n_backfilled"] % 16 == 0
    filtered_batches = r["n_batches"] - r["n_backfilled"] // 16
    assert filtered_batches == 16
    assert r["cnt"] >= 64 and r["efficiency"] == r["cnt"] / r["cnt_propose"]


def test_running_guard_quirk_drops_rows_when_the_base_call_accepts_nothing():
    calls = {"n": 0}

    def sampling(x, s):                                     # nothing from the base call, everything afterwards
        calls["n"] += 1
        return x[:0] if calls["n"] == 1 else x

    propose = _stream(7)
    base_x, base_s = propose(40)
    r = F.fill_up_nsgan(base_x, base_s, propose, sampling, 40, 16, store_guard="running")
    # nsgan/GAN.py:323 tests the RUNNING count: the first accepted batch is counted but not stored (slots stay unwritten)
    assert r["cnt"] == 48 and not r["samples"][:16].any() and r["samples"][16:40].any()
    calls["n"] = 0
    propose = _stream(7)
    base_x, base_s = propose(40)
    r2 = F.fill_up_nsgan(base_x, base_s, propose, sampling, 40, 16, store_guard="batch")
    assert r2["samples"][:16].any()


def test_synthetic_loop_only_counts_productive_batches():
    calls = {"n": 0}

    def sampling(x, s):
        calls["n"] += 1
        return x[:0] if calls["n"] in (1, 2, 3) else x[:30]

    propose = _stream(9, dim=2)
    base_x, base_s = propose(50)
    r = F.fill_up_synthetic(base_x, base_s, propose, sampling)
    assert r["n_batches"] == 4 and r["cnt"] == 60 and r["cnt_propose"] == 50 + 2 * 50   # two empty batches not counted
