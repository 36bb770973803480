"""The resident snapshot of the host-pointer entry points: which calls leave their uploaded snapshot on the device for
ust_apply_state_delta / _delta_sparse / ust_fetch_outputs, and which leave an earlier one untouched. Bit-exact against
the oracle. Run on the B200 box: python -m pytest tests -m gpu"""
import numpy as np
import pytest

import helpers
from helpers import abi
from ust import lib as ustlib

pytestmark = pytest.mark.gpu

COLS = ("state", "flags", "pod_rev", "ds_idx")
INVALID = abi.K["UST_ERR_INVALID_ARGUMENT"]


@pytest.fixture(scope="module")
def handle():
    h = ustlib.Handle(0)  # raises (never skips) when the extension or the device is missing
    yield h
    h.close()


def policy():
    return abi.make_policy(max_parallel_upgrades=0, max_unavailable="30%")


def full_call(handle, fmt, pol, soa):
    return handle.apply_state_packed(pol, soa) if fmt == "packed" else handle.apply_state(pol, soa)


def delta_matches_oracle(handle, rng, pol, soa, m):
    """Re-encodes m random nodes of `soa` (in place), sends them as a dense delta and checks the result against the
    oracle on the updated arrays. Returns the delta's result."""
    n = soa["state"].shape[0]
    idx = rng.choice(n, size=m, replace=False).astype(np.int64)
    fresh, _ = helpers.random_soa(rng, m, wild=True)
    for k in COLS:
        soa[k][idx] = fresh[k]
    got = handle.apply_state_delta(pol, n, idx, {k: fresh[k] for k in COLS}, soa["ds_rev"])
    helpers.assert_same(got, helpers.oracle_apply(pol, soa, variant=1), f"delta of {m} nodes")
    return got


def test_pod_lists_leave_no_resident_snapshot(handle):
    """A call with pod lists drops the resident snapshot: the delta calls evaluate no pod lists."""
    rng = np.random.default_rng(11)
    soa, pods = helpers.random_soa(rng, 5000, with_pods=True)
    pol = policy()
    assert handle.apply_state(pol, soa)[0] == 0
    helpers.assert_same(handle.apply_state(pol, soa, pods), helpers.oracle_apply(pol, soa, pods, variant=0), "with pod lists")
    rc = handle.apply_state_delta(pol, 5000, np.zeros(0, np.int64), {k: soa[k][:0] for k in COLS}, soa["ds_rev"])[0]
    assert rc == INVALID


@pytest.mark.parametrize("fmt", ["wide", "packed"])
@pytest.mark.parametrize("n", [5000, 700_001])
def test_data_abort_keeps_the_snapshot(handle, fmt, n):
    """A reference-level abort (UST_ERR_REVISION_HASH) is an answer about the data: the uploaded snapshot stays
    resident and takes delta updates, on the direct and on the pipelined upload path."""
    rng = np.random.default_rng(100 + n)
    soa, _ = helpers.random_soa(rng, n, wild=True, p_err=20.0 / n)
    pol = policy()
    got = full_call(handle, fmt, pol, soa)
    ref = helpers.oracle_apply(pol, soa, variant=1)
    assert ref[0] == abi.K["UST_ERR_REVISION_HASH"]
    helpers.assert_same(got, ref, f"{fmt} abort")
    delta_matches_oracle(handle, rng, pol, soa, n // 100)


def test_rejected_call_keeps_the_snapshot(handle):
    """A call rejected for its arguments touches nothing: the resident snapshot of the call before stays usable."""
    rng = np.random.default_rng(12)
    n = 5000
    soa, pods = helpers.random_soa(rng, n, with_pods=True)
    pol = policy()
    assert handle.apply_state(pol, soa)[0] == 0
    too_many = dict(soa, ds_rev=np.zeros(128, np.int32))
    assert handle.apply_state_packed(pol, too_many)[0] == INVALID
    bad_off = pods["pod_off"].copy()
    bad_off[n // 2] = bad_off[n // 2 + 1] + 1        # offsets must not decrease
    assert handle.apply_state(pol, soa, {"pod_off": bad_off, "pod_flags": pods["pod_flags"]})[0] == INVALID
    delta_matches_oracle(handle, rng, pol, soa, 50)


@pytest.mark.parametrize("n", [5000, 700_001])
def test_fetch_outputs_after_a_dense_delta(handle, n):
    """ust_fetch_outputs returns the outputs of the last call on the resident snapshot, here a dense delta."""
    rng = np.random.default_rng(13 + n)
    soa, _ = helpers.random_soa(rng, n, wild=True)
    pol = policy()
    assert handle.apply_state(pol, soa)[0] == 0
    _, nxt, act, _, _ = delta_matches_oracle(handle, rng, pol, soa, n // 50)
    rc, fnxt, fact = handle.fetch_outputs(n)
    assert rc == 0
    assert np.array_equal(fnxt, nxt) and np.array_equal(fact, act)
