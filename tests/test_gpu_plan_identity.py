"""Launch plans stay what they were: the stats and launch info of every committed batch of tests/golden/make_golden_plan.py
against the fixture it wrote (cells, useful cells, pairs, 32-bit entries and uploaded bytes).  Stripe heights depend on
the SM count, so the fixture only applies to a device with the count it was made on."""
import sys

import pytest

from conftest import GOLDEN_DIR, load_golden

sys.path.insert(0, GOLDEN_DIR)
import make_golden_plan  # noqa: E402

pytestmark = pytest.mark.gpu

FIXTURE = load_golden("plan_fingerprints")
CASES = make_golden_plan.cases()


def test_fixture_covers_every_case():
    assert sorted(FIXTURE["cases"]) == sorted(CASES)


@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_matches_fixture(engine, name):
    sm = engine.device_info()["sm_count"]
    if sm != FIXTURE["sm_count"]:
        pytest.skip(f"fixture made on a device with {FIXTURE['sm_count']} SMs, this one has {sm}")
    assert CASES[name]() == FIXTURE["cases"][name], name
