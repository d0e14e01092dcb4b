"""The CPU restatement on every case of the live comparisons with the reference, against the digests stored in
tests/golden/restatement_digests.json (see restatement_snapshots.py): runs without the reference's sources."""
import pytest

import restatement_snapshots as rs

CASES = rs.cases()


def test_every_case_has_a_stored_digest():
    assert sorted(rs.stored()) == sorted(CASES)


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_matches_stored_digest(port, name):
    assert rs.digest(CASES[name](port)) == rs.stored()[name], f"{name}: the restatement's output changed"
