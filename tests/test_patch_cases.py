"""The scripted scatter sequences of ``patch_cases`` on the CPU: each stays a small update, keeps the matrix Hermitian
and its zero pattern where it should, and carries the path the plain rebuild rule gives."""

import numpy as np
import pytest

import patch_cases as pc
from oracle import bdg_oracle as orc


@pytest.fixture(scope="module", params=pc.SEQUENCES, ids=[f"{g}-{m}" for g, m in pc.SEQUENCES])
def seq(request):
    return pc.sequence(*request.param)


def test_every_update_is_small(seq):
    for step in seq.steps:
        assert step.n_written * 4 <= len(seq.indices), step.name


def test_hermitian_except_the_one_sided_write(seq):
    assert pc.hermitian(seq.indptr, seq.indices, seq.initial)
    for step in seq.steps:
        assert step.hermitian == (step.name != "U10"), step.name
        dev = orc.hermitian_deviation(seq.indptr, seq.indices, step.data)
        assert dev == 0.0 if step.hermitian else dev > 1e-6, step.name   # (1e-6: the check's tolerance)


def test_zero_pattern_changes_only_when_a_block_is_zeroed(seq):
    before = pc.nonzero(seq.initial)
    for step in seq.steps:
        after = pc.nonzero(step.data)
        assert np.array_equal(before, after) == (step.name != "U11"), step.name
        before = after


def test_labels_follow_the_rebuild_rule(seq):
    """Rebuild iff the zero pattern changes, or (where a dictionary exists) an off-site block is not real-diagonal
    after the step while every off-site block was before it."""
    before = seq.initial
    for step in seq.steps:
        pattern = not np.array_equal(pc.nonzero(before), pc.nonzero(step.data))
        breaks_diag = pc.offsite_real_diagonal(seq.indptr, seq.indices, before) and \
            not pc.offsite_real_diagonal(seq.indptr, seq.indices, step.data)
        want = "rebuild" if pattern or (seq.dictionary and breaks_diag) else "patch"
        assert step.path == want, step.name
        before = step.data


def test_the_sequences_reach_what_they_are_for(seq):
    """U2 takes on-site blocks off real-diagonal, U4 writes both orientations of every bond it names, U5 and U6 are
    rebuilds exactly where real-diagonal hopping met a dictionary."""
    steps = {s.name: s for s in seq.steps}
    assert not pc.onsite_real_diagonal(seq.indptr, seq.indices, steps["U2"].data)
    h_i, h_j = steps["U4"].packed[:2]
    assert {(int(a), int(b)) for a, b in zip(h_i, h_j)} == {(int(b), int(a)) for a, b in zip(h_i, h_j)}
    diag_hopping = seq.model in ("diag", "normal") and seq.dictionary
    assert steps["U5"].path == ("rebuild" if diag_hopping else "patch")
    assert steps["U6"].path == "patch" and steps["U11"].path == "rebuild"
