"""CPU: the rules the wide traceback's planted pairs (tests/wide_trace_cases.py) rely on, and every planted case's
geometry on the C oracle's path under both tie rules -- the catalogue of test_gpu_wide_trace.py, checked without a
GPU."""
import pytest

from tests import wide_trace_cases as W
from tests.helpers import OP_DEL, OP_INS, oracle_arrays

GROUPS = W.all_groups()


def test_pick_kl_matches_the_cost_rule():
    bad = [m for m in range(1, 20001) if W.pick_kl(m) != W.pick_kl_cost(m)]
    assert not bad, bad[:10]


def test_grouping_rows():
    sm = 148
    assert [W.grouping(n, sm) for n in (1, sm, sm + 1, 256 * sm - 1, 256 * sm)] == ["cluster"] * 2 + ["warp"] * 2 + ["thread"]
    assert [W.cluster_c(n, sm) for n in (sm // 3, sm // 3 + 1, sm // 2, sm // 2 + 1, sm)] == [3, 2, 2, 1, 1]


@pytest.mark.parametrize("gi", range(len(GROUPS)), ids=[g.name for g in GROUPS])
def test_planted_geometry(gi):
    g = GROUPS[gi]
    assert len({c.name for c in g.cases}) == len(g.cases)
    ge = {}
    for c in g.cases:
        for tie_gt in (False, True):
            exp = oracle_arrays(g.ref, c.read, g.scores, tie_gt=tie_gt, lowmem=not tie_gt)
            c.assert_geometry(exp, g.scores, g.ref, g.kl)
            if not tie_gt:
                ge[c.name] = exp
            elif c.name.rsplit("/", 1)[1].startswith("tie-"):
                assert (exp["ops"] != ge[c.name]["ops"]).any() or exp["beginnings"][0] != ge[c.name]["beginnings"][0], \
                    f"{c.name}: the tie rules chose the same path"


def test_catalogue_covers_every_item():
    """Every gap length and position, for both ops, in every class the catalogue runs with cheap gaps."""
    scores = (5, -3, -1)
    for kl in W.SCORE_SETS[scores]:
        names = [c.name.rsplit("/", 1)[1] for c in W.gap_group(kl, scores).cases]
        positions = [p[0] for p in W._tile_positions(kl)] + (["seam-jump", "seam-above", "seam-below"] if kl > 8 else [])
        for ev, op in (("ins", OP_INS), ("del", OP_DEL)):
            lengths = {int(n[3:].split("@")[0]) for n in names if n.startswith(ev) and n.split("@")[1] not in ("round-edge", "narrow")}
            fits = {L for L in W.GAP_LENGTHS(kl) if 2 * W.flank(L, scores) + (L if op == OP_INS else 0) <= W.KL_READS[kl][1]}
            assert lengths == fits, (kl, ev, sorted(fits - lengths))
            assert {n.split("@")[1] for n in names if n.startswith(ev)} >= set(positions), (kl, ev)
        if kl > 8:
            assert f"ins{32 * kl + 1}@round-edge" in names and {"del129@narrow", "del257@narrow"} <= set(names), kl
    # paths that end in every round 0 .. 4, on a round's first and last lane-row too
    ends = [c.name.rsplit("/", 1)[1] for kl in W.SCORE_SETS[scores] for c in W.ends_group(kl, scores).cases]
    for R in range(5):
        assert any(n.startswith(f"round{R}-mid") for n in ends), R
        assert any(n.startswith(f"round{R}-first") for n in ends) or R == 0, R
        assert any(n.startswith(f"round{R}-last") for n in ends), R
