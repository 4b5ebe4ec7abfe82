"""CPU: the oracles at the int32 edge of the call domain.  An align call accepts max(|match|, |mismatch|, |gap|) *
(m + n + 2) < 2^30 (check_call, swb_align.cu); the GPU tests of tests/test_gpu_score_domain.py compare the engine with
the C oracle at that edge, where scores reach about 10^9.  Here the C oracle, its low-memory variant and the
independent Python twin (oracle/sw_twin.py) must agree on short pairs at the same score sets.  The file also holds
what the GPU tests derive on the host: the edge's score bounds and the wide path's band-edge read lengths."""
import random

import pytest

import oracle
from oracle import sw_twin

DOMAIN = 1 << 30

# the wide-path workload at the edge: reads of up to EDGE_M rows against references of up to EDGE_N bases
EDGE_M, EDGE_N = 600, 1000
EDGE_L = EDGE_M + EDGE_N + 2
BIG_IN = (DOMAIN - 1) // EDGE_L               # largest |score| the call accepts for that workload
BIG_OUT = BIG_IN + 1                          # smallest it refuses


def edge_score_sets(big):
    """big as the match, as a negative gap and as a positive mismatch."""
    return [(big, -3, -4), (5, -3, -big), (5, big, -4)]


def wrap32(x):
    x &= 0xFFFFFFFF
    return x - (1 << 32) if x & 0x80000000 else x


def _pick_kl(m):
    """Rows per lane of the wide path (pick_kl, swb_wide_host.cu): the fewest band steps, 3 ops per row + 25 per step."""
    best, best_cost = 0, 0
    for kl in (8, 16, 32):
        cost = -(-m // (32 * kl)) * (3 * kl + 25)
        if not best or cost <= best_cost:
            best, best_cost = kl, cost
    return best


# read lengths with two or more bands of 32 * KL rows that sit on a band edge: a multiple, one row less, one row more
BAND_EDGE_LENGTHS = [m for m in range(257, 2050)
                     if m % (32 * _pick_kl(m)) in (0, 1, 32 * _pick_kl(m) - 1) and m > 32 * _pick_kl(m)]


def test_band_edge_lengths():
    assert BAND_EDGE_LENGTHS == [1025, 1535, 1536, 2047, 2048, 2049]
    assert {_pick_kl(m) for m in BAND_EDGE_LENGTHS} == {16, 32}


def test_edge_constants():
    assert BIG_IN * EDGE_L < DOMAIN <= BIG_OUT * EDGE_L
    assert wrap32(2**31) == -2**31 and wrap32(2**32 + 5) == 5 and wrap32(-1) == -1


def _pairs(seed):
    rnd = random.Random(seed)

    def rand(n):
        return "".join(rnd.choice("ACGT") for _ in range(n))
    a = rand(60)
    anti = a.translate(str.maketrans("ACGT", "CGTA"))               # mismatches a everywhere
    return [(a, a[10:45]), (a, anti[5:50]), (a, a[:20] + rand(7) + a[30:55]), ("AC" * 30, "AC" * 11 + "G"),
            (rand(45), rand(38)), (a[:25], a)]


def _agree(ref, read, scores):
    exp = oracle.align(ref, read, *scores)
    low = oracle.align(ref, read, *scores, lowmem=True)
    score, cells, sites = sw_twin.align(ref, read, *scores)
    assert (low.score, low.cells, low.sites) == (exp.score, exp.cells, exp.sites), scores
    assert (score, cells, sites) == (exp.score, exp.cells, exp.sites), scores
    assert oracle.score(ref, read, *scores) == (exp.score, len(exp.cells))
    gt = oracle.align(ref, read, *scores, tie_gt=True)
    assert sw_twin.align_gt(ref, read, *scores) == (gt.score, gt.cells, gt.sites), scores
    return exp.score


@pytest.mark.parametrize("scores", edge_score_sets(BIG_IN) + edge_score_sets(BIG_OUT), ids=lambda s: "%d,%d,%d" % s)
def test_oracles_agree_at_the_wide_edge(scores):
    best = max(_agree(ref, read, scores) for ref, read in _pairs(sum(scores) % 1000))
    assert best >= 35 * max(scores[:2])                                 # a run of 35 diagonal steps of the larger score


def test_oracles_agree_at_each_pairs_own_edge():
    """The largest |score| each short pair itself would be accepted with, and a positive gap at that size: the
    maximum then lies near 2^30, the largest value a call inside the domain can produce."""
    for ref, read in _pairs(7):
        big = (DOMAIN - 1) // (len(ref) + len(read) + 2)
        for scores in edge_score_sets(big) + [(1, -1, big), (big, big, big)]:
            s = _agree(ref, read, scores)
            assert 0 <= s < DOMAIN
        assert _agree(ref, read, (1, -1, big)) == big * (len(ref) + len(read) - 1)   # the all-gap path to (m, n)
