"""CPU checks of the two re-formulations inside the LSD region walker (structure-slam-pointline_b200/csrc/line.cu) against
plain sequential models of the reference algorithm (OpenCV lsd.cpp region_grow / reduce_region_radius):
 * speculative multi-accept rounds of l_region_grow == the sequential neighbour scan (same accepted set, order, float sums);
 * ballot-based compaction of l_reduce_region_radius == swap-with-last removal (same resulting list order)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def test_speculative_grow_matches_sequential_scan():
    import sim_speculative_grow as m
    acc, rounds = m.run(iters=3000, seed=7)
    assert acc > 1.0 and rounds < acc          # several acceptances per round on average


def test_reduce_radius_compaction_matches_swap_with_last():
    import sim_reduce_radius as m
    assert m.run(iters=1500, seed=3)

