"""-m gpu: the number of kernels one call launches (b200mpc_launch_count) under each launch schedule of the solver.
A default solve at N = 25 is DESIGN §4's 84 launches: init, 20 x (factor, forward, step), 16 repack attempts, 6
conditional hand-overs and the finisher.  Every count holds for a captured CUDA graph, its replay and plain launches; a
graph that a setting change failed to replace would replay the old count."""
import pytest

import udacitympc_b200 as mp
from udacitympc_b200 import synth

pytestmark = pytest.mark.gpu

# (N, B, settings made before the first call, call, launches per call)
CASES = {
    "default": (25, 4096, [], "solve", 84),
    "traj": (25, 4096, [], "traj", 85),                           # + the trajectory transpose
    "split": (25, 16384, [], "solve", 336),                       # 4 concurrent parts of 84
    "latency": (25, 100, [], "solve", 1),                         # the cooperative kernel alone
    "closed_loop": (25, 300, [], "loop", 3),                      # 3 steps of 1
    "fused": (25, 4096, [("set_solver_mode", 1, 0, -1)], "solve", 1),
    "fixed_rounds": (25, 3999, [("set_solver_mode", 0, 12, 0), ("set_batch_split", 1)], "solve", 46),
    "no_compaction": (25, 4096, [("set_compaction", 0.0)], "solve", 56),
    "no_handover": (25, 4096, [("set_handover", 0, 14)], "solve", 70),
    "pipelined": (25, 16384, [("set_pipeline", 2, 1024)], "solve", 132),   # bulk 80 + tail 52
    # N = 100: 4 parts of 584 (init, 120 x 3 sweeps, 116 repack attempts, 106 conditional hand-overs, the finisher)
    "long_default": (100, 16384, [], "solve", 2336),
    # N = 100: bulk 480 (reset, init, 120 x 3 sweeps, 117 repacks, finisher) + tail 2477 (600 x (3 sweeps, repack),
    # 75 hand-overs to the cooperative kernel, one every 8 rounds, then one more and the finisher)
    "long_pipelined": (100, 16384, [("set_pipeline", 2, 1024)], "solve", 2957),
    "long_latency": (200, 40, [], "solve", 1),                    # the cooperative kernel, one problem per block
    "long_rounds": (200, 40, [("set_solver_mode", 0, 12, 0)], "solve", 46),
}


@pytest.fixture(params=["graphs", "plain"])
def launches(request, monkeypatch):
    monkeypatch.setenv("B200MPC_NO_GRAPHS", "1" if request.param == "plain" else "0")
    return request.param


def launches_of(m, how, st, cf):
    n = m.launch_count()
    if how == "loop":
        m.closed_loop(st, cf, 3)
    else:
        m.solve_batch(st, cf, want_traj=how == "traj")
    return m.launch_count() - n


@pytest.mark.parametrize("case", sorted(CASES))
def test_launches_per_call(case, launches):
    N, B, settings, how, expected = CASES[case]
    st, cf = synth.line_problems(B)
    with mp.MPC(device=0, N=N, max_iter=400 if N > 25 else 3000) as m:
        for name, *args in settings:
            getattr(m, name)(*args)
        assert [launches_of(m, how, st, cf) for _ in range(2)] == [expected, expected]   # capture, replay


def test_setting_changes_take_effect_on_the_next_call(launches):
    """One handle, settings changed between calls: every setter that changes the launch sequence is seen by the next
    call.  The hand-over change comes last: with hand-over off the B = 16384 calls would run 18 and 16 fixed rounds."""
    st, cf = synth.line_problems(16384)
    steps = [
        (4096, [], 84),
        (4096, [("set_compaction", 0.0)], 56),
        (4096, [("set_compaction", 0.7, 4)], 84),
        (4096, [("set_solver_mode", 1, 0, -1)], 1),
        (4096, [("set_solver_mode", 0, 0, -1)], 84),
        (16384, [("set_batch_split", 1)], 84),
        (16384, [("set_batch_split", 4)], 336),
        (4096, [("set_handover", 0, 14)], 70),
    ]
    with mp.MPC(device=0) as m:
        for B, settings, expected in steps:
            for name, *args in settings:
                getattr(m, name)(*args)
            assert launches_of(m, "solve", st[:B], cf[:B]) == expected, (B, settings)
