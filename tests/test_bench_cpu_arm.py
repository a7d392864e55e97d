"""bench.py's CPU arm (`--impl reference` / `cpu_baseline`) runs without a GPU: the sequential PUCT oracle in lock step over a
few games with the fp32 network on torch's CPU kernels.  A small instance here keeps the arm from rotting."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def test_cpu_arm_small_instance():
    import bench_mcts as B
    arm = B.CpuSelfPlay(sims=6, n_games=3)
    s, e, dt = arm.run_waves(1)
    assert s == 3 and e <= 3 and dt > 0                       # one root expansion per game
    s2, e2, _ = arm.run_waves(8)                              # crosses a move boundary (6 sims per move)
    info = [t.info() for t in arm.trees]
    assert all(i["ply"] >= 1 for i in info) and s2 >= 8 * 3 - 3
    assert arm.evals + arm.served >= s + s2 - 3               # every non-terminal simulation was evaluated or served
    assert arm.threads == (os.cpu_count() or 1)               # not the launcher's OMP_NUM_THREADS


def test_random_start_lines_are_legal_positions():
    import numpy as np
    import bench_mcts as B
    from oracle import kv_oracle as O
    lines = B.random_start_lines(16, 5, 1234)
    moves, counts, flags, _ = O.movegen(lines.copy())
    assert (counts > 0).all() and (lines[:, 13:] == 0).all()
    assert np.array_equal(lines, B.random_start_lines(16, 5, 1234))      # seeded


def test_dump_outputs_directory_checked_before_gpu_work(tmp_path, monkeypatch):
    """A --dump-outputs directory that cannot be made is an argument error (exit 2) before the benchmark starts."""
    import pytest
    import bench
    blocker = tmp_path / "a_file"
    blocker.write_text("")
    monkeypatch.setattr(sys, "argv", ["bench.py", "--dump-outputs", str(blocker / "out")])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2


def test_dump_games_sample_bounds_the_records():
    """At the bench's size (4 096 games, 3 warm-up + 5 timed moves): a fixed sample of games, at most DUMP_RECORDS records
    (one per game and move), so the dump stays far below 64 MB."""
    import numpy as np
    import bench_mcts as B
    g = B.dump_games(4096, 8)
    assert len(g) * 8 <= B.DUMP_RECORDS and len(set(g.tolist())) == len(g) and np.array_equal(g, np.sort(g))
    assert np.array_equal(g, B.dump_games(4096, 8)) and len(g) == 1024
    assert B.DUMP_RECORDS * (12 * 64 * 4 + 3 * 8) + len(g) * (64 * 4 + 8) < 28e6
    assert np.array_equal(B.dump_games(40, 5), np.arange(40))
