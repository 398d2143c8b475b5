"""tests/process_tree.run_tree on the CPU: a 2-rank torchrun whose ranks never finish -- one of them ignoring SIGTERM --
is stopped at its time limit, the call returns promptly, and no rank survives it (torchrun starts each rank in a
session of its own, so killing torchrun's process group alone would leave them running)."""
import os
import sys
import textwrap
import time

from tests.process_tree import run_tree

WORKER = textwrap.dedent("""
    import os, signal, sys, time
    rank = int(os.environ["RANK"])
    if rank == 1:
        signal.signal(signal.SIGTERM, signal.SIG_IGN)  # only SIGKILL stops this one
    open(os.path.join(sys.argv[1], f"pid_{rank}"), "w").write(str(os.getpid()))
    time.sleep(600)
""")


def _alive(pid: int) -> bool:
    try:
        with open(f"/proc/{pid}/stat") as f:
            return f.read().rsplit(")", 1)[1].split()[0] != "Z"  # a zombie has ended
    except OSError:
        return False


def test_timeout_leaves_no_rank_behind(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    timeout, grace = 30, 5
    t0 = time.time()
    rc, _ = run_tree([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", "2",
                      str(script), str(tmp_path)], timeout, grace=grace, env=env)
    took = time.time() - t0
    assert rc is None
    assert took < timeout + 2 * grace + 5, f"returned after {took:.1f} s"
    pids = [int((tmp_path / f"pid_{r}").read_text()) for r in range(2)]
    assert not [p for p in pids if _alive(p)], "a rank outlived run_tree"


def test_normal_exit_returns_code_and_output():
    rc, out = run_tree([sys.executable, "-c", "print('hello'); raise SystemExit(3)"], 60)
    assert rc == 3 and out.strip() == "hello"
