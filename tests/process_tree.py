"""Run a command that starts processes of its own (torchrun and its ranks) under a time limit, and leave none behind.

torchrun starts every rank in a session of its own, so killing torchrun's process group does not reach the ranks, and
a SIGKILLed torchrun cannot stop them: they are reparented to init and keep the GPU (and the output pipe).  On timeout
`run_tree` therefore sends SIGTERM to the command, whose handler (torchrun's) terminates its workers, waits `grace`
seconds, and then SIGKILLs the process group of every process that was below the command, as well as the command."""
from __future__ import annotations

import os
import signal
import subprocess


def _children() -> dict:
    """{ppid: [pid, ...]} of every process, from /proc/<pid>/stat."""
    kids = {}
    for d in os.listdir("/proc"):
        if not d.isdigit():
            continue
        try:
            with open(f"/proc/{d}/stat") as f:
                stat = f.read()
        except OSError:  # the process ended while we looked
            continue
        ppid = int(stat[stat.rindex(")") + 2:].split()[1])  # "pid (comm) state ppid ..."
        kids.setdefault(ppid, []).append(int(d))
    return kids


def descendants(pid: int) -> list:
    kids, out, todo = _children(), [], [pid]
    while todo:
        for c in kids.get(todo.pop(), []):
            out.append(c)
            todo.append(c)
    return out


def _kill_group_and_process(pid: int) -> None:
    try:
        pgid = os.getpgid(pid)
        if pgid != os.getpgrp():
            os.killpg(pgid, signal.SIGKILL)
        os.kill(pid, signal.SIGKILL)
    except ProcessLookupError:
        pass


def run_tree(cmd, timeout: float, grace: float = 10.0, **popen_kw):
    """Run `cmd` in a new session with stdout and stderr combined -> (returncode, output); returncode is None when
    `timeout` seconds passed, and then no process of the tree is left when this returns."""
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, start_new_session=True,
                         **popen_kw)
    try:
        out, _ = p.communicate(timeout=timeout)
        return p.returncode, out
    except subprocess.TimeoutExpired:
        pass
    tree = descendants(p.pid)
    p.send_signal(signal.SIGTERM)
    try:
        p.wait(grace)
    except subprocess.TimeoutExpired:
        pass
    for pid in [*tree, *descendants(p.pid), p.pid]:
        _kill_group_and_process(pid)
    try:
        out, _ = p.communicate(timeout=grace)
    except subprocess.TimeoutExpired:  # a process started after the snapshot still holds the pipe: stop reading
        p.stdout.close()
        p.wait()
        out = ""
    return None, out
