"""CPU: the ownership protocol of the credit pool's shared entries (state-block control words, attachment entries), one
race at a time.  tests/native/pool_ownership.cpp includes gh_pool.cpp and drives each interleaving through its
transition functions deterministically:
 a  a committer preempted between its publication CAS and freeing the superseded block cannot free that block after
    another handle recycled and claimed it;
 b  the same across processes, with a client stopped (SIGSTOP) right after its publication CAS and resumed later;
 c  a recycler's judgement of a dead owner's word does not carry over to a claim made after the owner's attachment entry
    was re-taken, and a dead owner's blocks are recycled even if its entry is re-taken before they are;
 d  the reaper's last step frees only an entry that is still REAPING, and a closing owner's entry reads FREE before its
    byte is unlocked."""
import os
import subprocess as sp
import tempfile

import pytest

import kubeshare_b200 as kb

GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


@pytest.fixture(scope="module")
def exe():
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "pool_ownership")
        cmd = [GXX, "-std=c++17", "-O1", "-g", "-DGEMHOOK_FAULT_INJECTION", "-I/usr/local/cuda/include",
               os.path.join(kb.ROOT, "tests", "native", "pool_ownership.cpp"), os.path.join(kb.HERE, "csrc", "gh_core.cpp"),
               "-o", out, "-ldl", "-lpthread"]
        p = sp.run(cmd, stdout=sp.PIPE, stderr=sp.PIPE)
        assert p.returncode == 0, p.stderr.decode()[-3000:]
        yield out


@pytest.mark.parametrize("case", ["a", "b", "c", "d"])
def test_pool_ownership_race(exe, case):
    with tempfile.TemporaryDirectory() as tmp:
        p = sp.run([exe, case, tmp], stdout=sp.PIPE, stderr=sp.PIPE, timeout=60)
        assert p.returncode == 0 and p.stdout.strip() == b"ok", (p.returncode, p.stderr.decode()[-3000:])
