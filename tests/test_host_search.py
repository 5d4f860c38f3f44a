"""CPU: csrc/host_search.h (the rotation queue of the host schedulers) pops in exactly the order of std::priority_queue over the
reference's ROTNODE (jly_goicp.h:59-73), ties between equal (lb, w) keys included, and prune_in_pop_order leaves the queue the
reference's pruning loop (jly_goicp.cpp:843-853) leaves.  prune_any_order keeps the same nodes in a different heap, so it must
disagree on some sequence: that is why the exact-order scheduler may not use it.  The header is plain C++, so no GPU is needed."""
import os
import subprocess

from conftest import ROOT


def test_host_queue_matches_reference_priority_queue(tmp_path):
    exe = str(tmp_path / "host_search_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "go-icp-protein-cavities_b200", "csrc"),
                           "-o", exe, os.path.join(ROOT, "tests", "host_search_check.cpp"), "-lm"])
    out = subprocess.run([exe, "2000"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:]
    f = out.stdout.split()
    assert f[0] == "cases" and int(f[1]) == 2000, out.stdout
    assert int(f[3]) == 0 and int(f[5]) == 0, out.stdout
    assert int(f[7]) > 0, out.stdout   # the check can tell the two prunes apart
