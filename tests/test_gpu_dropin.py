"""The C++ drop-in front end (include/superbblas.h) exercised by a caller written against the
reference's API (tests/cxx/dropin_test.cpp), run on the GPU."""
import os
import subprocess

import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def test_cxx_dropin_program():
    exe = os.path.join(HERE, "cxx", "dropin_test")
    if not os.path.exists(exe):
        r = subprocess.run(["make", "-C", os.path.join(HERE, "cxx")], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Everything went ok!" in r.stdout


def _run_reference_suite(args, timeout=900):
    exe = os.path.join(HERE, "cxx", "ref_contract_wrapper")
    if not os.path.exists(exe):
        pytest.skip("tests/cxx/ref_contract_wrapper not built (needs /root/reference at build time)")
    r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "Everything went ok!" in r.stdout


@pytest.mark.parametrize("nt,typ", [(0, "d"), (1, "d"), (0, "z"), (1, "z"), (1, "s"), (0, "c")])
def test_reference_own_contraction_suite(nt, typ):
    """The reference's tests/contract.cpp, unmodified (included from /root/reference at build time
    by tests/cxx/ref_contract_wrapper.cpp), compiled against include/superbblas.h and run on the GPU:
    every label-group arrangement, order, conjugation, alpha/beta and partition of its enumeration
    (1.3 million contractions over the four parametrisations)."""
    _run_reference_suite(["--nt=%d" % nt, "--type=%s" % typ])


def test_reference_own_dist_program():
    """The reference's tests/dist.cpp, unchanged (tests/cxx/ref_dist_wrapper.cpp includes it from
    /root/reference at build time), against include/superbblas.h: partition known answers and
    make_hole checks (they throw on a wrong answer), then its permuting copies, shifts, halo fills,
    detail::xgemm_batch_strided shapes and contractions with host and with GPU components.
    Log of a run on a B200: profiles/r1_reference_dist_cpp_on_b200.log."""
    exe = os.path.join(HERE, "cxx", "ref_dist_wrapper")
    if not os.path.exists(exe):
        pytest.skip("tests/cxx/ref_dist_wrapper not built (needs /root/reference at build time)")
    r = subprocess.run([exe, "--dim=16 16 16 32 16", "--reps=2"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert ">>> GPU tests:" in r.stdout and "Time in copying halos out" in r.stdout


def test_sb_debug_2_self_check_of_the_dropin_program():
    """SB_DEBUG=2 (reference: tests/Makefile:78-79 runs its dist test that way; dist.h:2282-2285):
    every copy of the drop-in program first verifies itself on index-valued mock tensors through
    the whole path; a wrong element throws."""
    env = dict(os.environ, SB_DEBUG="2")
    exe = os.path.join(HERE, "cxx", "dropin_test")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "Everything went ok!" in r.stdout, (r.stdout + r.stderr)[-2000:]


def test_sb_debug_2_self_check_of_every_copy():
    """SB_DEBUG=2 on every copy of the reference's tests/dist.cpp (as
    test_sb_debug_2_self_check_of_the_dropin_program does for the drop-in program)."""
    env = dict(os.environ, SB_DEBUG="2")
    exe = os.path.join(HERE, "cxx", "ref_dist_wrapper")
    if not os.path.exists(exe):
        pytest.skip("tests/cxx/ref_dist_wrapper not built (needs /root/reference at build time)")
    r = subprocess.run([exe, "--dim=4 4 4 8 4", "--reps=1"], capture_output=True, text=True, timeout=600,
                       env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "Time in copying halos out" in r.stdout


# The wrapper also accepts --components=N (several components per process) and --cpu (host contexts,
# staged through the GPU); they run the same enumeration but take much longer, so they are not part of
# the default GPU test run.
