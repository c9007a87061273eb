"""Every `_begin` entry point of include/superbblas_b200.h refuses a null `request` before it reads any
other argument or touches a device: it returns 1 with "<name>_begin: null request" and writes nothing.
Each call runs in a child process, so that a crash fails its own case instead of the run."""
import os
import re
import subprocess
import sys

import superbblas_b200 as sb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "superbblas_b200.h")).read()
BEGINS = dict(re.findall(r"\bint\s+(sbb_\w+_begin)\s*\(([^)]*)\)\s*;", HEADER))

# Every argument is null (0 for the integers), except the handle out-pointer of the creates, which holds
# a value that the call must leave alone
CHILD = r"""
import ctypes, sys
lib = ctypes.CDLL(sys.argv[1])
lib.sbb_last_error.restype = ctypes.c_char_p
bsr = ctypes.c_void_p(0x5bb)
args = [ctypes.byref(bsr) if p == "out" else None for p in sys.argv[3:]]
rc = getattr(lib, sys.argv[2])(*args)
print(rc, bsr.value == 0x5bb, lib.sbb_last_error().decode())
"""


def test_null_request_is_refused():
    assert sorted(BEGINS) == sorted("sbb_%s_begin" % n for n in (
        "copy", "cholesky", "inversion", "trsm", "gesm", "bsr_krylov", "create_bsr", "create_kron_bsr"))
    got = {}
    for name, decl in sorted(BEGINS.items()):
        params = [p.strip() for p in decl.split(",")]
        assert params[-1] == "sbb_request_t *request", name
        kinds = ["out" if re.match(r"sbb_bsr_t\s*\*", p) else "null" for p in params]
        r = subprocess.run([sys.executable, "-c", CHILD, sb.LIB_PATH, name] + kinds, capture_output=True,
                           text=True, timeout=120)
        got[name] = r.stdout.strip() if r.returncode == 0 else "exit %d" % r.returncode
    assert got == {name: "1 True %s: null request" % name[len("sbb_"):] for name in BEGINS}
