"""ctypes wrapper around ``tests/fsai_oracle.c``, the test oracle of the FSAI kernel (``dp_fsai_f64``).

The C file is compiled on first use into a private temporary directory (the checkout may be read-only), with the flags of
the project's other C oracle: ``-ffp-contract=off`` keeps every operation rounded separately, like the kernel.
"""

from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_SRC = Path(__file__).resolve().parent / "fsai_oracle.c"
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = Path(tempfile.mkdtemp(prefix="fsai_oracle_"))
        atexit.register(shutil.rmtree, out, ignore_errors=True)
        so = out / "libfsai_oracle.so"
        subprocess.run([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                        "-Wextra", "-shared", "-o", str(so), str(_SRC), "-lm"], check=True, capture_output=True)
        _lib = ctypes.CDLL(str(so))
        _lib.oracle_fsai.restype = ctypes.c_int
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def fsai(a_rowptr, a_col, a_val, u_rowptr, u_col, fp32: bool = True):
    """FSAI values of ``U = L^T`` on the pattern ``(u_rowptr, u_col)`` for the full symmetric ``A`` (``dp_fsai_f64``'s
    arithmetic order). Raises ``ValueError`` on a structure error and ``FloatingPointError`` on a non-positive pivot."""
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    a_rowptr, a_col, u_rowptr, u_col = i32(a_rowptr), i32(a_col), i32(u_rowptr), i32(u_col)
    a_val = np.ascontiguousarray(a_val, dtype=np.float64)
    n = u_rowptr.shape[0] - 1
    out = np.zeros(u_col.shape[0], np.float64)
    status = lib().oracle_fsai(ctypes.c_int(n), _p(a_rowptr), _p(a_col), _p(a_val), _p(u_rowptr), _p(u_col),
                               ctypes.c_int(int(fp32)), _p(out))
    if status == 5:
        raise ValueError("FSAI: a row of U does not start with its diagonal, is not ascending, is longer than 32 "
                         "entries, or A misses a diagonal entry")
    if status:
        raise FloatingPointError("FSAI: non-positive pivot (A is not SPD)")
    return out
