"""CPU tests of the refusals of b200sa_hamming_batch and b200sa_levenshtein_batch (include/b200sa.h) that come before
the indices are read.

As in test_api_errors.py, each call runs on a fresh host thread, so a non-empty b200sa_last_error() proves that the
refusal wrote one, and without a device each refusal still comes back as its own code.  The refusals that need a
built index (NOT_BUILT, a mismatched or records reverse index) are in test_gpu_hamming.py and test_gpu_levenshtein.py.
"""
import ctypes as C
import threading

import numpy as np
import pytest

BAD_ARGUMENT, TOO_LARGE = 2, 4

# Handles for refusals that happen before a handle is read: zeroed host memory, never dereferenced.
_UNREAD = np.zeros(1 << 20, np.uint8)
_UNREAD_REV = np.zeros(1 << 20, np.uint8)

# every test runs on each entry point, with the budgets above its limit: k <= 8 mismatches, k <= 4 edits
pytestmark = pytest.mark.parametrize("search", [
    pytest.param(("b200sa_hamming_batch", (9, 100, 2 ** 32 - 1)), id="hamming"),
    pytest.param(("b200sa_levenshtein_batch", (5, 8, 2 ** 32 - 1)), id="levenshtein"),
])


@pytest.fixture(scope="module")
def lib():
    import stralg_b200
    return stralg_b200.load()


def ptr(a):
    return C.c_void_p(a.ctypes.data)


def refused(lib, search, code, *args):
    err = C.c_int(-1)
    out = {}

    def run():
        out["h"] = getattr(lib, search[0])(*args, C.byref(err))
        out["msg"] = lib.b200sa_last_error()

    t = threading.Thread(target=run)
    t.start()
    t.join()
    assert not out["h"]
    assert err.value == code, (err.value, out["msg"])
    assert out["msg"]


def test_null_arguments(lib, search):
    h, rv = ptr(_UNREAD), ptr(_UNREAD_REV)
    pats = np.ones(8, np.uint8)
    refused(lib, search, BAD_ARGUMENT, None, rv, ptr(pats), None, 8, 1, 1)
    refused(lib, search, BAD_ARGUMENT, h, None, ptr(pats), None, 8, 1, 1)   # rev_idx is required
    refused(lib, search, BAD_ARGUMENT, h, rv, None, None, 8, 1, 1)          # no patterns with npat > 0


def test_budget_above_limit(lib, search):
    h, rv = ptr(_UNREAD), ptr(_UNREAD_REV)
    pats = np.ones(8, np.uint8)
    for k in search[1]:
        refused(lib, search, BAD_ARGUMENT, h, rv, ptr(pats), None, 8, 1, k)


def test_decreasing_offsets(lib, search):
    h, rv = ptr(_UNREAD), ptr(_UNREAD_REV)
    pats = np.ones(8, np.uint8)
    off = np.array([0, 5, 3], np.uint64)
    refused(lib, search, BAD_ARGUMENT, h, rv, ptr(pats), ptr(off), 0, 2, 1)


def test_pattern_longer_than_65000(lib, search):
    h, rv = ptr(_UNREAD), ptr(_UNREAD_REV)
    pats = np.ones(65004, np.uint8)
    refused(lib, search, TOO_LARGE, h, rv, ptr(pats), None, 65001, 1, 1)
    off = np.array([0, 3, 65004], np.uint64)
    refused(lib, search, TOO_LARGE, h, rv, ptr(pats), ptr(off), 0, 2, 1)
