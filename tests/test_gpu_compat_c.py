"""The reference's OWN C tests and read-mapper, compiled unchanged and linked against the drop-in
(VERDICT r1 item 4; SURVEY 7.1 step 2: "suffix_array_test.c, bwt_test.c, match_test.c, serialise_test.c
must compile against compat/ unchanged and pass").

oracle/Makefile (target `compat`, REFERENCE=<stralg source tree>) builds them into oracle/_ref/compat/
from the sources where they lie in that tree (tests/stralg/*_test.c:main,
tools/readmappers/bwt_readmapper/bwt_readmapper.c), with every symbol libstralg_b200.so exports renamed
away in the reference's helper objects, so the hot-path calls can only bind to the drop-in.  The stralg
sources are not part of this repository: where `make compat` found no such tree (it then writes
oracle/_ref/compat/reference-absent) the tests skip; a program missing after a build from the tree fails.
STRALG_B200_TRACE=1 makes the drop-in report, at exit, how many calls it served.
"""
import hashlib
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

COMPAT = os.path.join(ROOT, "oracle", "_ref", "compat")
GOLD = os.path.join(ROOT, "tests", "golden", "readmapper")


def _need(name):
    p = os.path.join(COMPAT, name)
    if not os.path.exists(p):
        if not os.path.exists(os.path.join(COMPAT, "reference-absent")):
            pytest.fail(f"oracle/_ref/compat/{name} is missing: run `make -C oracle compat`")
        pytest.skip(f"oracle/_ref/compat/{name} not built: it is compiled from the stralg sources, which are not "
                    "part of this repository (`make -C oracle compat REFERENCE=<stralg source tree>`)")
    return p


def _run(cmd, cwd, env_extra=None, timeout=600):
    env = dict(os.environ, STRALG_B200_TRACE="1")
    env.update(env_extra or {})
    r = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, timeout=timeout)
    return r


def _served(stderr):
    m = re.search(rb"stralg_b200: served constructions=(\d+) tables=(\d+) exact_iters=(\d+) approx_iters=(\d+)", stderr)
    assert m, "the drop-in did not report: " + stderr[-500:].decode(errors="replace")
    return [int(x) for x in m.groups()]


@pytest.mark.parametrize("test,args,expect", [
    ("suffix_array_test", [], "constructions"),        # tests/stralg/suffix_array_test.c:205-234
    ("bwt_test", [], "tables"),                        # tests/stralg/bwt_test.c:187-189
    ("match_test", [], "exact_iters"),                 # tests/stralg/match_test.c:682-696
    ("match_test", ["the", "test-data/modest-proposal.txt"], "exact_iters"),
    ("match_test", ["ababaaba", "test-data/repetitive-string.txt"], "exact_iters"),
    ("serialise_test", [], "tables"),                  # tests/stralg/serialise_test.c:13-43
    ("remap_test", [], None),
    ("approx_match_test", [], "approx_iters"),         # tests/stralg/approx_match_test.c:228-259, 360
])
def test_reference_c_test_passes_against_the_drop_in(engine, test, args, expect):
    exe = _need(test)
    r = _run([exe] + args, COMPAT)
    assert r.returncode == 0, (test, args, r.returncode, r.stderr[-1500:].decode(errors="replace"))
    if expect:
        c = dict(zip(["constructions", "tables", "exact_iters", "approx_iters"], _served(r.stderr)))
        assert c[expect] > 0, (test, c)
        print(f"[compat-c] {test} {' '.join(args)}: rc 0, drop-in served {c}")


def _readmapper(exe, tmp_path, env_extra=None):
    """`-p ref.fa` then `-d k ref.fa reads.fq` exactly as tests/golden/readmapper/meta.json records."""
    work = tmp_path / "rm"
    work.mkdir()
    for f in ("ref.fa", "reads.fq", "reads_d1.fq"):
        shutil.copy(os.path.join(GOLD, f), work / f)
    r = _run([exe, "-p", "ref.fa"], work, env_extra)
    assert r.returncode == 0, r.stderr[-1500:].decode(errors="replace")
    served = _served(r.stderr)
    sha = hashlib.sha256(open(work / "ref.fa.bwttables", "rb").read()).hexdigest()
    out = {}
    for d, reads, gold in ((0, "reads.fq", "expected.sam"), (1, "reads_d1.fq", "expected_d1.sam")):
        r = _run([exe, "-d", str(d), "ref.fa", reads], work, env_extra)
        assert r.returncode == 0, r.stderr[-1500:].decode(errors="replace")
        c = _served(r.stderr)
        assert c[3] > 0, ("no approximate iterator was served by the drop-in", c)
        out[d] = (r.stdout, open(os.path.join(GOLD, gold), "rb").read())
    return served, sha, out


def test_bwt_readmapper_linked_against_the_drop_in(engine, tmp_path):
    """tools/readmappers/bwt_readmapper/bwt_readmapper.c (unchanged) + -lstralg_b200: the index file and the
    SAM output are those of the stock tool (tests/golden/readmapper, written by the reference build)."""
    import json
    meta = json.load(open(os.path.join(GOLD, "meta.json")))
    served, sha, out = _readmapper(_need("bwt_readmapper"), tmp_path)
    assert served[0] > 0 and served[1] > 0, served
    assert sha == meta["bwttables_sha256"]
    for d, (got, exp) in out.items():
        assert got == exp, f"-d {d}: SAM output differs from the stock tool's"


def test_stock_bwt_readmapper_with_ld_preload(engine, tmp_path):
    """INTEGRATION.md's second route: the STOCK tool (linked against the stock libstralg) with
    LD_PRELOAD=libstralg_b200.so -- the preloaded definitions win, the output does not change."""
    import json
    meta = json.load(open(os.path.join(GOLD, "meta.json")))
    shim = os.path.join(ROOT, "stralg_b200", "lib", "libstralg_b200.so")
    served, sha, out = _readmapper(_need("bwt_readmapper_stock"), tmp_path, {"LD_PRELOAD": shim})
    assert served[0] > 0 and served[1] > 0, served
    assert sha == meta["bwttables_sha256"]
    for d, (got, exp) in out.items():
        assert got == exp, f"-d {d}: SAM output differs from the stock tool's"
