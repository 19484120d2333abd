"""build.py compiles a split source once per translation unit k = 0..n-1, n derived from the SMARL_TU_IS(k) guards.
A gap in those indices would compile an empty object, and SMARL_TU_IS is defined once, in common.cuh."""
import os
import re

from safe_multiagent_rl_b200 import build

CSRC = build.CSRC


def test_tu_count_matches_the_guards():
    sources = build.sources()
    assert any(build.tu_count(f) > 1 for f in sources)
    for f in sources:
        ks = {int(k) for k in re.findall(r"\bSMARL_TU_IS\((\d+)\)", open(os.path.join(CSRC, f)).read())}
        n = build.tu_count(f)
        assert n == len(ks) and ks == set(range(n)) if ks else n == 1, (f, n, sorted(ks))


def test_no_source_defines_the_tu_macro():
    define = re.compile(r"^\s*#\s*define\s+SMARL_TU_IS\b", re.M)
    offenders = [f for f in sorted(os.listdir(CSRC)) if f.endswith(".cu") and define.search(open(os.path.join(CSRC, f)).read())]
    assert not offenders, offenders
