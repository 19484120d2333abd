"""build.py rebuilds an object only when its own source or some header changed.  A source that included another .cu
file would therefore link stale code after that file changed, so shared code lives in headers (.cuh)."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "safe_multiagent_rl_b200", "csrc")


def test_no_source_includes_a_cu_file():
    include_cu = re.compile(r'^\s*#\s*include\s*[<"][^">]*\.cu[">]', re.M)
    files = sorted(os.listdir(CSRC))
    assert any(f.endswith(".cu") for f in files)
    offenders = [f"{f}: {m.group(0).strip()}" for f in files if f.endswith((".cu", ".cuh", ".h"))
                 for m in include_cu.finditer(open(os.path.join(CSRC, f)).read())]
    assert not offenders, offenders
