"""CPU: the environment variables the native library reads are a short, deliberate list.

Each one is either a documented setting or a hook the GPU tests use to pin a code path.  A switch added for a one-off
experiment has to be added here too, so it cannot stay in the library without a decision.  CUVS_B200_LIB and
CUVS_B200_PROFILE are read by Python (cuvs_b200/_capi.py, bench.py), not by the library."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LIBRARY_ENV = {
    "CUVS_B200_PQ_PATH",               # IVF-PQ fine-scan path: lut | tc | stream (tests compare the paths)
    "CUVS_B200_PQ_GROUP",              # queries per work item of the code-streaming scan (tests cover each group)
    "CUVS_B200_PQ_DECODED_BUDGET_MB",  # memory budget of the decoded-row cache (DESIGN.md section 5)
    "CUVS_B200_COARSE_FUSED",          # "0" = dense coarse search (a test compares it with the fused one)
}


def _sources():
    for f in sorted(glob.glob(os.path.join(ROOT, "cuvs_b200", "csrc", "*"))):
        if os.path.isfile(f):
            yield f, open(f, errors="ignore").read()


def _library_env_names():
    # every string literal that is exactly a CUVS_B200_* name: what getenv / env_int are called with
    return {m for _, txt in _sources() for m in re.findall(r'"(CUVS_B200_\w+)"', txt)}


def test_library_reads_only_the_listed_environment_variables():
    assert _library_env_names() == LIBRARY_ENV


def test_getenv_takes_a_literal_name_outside_the_shared_helper():
    # a name built at run time would escape the scan above; common.hpp's env_int is the one helper that forwards its argument
    bad = []
    for f, txt in _sources():
        for arg in re.findall(r"\bgetenv\(\s*([^)]*)\)", txt):
            if not arg.startswith('"') and not (os.path.basename(f) == "common.hpp" and arg == "name"):
                bad.append(f"{os.path.basename(f)}: getenv({arg})")
    assert not bad, bad


def test_every_variable_the_tests_set_is_read_by_the_library():
    me = os.path.abspath(__file__)
    set_by_tests = set()
    for f in glob.glob(os.path.join(ROOT, "tests", "**", "*.py"), recursive=True):
        if os.path.abspath(f) == me:
            continue
        txt = open(f, errors="ignore").read()
        set_by_tests |= set(re.findall(r"""(?:environ\[|setenv\(|putenv\()\s*["'](CUVS_B200_\w+)["']""", txt))
        set_by_tests |= set(re.findall(r"\b(CUVS_B200_\w+)\s*=(?!=)", txt))  # env=dict(os.environ, NAME=...)
    assert set_by_tests, "no test sets a CUVS_B200_* variable: the scan above is broken"
    assert set_by_tests <= LIBRARY_ENV, sorted(set_by_tests - LIBRARY_ENV)
