"""The environment variables the library reads are exactly the documented ones (DESIGN §4.1).

None of them changes what a training step computes: they find faults, drive the profiler, select the layer API's
precision, load a build variant, or belong to the conv-kernel harness.  A new getenv() in the library is added here
and to DESIGN §4.1 together."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "unet.cu_b200")

# read by the library (unet.cu_b200/csrc, unet.cu_b200/host)
LIBRARY = {
    "UB_DEBUG_SYNC",       # synchronise after every op of an eager step and name the failing one
    "UB_DEBUG_BUCKETS",    # print the gradient buckets
    "UB_NO_PDL",           # launch without programmatic dependent launch: a fully serialised step
    "UB_PROFILE_DUMP",     # ub_trainer_profile: per-op times to a file
    "UB_PROFILE_REPLAY",   # ub_trainer_profile: repetitions
    "UB_LAYER_PRECISION",  # layer API: exact fp32 operators (include/unet_b200.h)
}
# build plumbing and the conv-kernel harness (tools/igemm_test.cu)
OTHER = {"UB_LIB_VARIANT", "UB_TRACE", "UB_TRACE_MODE", "UB_TEST_STATS"}


def _sources(*dirs):
    for d in dirs:
        for dirpath, _, files in os.walk(d):
            for f in files:
                if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp", ".py")):
                    yield os.path.join(dirpath, f)


def _getenv_names(*dirs):
    names = {}
    for path in _sources(*dirs):
        with open(path, encoding="utf-8") as fh:
            for name in re.findall(r"getenv\(\s*[\"'](\w+)[\"']", fh.read()):
                names.setdefault(name, []).append(os.path.relpath(path, ROOT))
    return names


def test_library_reads_only_documented_variables():
    names = _getenv_names(os.path.join(PKG, "csrc"), os.path.join(PKG, "host"))
    unexpected = {n: p for n, p in names.items() if n not in LIBRARY}
    assert not unexpected, f"undocumented environment switches: {unexpected}"
    assert set(names) == LIBRARY, f"documented but no longer read: {sorted(LIBRARY - set(names))}"


def test_launch_header_has_no_pdl_variant_macros():
    with open(os.path.join(PKG, "csrc", "launch.cuh"), encoding="utf-8") as fh:
        src = fh.read()
    assert not re.findall(r"#\s*(?:define|ifndef|ifdef|if)\s+UB_PDL_\w*", src)


def test_design_lists_the_same_variables():
    with open(os.path.join(ROOT, "DESIGN.md"), encoding="utf-8") as fh:
        design = fh.read()
    sec = design[design.index("### 4.1"):design.index("## 5.")]
    assert set(re.findall(r"`(UB_[A-Z_]+)", sec)) == LIBRARY | OTHER
