import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "urmap_b200", "bin", "urmap_b200")

# What the unmodified reference binary writes for the seeded inputs of the tests that compare with it: digests of its
# UFI, SAM and -tabbedout files and the option names of its "not used" warnings (tests/golden/README.md says where they
# come from).  URMB_GOLDEN_RECORD=1 records the values a run observes instead of checking them and rewrites the file.
EXPECTED_PATH = os.path.join(GOLDEN, "reference_outputs.json")
EXPECTED = json.load(open(EXPECTED_PATH))
RECORD = {} if os.environ.get("URMB_GOLDEN_RECORD") else None


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_sessionfinish(session, exitstatus):
    if RECORD:
        merged = dict(EXPECTED, **RECORD)
        with open(EXPECTED_PATH, "w") as f:
            json.dump(dict(sorted(merged.items())), f, indent=1)
            f.write("\n")


def expect(key, value):
    """`value` must equal the stored reference output `key` of tests/golden/reference_outputs.json."""
    if RECORD is not None:
        RECORD[key] = value
        return
    assert key in EXPECTED, f"no stored reference output {key!r}"
    assert value == EXPECTED[key], (key, value, EXPECTED[key])


def file_digest(path):
    """sha256 and size of a file."""
    data = open(path, "rb").read()
    return {"sha256": hashlib.sha256(data).hexdigest(), "size": len(data)}


def sam_digest(path_or_bytes):
    """sha256 of a SAM file without its @PG line (it carries the command line), records in file order."""
    data = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, "rb").read()
    lines = [l for l in data.split(b"\n") if l and not l.startswith(b"@PG")]
    return {"sha256": hashlib.sha256(b"\n".join(lines)).hexdigest(), "records": sum(1 for l in lines if not l.startswith(b"@"))}


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle_py as O
    O.build(ref=True)
    return O


@pytest.fixture(scope="session")
def golden_dir(built_lib):
    import __graft_entry__
    __graft_entry__.golden_ufi()
    return GOLDEN


@pytest.fixture(scope="session")
def golden_oix(oracle, golden_dir):
    ix = oracle.Index(os.path.join(GOLDEN, "ref.ufi"))
    yield ix
    ix.close()


@pytest.fixture(scope="session")
def built_lib():
    """liburmb.so built in-tree (nvcc cross-compiles without a GPU)."""
    from urmap_b200 import build as B
    B.build_engine()
    from urmap_b200 import engine
    return engine


def make_ufi(key, fa, out, extra=()):
    """UFI file of `fa` from the drop-in's host builder (-make_ufi): byte-identical to the reference's file for the same
    genome and options, whose digest is the stored reference output `ufi/<key>`.  Where the unmodified reference binary
    has been built (oracle/_ref/urmap), it writes the same file."""
    r = subprocess.run([CLI, "-make_ufi", fa, "-output", out, "-quiet"] + list(extra), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    expect("ufi/" + key, file_digest(out))
    from oracle import oracle_py as O
    if os.path.exists(O.REF_BIN):
        ref = out + ".ref"
        O.run_reference(["-make_ufi", fa, "-output", ref] + list(extra))
        assert open(ref, "rb").read() == open(out, "rb").read(), extra
        os.unlink(ref)
    return out


def have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False
