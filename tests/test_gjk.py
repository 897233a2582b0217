"""GJK closest point (sphere - hull contacts): pins madrona_b200/device/madrona/gjk.hpp
to the reference's src/physics/gjk.hpp + geo::hullClosestPointToOriginGJK.

* oracle/gjk_probe.cpp compiled against the engine's header must print the bits
  it printed compiled against the reference (private header + libmadrona_ref.a;
  tests/golden holds the digest of that output and its known answers):
  900 sub-simplex solves, 1200 hull distance queries (a third of
  them with the origin inside the hull);
* the assertions of the reference's own tests (tests/gjk.cpp:18-47) are applied
  to both outputs.
"""
import hashlib
import os
import struct

import pytest

from trace_utils import build_engine_probe, reference_probe_output

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "gjk_probe.sha256")


@pytest.fixture(scope="module")
def mine(tmp_path_factory):
    return build_engine_probe("gjk_probe_mine", tmp_path_factory.mktemp("probe"))


def _f(hexbits):
    return struct.unpack("<f", struct.pack("<I", int(hexbits, 16)))[0]


def _tagged(text):
    out = {}
    for ln in text.splitlines():
        tag, val = ln.split()
        out.setdefault(tag, []).append(_f(val))
    return out


def test_engine_header_matches_reference_bit_for_bit(mine):
    # the digest of the reference build's output (tests/golden/make_golden.py)
    assert len(mine.splitlines()) > 10000
    assert hashlib.sha256(mine.encode()).hexdigest() == open(GOLDEN).read().strip()
    # its known answers, stored whole
    ref_kat = reference_probe_output("gjk_probe_ref")
    assert ref_kat.splitlines() == [ln for ln in mine.splitlines() if ln.startswith("kat_")]


@pytest.mark.parametrize("binary", ["reference", "engine"], ids=["reference", "engine"])
def test_reference_gjk_known_answers(binary, mine):
    vals = _tagged(reference_probe_output("gjk_probe_ref") if binary == "reference" else mine)
    # tests/gjk.cpp:18-32 Solve4SimplexDuplicatePoint
    assert vals["kat_dup_diff"][0] <= 1e-5
    # tests/gjk.cpp:34-47 Solve4SimplexAroundOrigin
    vx, vy, vz, len2 = vals["kat_origin_s4"][:4]
    assert abs(vx) < 1e-5 and abs(vy) < 1e-5 and abs(vz) < 1e-5
    assert len2 < 1e-5


def test_engine_header_against_committed_digest(mine):
    assert hashlib.sha256(mine.encode()).hexdigest() == open(GOLDEN).read().strip()
