"""Pins the oracle (and the engine's math / RNG headers) to the reference's own
known-answer tests and headers.

* reference KATs: tests/rand.cpp:131-141 (bits32 / sampleI32 upper limit),
  tests/math.cpp:23-48 (quaternion values, 1e-4);
* header equivalence: oracle/kat_probe.cpp compiled against madrona_b200/device/madrona
  must print the bits it printed compiled against the reference headers
  (tests/golden/kat_probe_ref.txt.gz, 2500+ values: threefry streams,
  quaternion / matrix / AABB algebra);
* the numpy restatement (oracle/restate.py) must reproduce the same streams and
  the initial states the reference CPU backend produced in the golden traces.
"""
import struct

import numpy as np
import pytest

from oracle import restate
from trace_utils import build_engine_probe, reference_probe_output


def _ref():
    return reference_probe_output("kat_probe_ref").splitlines()


@pytest.fixture(scope="module")
def mine(tmp_path_factory):
    return build_engine_probe("kat_probe_mine", tmp_path_factory.mktemp("probe")).splitlines()


def _f(hexbits):
    return struct.unpack("<f", struct.pack("<I", int(hexbits, 16)))[0]


def test_restatement_known_answers():
    k = (0xFFFFFFFF, 0)
    assert restate.bits32(k) == 0xFFFFFFFF
    assert restate.sample_i32(k, 0, 64) == 63
    assert restate.sample_i32_biased(k, 0, 64) == 63


def test_reference_headers_known_answers():
    lines = dict()
    for ln in _ref():
        tag, *vals = ln.split()
        lines.setdefault(tag, []).append(vals)
    assert lines["kat_bits32"][0][0] == "ffffffff"
    assert lines["kat_sampleI32"][0][0] == "63"
    assert lines["kat_sampleI32Biased"][0][0] == "63"
    want = {"kat_q1": (1, 0, 0, 0), "kat_q2": (0.9238795, 0, 0.3826834, 0),
            "kat_q3": (0.9238795, 0.3826834, 0, 0),
            "kat_m1": (0.853553, 0.353553, 0.353553, -0.146447)}
    for tag, q in want.items():
        got = [_f(v[0]) for v in lines[tag]]
        assert np.allclose(got, q, atol=1e-4), (tag, got)


def test_engine_headers_match_reference_headers_bit_for_bit(mine):
    ref = _ref()
    assert len(ref) > 2000
    assert ref == mine


def test_restatement_matches_reference_streams():
    lines = _ref()
    it = iter(lines)
    checked = 0
    for seed in range(4):
        key = restate.init_key(seed * 7919 + 1, seed)
        ln = next(l for l in it if l.startswith("key "))
        assert ln.split()[1:] == [f"{key[0]:08x}", f"{key[1]:08x}"]
        for i in range(4):
            s = restate.split_i(key, i, i * 3)
            ln = next(l for l in it if l.startswith("split "))
            assert ln.split()[1:] == [f"{s[0]:08x}", f"{s[1]:08x}"]
            ln = next(l for l in it if l.startswith("i32 "))
            assert [int(v) for v in ln.split()[1:]] == [
                restate.sample_i32(s, -20, 2), restate.sample_i32(s, 0, 1000003),
                restate.sample_i32_biased(s, 3, 77)]
            ln = next(l for l in it if l.startswith("uniform "))
            assert _f(ln.split()[1]) == float(restate.sample_uniform(s))
            checked += 1
    assert checked == 16


def test_restatement_reproduces_reference_backend_initial_state():
    # cartpole world w is seeded RNG(seed + w); its first four uniforms give the
    # initial state the reference CPU backend exported at step 0 of the golden
    from trace_utils import load_golden
    W, steps, ins, outs = load_golden("cartpole_w64_s300")
    for w in (0, 1, 17, 63):
        rng = restate.RNG(0 + w)
        want = [np.float32(rng.sample_uniform() * np.float32(0.1) - np.float32(0.05)) for _ in range(4)]
        assert np.array_equal(np.array(want, dtype=np.float32), outs["state"][0, w])


def test_sort_restatement_semantics():
    keys = np.array([2, 0, -1, 1, 0, 2, -1, 5], dtype=np.int32)
    perm, new_n, off, cnt = restate.sort_archetype(keys, num_worlds=6)
    assert new_n == 6
    assert perm.tolist() == [1, 4, 3, 0, 5, 7]          # stable inside each world
    assert off.tolist() == [0, 2, 3, 6, 6, 5]            # empty worlds -> offset = numRows
    assert cnt.tolist() == [2, 1, 2, 0, 0, 1]
    assert restate.world_sort_passes(255) == 1 and restate.world_sort_passes(256) == 2
    assert restate.world_sort_passes(8192) == 2 and restate.world_sort_passes(65536) == 3


def test_sort_restatement_matches_reference_compaction_in_golden():
    # the Item table of the gridworld golden is the reference CPU backend's
    # compaction output: per-world blocks in world order, creation order inside
    from trace_utils import load_golden
    W, steps, ins, outs = load_golden("gridworld_w32_s150")
    for t in (0, 40, 97, 150):
        counts = outs["item_count"][t, :, 0]
        world_of_row = np.repeat(np.arange(W), counts)
        perm, new_n, off, cnt = restate.sort_archetype(world_of_row.astype(np.int32), W)
        assert new_n == counts.sum() and perm.tolist() == list(range(new_n))
        assert np.array_equal(cnt, counts)
        assert np.array_equal(off[counts > 0], (np.cumsum(counts) - counts)[counts > 0])
