"""The launch schedule of the MSDN step against tests/golden/msdn_schedule.json.

tests/golden/make_schedule_golden.py records one eager step per configuration in a subprocess: every launch with its
arguments named symbolically, its stream and the set of launches that happen before it (stream order plus event waits).
The four-stream phase-1 step must issue the same multiset of launches, each on the same stream (up to renumbering) at the
same priority, under exactly the same happens-before relation; the sequential steps (`overlap=False`, phase 2,
inference, TF32) must issue the same launch list in the same order.  Independently of the golden, no two launches that
may run concurrently may share a scratch workspace (`ctx.workspace` key and `ctx.ws_tag`).
"""
import json
import os
import subprocess
import sys
import tempfile
from collections import Counter

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "msdn_schedule.json")
GENERATOR = os.path.join(ROOT, "tests", "golden", "make_schedule_golden.py")


@pytest.fixture(scope="module")
def golden():
    with open(GOLDEN) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def recorded():
    env = {k: v for k, v in os.environ.items() if not k.startswith("A3D_")}
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "schedule.json")
        r = subprocess.run([sys.executable, GENERATOR, "--out", out], env=env, capture_output=True, text=True,
                           timeout=1500)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        with open(out) as f:
            return json.load(f)


def keys(cfg):
    """Each launch as (method, arguments, workspaces, occurrence): the same call twice in a step stays two launches."""
    seen, out = Counter(), []
    for ln in cfg["launches"]:
        k = json.dumps([ln["m"], ln["args"], ln["ws"]], sort_keys=True)
        out.append((k, seen[k]))
        seen[k] += 1
    return out


def before(ln):
    mask = int(ln["hb"], 16)
    return [j for j in range(mask.bit_length()) if mask >> j & 1]


def happens_before(cfg):
    ks = keys(cfg)
    return {(ks[j], ks[i]) for i, ln in enumerate(cfg["launches"]) for j in before(ln)}


def describe(k):
    return f"{json.loads(k[0])[0]} #{k[1]}: {k[0][:300]}"


def test_configurations_match_golden(golden, recorded):
    assert sorted(recorded) == sorted(golden)


@pytest.mark.parametrize("name", sorted(json.load(open(GOLDEN))))
def test_schedule_matches_golden(golden, recorded, name):
    old, new = golden[name], recorded[name]
    assert new["kind"] == old["kind"]
    ko, kn = keys(old), keys(new)
    if old["kind"] == "sequential":
        lo = [(k, old["lanes"][ln["lane"]]) for k, ln in zip(ko, old["launches"])]
        ln_ = [(k, new["lanes"][ln["lane"]]) for k, ln in zip(kn, new["launches"])]
        for i, (a, b) in enumerate(zip(lo, ln_)):
            assert a == b, f"launch {i}: expected {describe(a[0])}, got {describe(b[0])}"
        assert len(lo) == len(ln_)
        assert [ln["lane"] for ln in old["launches"]] == [ln["lane"] for ln in new["launches"]]
        assert old["lanes"] == new["lanes"]
        return
    missing, extra = set(ko) - set(kn), set(kn) - set(ko)
    assert not missing and not extra, ("missing: " + "; ".join(describe(k) for k in sorted(missing)) +
                                       " | new: " + "; ".join(describe(k) for k in sorted(extra)))
    # the same stream for each launch, up to renumbering, at the same priority
    lane_old = {k: ln["lane"] for k, ln in zip(ko, old["launches"])}
    lane_new = {k: ln["lane"] for k, ln in zip(kn, new["launches"])}
    mapping = {}
    for k in ko:
        assert mapping.setdefault(lane_old[k], lane_new[k]) == lane_new[k], f"{describe(k)} changed stream"
    assert len(set(mapping.values())) == len(mapping) == len(old["lanes"]) == len(new["lanes"])
    for a, b in mapping.items():
        assert old["lanes"][a] == new["lanes"][b], f"stream {a}: priority {old['lanes'][a]} -> {new['lanes'][b]}"
    hb_old, hb_new = happens_before(old), happens_before(new)
    lost = sorted(hb_old - hb_new)
    added = sorted(hb_new - hb_old)
    assert not lost, "orderings lost: " + "; ".join(f"{describe(a)} -> {describe(b)}" for a, b in lost[:10])
    assert not added, "orderings added: " + "; ".join(f"{describe(a)} -> {describe(b)}" for a, b in added[:10])


@pytest.mark.parametrize("source", ["golden", "recorded"])
def test_concurrent_launches_use_separate_workspaces(golden, recorded, source):
    """The `ws_tag` convention: launches that may overlap in time never share a scratch buffer."""
    for name, cfg in (golden if source == "golden" else recorded).items():
        launches = cfg["launches"]
        ws = [{tuple(w) for w in ln["ws"]} for ln in launches]
        for i, ln in enumerate(launches):
            ordered = set(before(ln))
            for j in range(i):                       # a launch can only wait for launches enqueued before it
                shared = ws[i] & ws[j]
                assert j in ordered or not shared, (f"{name}: {launches[j]['m']} (#{j}) and {ln['m']} (#{i}) may run "
                                                     f"concurrently and share workspace {sorted(shared)}")
