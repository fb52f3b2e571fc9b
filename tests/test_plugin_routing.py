"""Which jobs the B200 executor plugin takes and which it leaves to the reference's CPU path (ShouldRunLocal,
db/compaction/compaction_executor.h:162): decided from the job's options by WhyLocal() in toplingdb_b200/plugin/b200_compaction_executor.cc
and reported, one line per job, when B200C_PLUGIN_TRACE is set.  The decision does not need a device, so it is checked here on the CPU,
with any CUDA device hidden from the reference (a device would also run the jobs, and reject the data of some of them):
every scenario of the GPU integration tests must be device-eligible (otherwise those tests would silently exercise the CPU path), and
option shapes outside the device rule set must be recognised -- with the reference then producing its normal result."""
import os
import subprocess
import tempfile

import pytest

import helpers as H
import scenarios as S

pytestmark = pytest.mark.skipif(not os.path.exists(H.REF_B200_BIN), reason="oracle/_ref/ref_compact_b200 not built")


def _trace(fn, **extra):
    ops, opts = fn()
    opts = dict(opts, **extra)
    with tempfile.TemporaryDirectory(prefix="b200c_route_") as d:
        with open(os.path.join(d, "ops.bin"), "wb") as f:
            f.write(ops.bytes())
        args = [H.REF_B200_BIN, os.path.join(d, "ops.bin"), os.path.join(d, "w"), "executor=b200"] + [f"{k}={v}" for k, v in opts.items()]
        r = subprocess.run(args, capture_output=True, text=True, env=dict(os.environ, B200C_PLUGIN_TRACE="1", CUDA_VISIBLE_DEVICES=""))
        assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stderr.splitlines() if ln.startswith("B200Compact: job ")]
    assert lines, "the executor factory was never asked"
    return [ln.split(": ", 2)[2] for ln in lines]


@pytest.mark.parametrize("name", sorted(S.ALL))
def test_integration_scenarios_are_device_eligible(name):
    for why in _trace(S.ALL[name]):
        assert why.startswith("device-eligible"), why


@pytest.mark.parametrize("extra", [dict(bloom_bits=10), dict(paranoid=1), dict(max_subcompactions=4), dict(checksum="crc32c", block_size=1024)])
def test_supported_option_shapes_are_device_eligible(extra):
    for why in _trace(S.ALL["cfg3_mini"], **extra):
        assert why.startswith("device-eligible"), why
    for why in _trace(lambda: S.grandparent_cuts(n=8000, seed=18)):
        assert why.startswith("device-eligible"), why


@pytest.mark.parametrize("scenario,extra,reason", [
    ("snapshots_nonbottom", dict(blob=1), "blob files"), ("snapshots", dict(ingest_behind=1), "allow_ingest_behind"),
    ("snapshots_nonbottom", dict(ribbon=1), "filter policy other than"),
    ("snapshots_nonbottom", dict(partition_filters=1, bloom_bits=10), "filter policy other than"),
    ("snapshots_nonbottom", dict(format_version=2), "format subset")])
def test_option_shapes_outside_the_rule_set_stay_on_the_cpu(scenario, extra, reason):
    whys = _trace(S.ALL[scenario], **extra)
    assert all(reason in w for w in whys), whys
