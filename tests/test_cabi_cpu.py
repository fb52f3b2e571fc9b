"""CPU-side checks of the drop-in boundary: the library builds, loads, exports every symbol include/b200c.h declares,
and refuses to run without a device (there is no CPU data path)."""
import ctypes as C
import os
import re

import pytest

import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import toplingdb_b200 as T
    L = T.load_library()
    hdr = open(os.path.join(ROOT, "include", "b200c.h")).read()
    declared = set(re.findall(r"B200C_API [^;(]*?\b(b200c_[a-z_]+)\(", hdr))
    assert len(declared) >= 16
    for name in declared:
        assert hasattr(L, name), name
    assert set(T.native.EXPORTS) == declared
    assert L.b200c_abi_version() == 8


def test_params_defaults_match_reference_defaults():
    import toplingdb_b200 as T
    p = T.native.Params()
    T.lib().b200c_params_init(C.byref(p))
    # include/rocksdb/table.h:237-564, advanced_options.h:599
    assert (p.block_size, p.block_size_deviation, p.block_restart_interval, p.index_block_restart_interval) == (4096, 10, 16, 1)
    assert (p.format_version, p.checksum, p.max_output_file_size) == (5, 4, 64 << 20)


def test_no_cpu_fallback_without_a_device():
    import torch
    import toplingdb_b200 as T
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(T.B200cError) as ei:
        T.CompactionJob()
    assert ei.value.code == T.native.ERR_NO_DEVICE
    with pytest.raises(T.B200cError):
        T.block_checksums("xxh3", [b"abc"])


def test_product_does_not_reference_the_oracle():
    bad = []
    for dp, _, fs in os.walk(os.path.join(ROOT, "toplingdb_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cc", ".h")):
                s = open(os.path.join(dp, f), errors="replace").read()
                if "liboracle" in s or "compaction_oracle" in s or "oracle/" in s:
                    bad.append(f)
    assert not bad, bad


@pytest.mark.skipif(not (os.path.exists(H.REF_BIN) and os.path.exists(H.REF_B200_BIN)), reason="oracle/_ref not built")
def test_plugin_without_a_device_lets_the_reference_run_the_job_itself(monkeypatch):
    """No CUDA device: B200CompactionExecutorFactory::ShouldRunLocal() must answer true (compaction_executor.h:162), so the
    reference's CompactionJob::Run takes RunLocal() (compaction_job.cc:645-647) -- the plugin never computes anything on
    the CPU itself.  Same files as a run without the plugin, and no remote-compaction bytes accounted.  Any CUDA device is hidden
    from the reference (the device path is tests/test_gpu_plugin_integration.py)."""
    import scenarios as S
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    ops, opts = S.ALL["cfg2_mini"](per_run=300)
    want = H.run_reference(ops, **opts)
    got = H.run_reference(ops, binary=H.REF_B200_BIN, executor="b200", **opts)
    assert got["manifest"]["executor"] == "B200Compact"
    assert got["manifest"]["remote_compact_read_bytes"] == 0
    assert (got["manifest"]["scan_count"], got["manifest"]["scan_digest"]) == (want["manifest"]["scan_count"], want["manifest"]["scan_digest"])
    assert [len(o) for o in got["outputs"]] == [len(o) for o in want["outputs"]]


def test_ctypes_mirror_has_the_layout_of_the_header(tmp_path):
    """toplingdb_b200/native.py restates the structs of include/b200c.h by hand; a C program compiled against the header prints
    sizeof / offsetof of every field the mirror names, and they must agree (a drifted mirror would hand the library garbage)."""
    import subprocess
    import toplingdb_b200 as T
    pairs = [("b200c_grandparent", T.native.Grandparent), ("b200c_params", T.native.Params), ("b200c_file_meta", T.native.FileMeta),
             ("b200c_stats", T.native.JobStats)]
    src = ['#include <stddef.h>', '#include <stdio.h>', '#include "b200c.h"', 'int main(void) {']
    for cname, cls in pairs:
        src.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            src.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    src += ["  return 0;", "}"]
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c11", "-I" + os.path.join(ROOT, "include"), str(c), "-o", str(exe)])
    want = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    hdr = open(os.path.join(ROOT, "include", "b200c.h")).read()
    for cname, cls in pairs:
        assert C.sizeof(cls) == int(want[cname]), cname
        for fname, _ in cls._fields_:
            assert getattr(cls, fname).offset == int(want[f"{cname}.{fname}"]), (cname, fname)
        # and the mirror names every field of the C struct (same count of declarators)
        body = hdr[hdr.index("typedef struct " + cname + " {"):hdr.index("} " + cname + ";")]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        decls = [d for stmt in body.split("{", 1)[1].split(";") for d in stmt.split(",") if d.strip()]
        assert len(decls) == len(cls._fields_), (cname, len(decls), len(cls._fields_))
