"""The set read-back of the C++ host mirror (ct_mapreduce_b200/host/ctmr_storage.hpp): StoreBatch into a MockRemoteCache,
then RebuildRemoteCache from the device into a fresh mock -- identical serials:: sets and expiry times -- and
GetIssuerAndDatesFromDevice / KnownFromDevice answering what the cache holds (tests/cpp/sets_tests.cpp)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import NOW_NS, ROOT


@pytest.fixture(scope="module")
def sets_bin(tmp_path_factory):
    from ct_mapreduce_b200 import build
    build.build()
    out = tmp_path_factory.mktemp("setsbin") / "sets_tests"
    libdir = os.path.join(ROOT, "ct_mapreduce_b200")
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-o", str(out), os.path.join(ROOT, "tests", "cpp", "sets_tests.cpp"),
                    "-L" + libdir, "-lctmr", "-Wl,-rpath," + libdir], check=True)
    return str(out)


def test_sets_tests_compiles(sets_bin):
    r = subprocess.run([sets_bin], capture_output=True, text=True)
    assert r.returncode == 64 and "usage" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["per_entry", "pipelined", "group_of_three_shards"])
def test_rebuild_remote_cache_from_the_device(sets_bin, ora, tmp_path, mode):
    n = 6000
    cfg = ora.synth_cfg(n, len_mode=1, len_lo=512, len_hi=2048, dup_mode=1)
    blob, offs, idx = ora.synth_corpus(cfg, 0, n)
    iblob, ioffs = ora.synth_issuers(cfg)
    for name, arr in (("blob", blob), ("offsets", offs), ("issuer_blob", iblob), ("issuer_offsets", ioffs), ("issuer_idx", idx),
                      ("now_ns", np.array([NOW_NS], np.int64))):
        np.ascontiguousarray(arr).tofile(tmp_path / f"{name}.bin")
    extra = {"per_entry": ["plain", "1"], "pipelined": ["pipelined", "1"], "group_of_three_shards": ["plain", "3"]}[mode]
    r = subprocess.run([sets_bin, "gpu", str(tmp_path), "3"] + extra, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert "sets cpp ok" in r.stdout
