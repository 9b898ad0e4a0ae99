"""bench.py --dump-outputs: the arrays it writes are what the timed path returned in its last step -- checked against the
oracle's sequential run over the same seeded corpus -- in float32 / float64 and within 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import NOW_NS, ROOT

pytestmark = pytest.mark.gpu


@pytest.mark.timeout(900)
def test_dump_outputs_are_the_last_timed_step(ora, tmp_path):
    n, steps = 20000, 3
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                        "--entries", str(n), "--no-e2e", "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=850)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["config"]["entries_per_gpu_per_step"] == n

    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(got) == {"entry_index", "status", "exp_hour", "was_unknown", "first_issuer_hour", "sha256", "issuer_counts",
                        "status_counters"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 << 20
    assert np.array_equal(got["entry_index"], np.arange(n))   # fewer entries than the sample size: all of them

    # the default single-GPU workload (cfg2): seeded corpus, no CN filter, expired certificates kept
    cfg = ora.synth_cfg(n, seed=20260922, len_mode=0, len_lo=1436, len_hi=1564, dup_mode=0)
    blob, offs, idx = ora.synth_corpus(cfg, 0, n)
    iblob, ioffs = ora.synth_issuers(cfg)
    odb = ora.DB(b"", True)
    want = odb.process(blob, offs, iblob, ioffs, idx, NOW_NS)
    for f in ("status", "was_unknown", "first_issuer_hour", "sha256"):
        assert np.array_equal(got[f], getattr(want, f).astype(np.float32)), f
    ok = want.status == 0
    assert np.array_equal(got["exp_hour"][ok], want.exp_hour[ok].astype(np.float64))
    assert np.array_equal(got["status_counters"], odb.filter_counters().astype(np.float64))
    assert sorted(v for v in got["issuer_counts"].tolist() if v) == sorted(v for v in odb.issuer_counts().values() if v)
