"""bench.py at a small scale: `--steps` sets the number of timed steps of every leg, and `--dump-outputs` writes
the last timed step's results as float64 arrays; a seeded subset of the dumped sites is re-scored by the oracle
on the same seeded synthetic genome."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle
from conftest import ROOT

pytestmark = pytest.mark.gpu

SCALE = 0.01
SITE_FIELDS = {"genome_sites": ("motif", "chrom", "start", "score", "strand"),
               "configs1_sites": ("motif", "region", "start", "score", "strand")}


def rescore(pwm, window, strand):
    """The oracle's score of the one window of `window` on `strand` (1 forward, 2 reverse)."""
    _, _, _, score, strd = oracle.scan_arrays([pwm.tolist()], [-1e300], [window], 3)
    return score[list(strd).index(strand)]


def test_bench_steps_and_dump_outputs(tmp_path):
    out = tmp_path / "dump"
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                           "--no-cpu", "--scale", str(SCALE), "--dump-outputs", str(out)],
                          cwd=tmp_path, env=env, capture_output=True, text=True, timeout=1200)
    assert proc.returncode == 0, proc.stderr[-4000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2 and line["configs1"]["e2e"]["steps"] == 2

    names = ["genome_counts", "configs1_counts"] + [f"{p}_{f}" for p, fields in SITE_FIELDS.items() for f in fields]
    files = sorted(os.listdir(out))
    assert files == sorted(n + ".npy" for n in names)
    assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
    a = {f[:-4]: np.load(out / f) for f in files}
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["genome_counts"].shape == (bench.N_MOTIFS,) and a["genome_counts"].sum() == line["sites_per_step"] > 0
    assert a["configs1_counts"].shape == (bench.N_MOTIFS,)
    assert a["configs1_counts"].sum() == line["configs1"]["sites_per_step_rank0"] > 0

    pwms = bench.motif_workload()
    pg = bench.make_genome(0, SCALE)
    c1_chrom, c1_starts = bench.configs1_regions(pg, 0)
    rng = np.random.default_rng(7)
    for prefix, counts in (("genome_sites", a["genome_counts"]), ("configs1_sites", a["configs1_counts"])):
        motif, where, start, score, strand = (a[f"{prefix}_{f}"] for f in SITE_FIELDS[prefix])
        n = min(bench.DUMP_SITES, int(counts.sum()))
        assert all(v.shape == (n,) for v in (motif, where, start, score, strand))
        # a sample in site order (motif, sequence, start), no motif sampled more often than it has sites
        assert np.array_equal(np.lexsort((start, where, motif)), np.arange(n))
        assert np.all(np.bincount(motif.astype(np.int64), minlength=bench.N_MOTIFS) <= counts)
        assert set(np.unique(strand).tolist()) <= {1.0, 2.0}
        for i in rng.choice(n, size=min(n, 200), replace=False):
            pwm = pwms[int(motif[i])]
            if prefix == "genome_sites":
                chrom, a0 = pg.chroms[int(where[i])], int(start[i])
            else:
                chrom, a0 = c1_chrom, int(c1_starts[int(where[i])]) + int(start[i])
            window = pg.decode_bytes(chrom, a0, a0 + pwm.shape[1]).decode("ascii")
            assert rescore(pwm, window, int(strand[i])) == score[i], (prefix, i)
