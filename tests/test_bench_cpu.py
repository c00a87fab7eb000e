"""bench.py contract on CPU: the reference arm (the reference's own modules from oracle/_ref/py when `make -C oracle refpy` has run,
else the CPU oracle port) prints ONE JSON line with the agreed keys; the algorithmic byte model matches SURVEY.md §8(d)."""

import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--impl', 'reference', '--tiny', '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['higher_is_better'] is True and d['n_gpus'] == 1
    for k in ('metric', 'value', 'unit', 'steps', 'warmup', 'ms_per_step', 'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    have_ref = os.path.isdir(os.path.join(REPO, 'oracle', '_ref', 'py', 'core'))
    assert d['cpu_baseline']['kind'] == ('reference' if have_ref else 'port'), d['cpu_baseline']
    assert d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['value'] > 0 and 'workload' in d['config']


def test_dump_outputs_budget_and_sample(tmp_path):
    """--dump-outputs: every array in float64; one above its share of the 64 MB budget becomes a fixed seeded sample plus its indices."""
    import numpy as np
    import torch
    sys.path.insert(0, REPO)
    import bench
    arrays = {'loss': torch.tensor(1.5), 'tokens': torch.arange(7, dtype=torch.int32), 'logits': torch.arange(6_000_000, dtype=torch.float32).reshape(1000, 6000)}
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['logits.npy', 'logits_index.npy', 'loss.npy', 'tokens.npy']
    got = {f: np.load(tmp_path / 'a' / f) for f in files}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= bench.DUMP_BYTES
    assert got['loss.npy'] == 1.5 and np.array_equal(got['tokens.npy'], np.arange(7))
    idx = got['logits_index.npy']
    assert 0 < len(idx) < 6_000_000 and np.all(np.diff(idx) > 0) and np.array_equal(got['logits.npy'], idx)
    for f in files:
        assert np.array_equal(got[f], np.load(tmp_path / 'b' / f)), f


def test_algorithmic_byte_model():
    """SURVEY.md §8(d): bytes(L) = W + kv (L + 1) with W = 1,361,504,256 and kv = 147,456 for the ArAE preset; 45.5 TB for the 16k request."""
    sys.path.insert(0, REPO)
    import bench
    W, kv = 1361504256, 147456

    class Eng:                                       # the two engine introspection calls bench.py uses
        weight_bytes_per_token = staticmethod(lambda: W)
        kv_bytes_per_row = staticmethod(lambda: kv)
    assert bench.algorithmic_decode_bytes(Eng, 2050, 2) == W + kv * 2051            # one forward pass at L = 2050
    total = bench.algorithmic_decode_bytes(Eng, 2050, 16000)
    T = 15999
    assert total == T * (W + kv) + kv * (T * 2050 + T * (T - 1) // 2)
    assert 45.4e12 < total < 45.6e12
