"""bench.py's reference arm (the CPU restatement timed on the host) runs without a GPU and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert out.returncode == 0, out.stderr[-2000:]
  line = json.loads(out.stdout.strip().splitlines()[-1])
  assert line['impl'] == 'reference'
  for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
    assert key in line, key
  assert line['value'] > 0 and line['higher_is_better'] is True and line['vs_baseline'] is None
  assert 'workload' in line['config'] and 'model' not in line['config']
  cb = line['cpu_baseline']
  assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['value'] == line['value'] and cb['sample']
  e2e = line['e2e']
  assert e2e['value'] == line['value'] and e2e['h2d_bytes_per_step'] == 0 and e2e['d2h_bytes_per_step'] == 0


def test_product_path_refuses_to_run_without_a_gpu():
  """No CPU fallback: `bench.py` (our arm) must fail loudly on a box without CUDA rather than compute on the host."""
  import torch
  if torch.cuda.is_available():
    import pytest
    pytest.skip('this box has a GPU')
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert out.returncode != 0
  assert not any(l.startswith('{"metric"') for l in out.stdout.splitlines())


def test_parity_record_states_the_tested_tolerance():
  """The `parity` object of our arm's line: every arithmetic mode names its stated tolerance and the committed B200
  measurement it comes from; a missing profile degrades to nulls instead of breaking the bench line."""
  sys.path.insert(0, ROOT)
  import bench
  for precision, mode, td_tol in ((0, 'fp32', 2e-5), (1, 'tf32', 1e-2), (2, 'bf16', 2e-2)):
    rec = bench.parity_record(precision)
    assert rec['mode'] == mode and rec['tol']['td'] == td_tol
    assert 0 <= rec['max_rel_err_td'] <= td_tol and rec['max_rel_err_priority'] <= rec['tol']['priority']
    assert rec['shape'] == {'B': 256, 'A': 18, 'updates': 3} and rec['source'].startswith(f'profiles/parity_c2_{mode}.json')
    json.dumps(rec)
  old_root, bench.ROOT = bench.ROOT, os.path.join(ROOT, 'does-not-exist')
  try:
    rec = bench.parity_record(2)
  finally:
    bench.ROOT = old_root
  assert rec['mode'] == 'bf16' and rec['tol'] is None and rec['max_rel_err_td'] is None


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path):
  """`--dump-outputs` stores float32 / float64 only (integers exactly, as float64) and refuses a dump over its budget."""
  import numpy as np
  sys.path.insert(0, ROOT)
  import bench
  idx = np.array([0, 3, (1 << 40) + 7], np.int64)
  bench.dump_outputs(str(tmp_path / 'd'), {'idx': idx, 'td': np.arange(4, dtype=np.float32), 'w': np.ones(2, np.float64)})
  got = {p.stem: np.load(p) for p in (tmp_path / 'd').glob('*.npy')}
  assert got['idx'].dtype == np.float64 and np.array_equal(got['idx'].astype(np.int64), idx)
  assert got['td'].dtype == np.float32 and got['w'].dtype == np.float32
  with pytest.raises(ValueError):
    bench.dump_outputs(str(tmp_path / 'big'), {'x': np.zeros(bench.DUMP_BUDGET // 4 + 1, np.float32)})
  assert not (tmp_path / 'big').exists()
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dump-outputs', str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert out.returncode != 0 and '--dump-outputs' in out.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_update(tmp_path):
  """Our arm, small table: `--steps` is the number of timed updates (the dumped update count is warm-up + steps), and
  the same arguments give the same inputs, so two runs sample the same items and compute the same update."""
  import numpy as np
  steps, warmup = 4, 3
  runs = []
  for i in range(2):
    d = tmp_path / f'run{i}'
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', str(warmup),
                          '--items', '8192', '--no-cpu-baseline', '--dump-outputs', str(d)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['steps'] == steps and line['e2e']['steps'] == steps
    files = sorted(d.glob('*.npy'))
    assert sum(f.stat().st_size for f in files) <= 64_000_000
    runs.append({f.stem: np.load(f) for f in files})
  a, b = runs
  assert a.keys() == b.keys() and {'loss', 'td_error', 'priority', 'online_params', 'sample_index'} <= a.keys()
  assert all(v.dtype in (np.float32, np.float64) for v in a.values())
  assert a['num_steps'].tolist() == [warmup + steps]
  assert a['td_error'].shape == a['priority'].shape == a['sample_index'].shape == (256,)
  np.testing.assert_array_equal(a['sample_index'], b['sample_index'])
  for k in a:
    np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6 * float(np.abs(a[k]).max()), err_msg=k)
