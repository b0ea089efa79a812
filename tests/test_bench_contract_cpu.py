"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) prints the one JSON
line the driver parses, with the keys the measurement contract names, and the GPU arm's source never names oracle/."""
import ast
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1]
    d = json.loads(line)
    assert d['impl'] == 'reference' and d['unit'] == 'views/s' and d['higher_is_better'] is True and d['n_gpus'] == 1
    assert d['value'] > 0 and abs(d['value'] - 1e3 / d['ms_per_step']) < 1e-6 * d['value'] + 1e-9
    assert d['steps'] == 1 and d['scaling'] == 'weak' and d['vs_baseline'] is None and d['data'] == 'synthetic'
    assert 'workload' in d['config'] and '96+96' in d['config']['workload']
    cb = d['cpu_baseline']
    # kind "reference" = the unmodified reference imported from baseline/_ref (baseline/install_ref.sh), "port" = the oracle
    have_ref = os.path.isdir(os.path.join(ROOT, 'baseline', '_ref', '_train', 'eg3dc', 'src', 'training'))
    assert cb['kind'] == ('reference' if have_ref else 'port') and cb['cores'] >= 1 and cb['value'] == d['value'] and cb['sample']
    # same `config` as the GPU arm prints (the driver compares them); the per-step sample is described in cpu_baseline
    sys.path.insert(0, ROOT)
    import bench
    assert d['config'] == bench.workload_config(1, 'tc_3xbf16', 'fp32') and d['warmup'] == 1
    assert d['e2e'] == {'value': d['value'], 'unit': 'views/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['gpu_launches'] == 0


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv, capture_output=True, text=True, timeout=60, cwd=tmp_path)
    assert r.returncode == 2 and 'error:' in r.stderr and not os.listdir(tmp_path)


def test_gpu_arm_of_bench_does_not_touch_the_oracle():
    tree = ast.parse(open(os.path.join(ROOT, 'bench.py')).read())
    fns = {n.name: n for n in tree.body if isinstance(n, ast.FunctionDef)}
    for name in ('run_ours', 'run_e2e'):
        src_names = {n.id for n in ast.walk(fns[name]) if isinstance(n, ast.Name)}
        imports = [a.name for n in ast.walk(fns[name]) if isinstance(n, (ast.Import, ast.ImportFrom))
                   for a in n.names] + [n.module or '' for n in ast.walk(fns[name]) if isinstance(n, ast.ImportFrom)]
        calls_cpu_leg = 'cpu_reference_time' in src_names
        assert 'orc' not in src_names and not any('oracle' in i for i in imports), name
        if name == 'run_e2e':
            assert not calls_cpu_leg
