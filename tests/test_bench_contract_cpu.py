"""CPU: bench.py's output contract, checked on its real main() with the GPU work replaced by stand-ins (tests/_mock_bench.py):
exactly ONE JSON line on stdout carrying the driver's keys; an optional block that raises is reported inside the line; an
optional block that stalls past --extras-budget does not take the headline with it (the line is still printed, once, and
the process exits 0)."""
import json
import os
import subprocess
import sys
from conftest import ROOT

KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
        'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline', 'train', 'configs', 'sweep'}


def run(env=None, extra=()):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', '_mock_bench.py')] + list(extra), capture_output=True, text=True,
                       env=e, timeout=120)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_one_json_line_with_the_contract_keys():
    d = run()
    assert KEYS <= set(d), KEYS - set(d)
    assert d['higher_is_better'] is True and d['scaling'] == 'weak' and d['n_gpus'] == 1
    assert {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'} <= set(d['e2e'])
    assert d['e2e']['h2d_bytes_per_step'] == 3 * 600 * 1000 * 4
    assert d['train'] == {'graph': True} and d['configs']['3_fpn'] == {'test': 1, 'train': 2} and 'extras' not in d


def test_gpu_arm_dump_outputs(tmp_path):
    """main() hands the graphed step's outputs to --dump-outputs: one float32 .npy per output; the line reports --steps."""
    import numpy as np
    d = run(extra=['--steps', '7', '--dump-outputs', str(tmp_path)])
    assert d['steps'] == 7
    assert sorted(os.listdir(str(tmp_path))) == ['learn_nms_sorted_bbox.npy', 'nms_final_score_output.npy']
    a = np.load(str(tmp_path / 'learn_nms_sorted_bbox.npy'))
    assert a.dtype == np.float32 and a.shape == (100, 80, 4)


def test_timed_runs_exactly_steps_between_its_events(monkeypatch):
    """bench.timed: `warmup` calls before the opening event, exactly `steps` calls between the two events."""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    state = {'events': 0, 'calls': [0, 0, 0]}                  # calls before / inside / after the timed window

    class Event:
        def __init__(self, **kw):
            pass

        def record(self):
            state['events'] += 1

        def elapsed_time(self, other):
            return 12.5
    monkeypatch.setattr(torch.cuda, 'Event', Event)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda *a, **k: None)

    def step():
        state['calls'][state['events']] += 1
    assert bench.timed(step, 9, 4, False) == 12.5
    assert state['calls'] == [4, 9, 0]


def test_reference_arm_times_every_requested_step(monkeypatch, tmp_path):
    """--impl reference: the CPU arm times all --steps steps (no cap), reports them, and dumps the last step's outputs."""
    import argparse
    import types
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import relnet_b200  # noqa: F401
    from relnet_b200 import pipeline, trunk
    from oracle import pipeline_np
    calls, marks, lines = [0], [], []

    def head_forward(*a, **k):
        calls[0] += 1
        return dict(rois=np.arange(10, dtype=np.int64), cls_score=np.full((3, 4), calls[0], np.float64),
                    fc_all_2_relu=np.ones((3, 4), np.float16))

    def perf_counter():
        marks.append(calls[0])
        return float(len(marks))
    monkeypatch.setattr(trunk, 'make_trunk', lambda *a, **k: (lambda im: (torch.zeros(1), torch.zeros(1), torch.zeros(1))))
    monkeypatch.setattr(pipeline, 'init_head_params', lambda *a, **k: {})
    monkeypatch.setattr(pipeline_np, 'head_forward', head_forward)
    monkeypatch.setattr(bench, 'cpu_threads', lambda: 1)
    monkeypatch.setattr(bench, 'time', types.SimpleNamespace(perf_counter=perf_counter))
    monkeypatch.setattr(bench, 'emit', lines.append)
    monkeypatch.delenv('RANK', raising=False)
    bench.run_reference(argparse.Namespace(steps=8, warmup=5, gpus=1, dump_outputs=str(tmp_path)))
    assert marks == [1, 9] and lines[0]['steps'] == 8                  # one warm-up step, then 8 inside the clock
    out = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert sorted(out) == ['cls_score', 'fc_all_2_relu', 'rois']
    assert out['rois'].dtype == np.float64 and out['fc_all_2_relu'].dtype == np.float32
    assert out['cls_score'].dtype == np.float64 and (out['cls_score'] == 9).all()      # the last timed step's outputs


def test_failing_optional_block_is_reported_not_fatal():
    d = run({'MOCK_FAIL': '1'})
    assert d['train'] == {'failed': 'boom'} and d['configs']['2_deformable_faster'] == {'images_per_sec': 700}


def test_deadline_keeps_the_headline():
    d = run({'MOCK_HANG': '1'}, ['--extras-budget', '6'])
    assert 'stopped at the 6 s deadline' in d['extras']
    assert d['value'] > 0 and d['configs']['3_fpn'] == {'test': 1}          # the part reported before the stall is kept


def test_sticky_device_error_in_an_optional_block_still_prints_the_line():
    d = run({'MOCK_STICKY': '1'})
    assert d['value'] > 0 and d['train'] == {'eager': True}                # the part reported before the error is kept
    assert d['extras'].startswith('aborted: ') and 'device unusable' in d['extras']
    assert d['configs']['2_deformable_faster'] == {'images_per_sec': 700} and d['configs']['3_fpn'] is None


def test_roofline_object_and_sweep_keys_with_a_stand_in_timer(monkeypatch):
    """bench.relation_kernel_roofline on its real code with the per-point GPU timing replaced: the contract's roofline keys, the
    SURVEY 8(d) algorithmic bytes, the N=3000 entry with its ncu traffic, 16 sweep points; a failing sweep point is reported inside
    `sweep` and leaves the headline roofline intact."""
    sys.path.insert(0, ROOT)
    import torch
    import bench
    import relnet_b200  # noqa: F401

    def point(ops, synth, device, flush, N, d, H, reps):
        return dict(N=N, d=d, H=H, dk=d // H, F_tc_gflop=round(4.0 * N * N * d / 1e9, 4), path='stand-in',
                    module_us=45.0 + N / 10, nm_us=30.0 + N / 5, proj_us=18.0)
    real_empty = torch.empty
    monkeypatch.setattr(torch, 'empty', lambda *a, **k: real_empty(16, dtype=torch.uint8))
    monkeypatch.setattr(bench, '_relation_point', point)
    pk = dict(hbm_gbs=6570.6, tflops=1720.8, tflops_sustained=1500.0, source='test')
    roof, times, sw = bench.relation_kernel_roofline(None, pk, 'cpu', sweep=True)
    assert {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'} <= set(roof)
    assert roof['bound'] == 'tensor' and roof['unit'] == 'TFLOP/s' and roof['peak'] == 1720.8
    N = M = 300; d = 1024; E = 64; H = 16
    assert roof['algorithmic_bytes'] == 2 * (N * d + 2 * M * d) + 16 * max(N, M) + 4 * (E * H + H) + 2 * N * d       # SURVEY 8(d), s = 2
    assert abs(roof['achieved'] - 4.0 * N * M * d / (roof['duration_us'] * 1e-6) / 1e12) < 1e-3
    assert abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-5
    assert len(sw) == 16 and {(r['N'], r['d'], r['H']) for r in sw} == {(n, dd, hh) for n in (100, 300, 1000, 3000) for dd in (256, 1024) for hh in (4, 16)}
    big = roof['at_N3000']
    assert big['algorithmic_bytes'] == 2 * (3000 * 1024 * 3) + 16 * 3000 + 4 * (64 * 16 + 16) + 2 * 3000 * 1024
    assert big['traffic'] is None or big['traffic'] >= big['algorithmic_bytes']
    assert roof['xu']['at_N3000']['mufu_ops'] == 3000.0 * 3000 * (34 + 16)
    json.dumps(roof), json.dumps(sw)                                    # serialisable as they are
    assert set(times) == {'module', 'nm_stage', 'proj'}

    def flaky(ops, synth, device, flush, N, d, H, reps):
        if N == 1000:
            raise RuntimeError('CUDA error: launch failed')
        return point(ops, synth, device, flush, N, d, H, reps)
    monkeypatch.setattr(bench, '_relation_point', flaky)
    roof2, _, sw2 = bench.relation_kernel_roofline(None, pk, 'cpu', sweep=True)
    assert roof2['frac'] == roof['frac'] and 'at_N3000' not in roof2
    assert sw2[-1] == {'failed': 'CUDA error: launch failed'} and len(sw2) == 9


def test_a_rank_that_aborts_its_optional_blocks_leaves_with_its_peers_not_before_them():
    """Under torchrun a process that disappears while the others sit in a collective turns a reported failure into a job abort:
    the aborting rank stays until the common deadline (rank 0 prints its line at once), then every rank exits 0."""
    import time
    e = dict(os.environ, MOCK_STICKY='1', MOCK_RANK='1')
    t0 = time.time()
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', '_mock_bench.py'), '--extras-budget', '7'], capture_output=True,
                       text=True, env=e, timeout=120)
    assert p.returncode == 0 and p.stdout.strip() == ''                  # rank 1 never prints the line
    assert 'optional blocks aborted on rank 1' in p.stderr
    assert time.time() - t0 >= 7.0                                       # it waited for the deadline
    e['MOCK_RANK'] = '0'
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', '_mock_bench.py'), '--extras-budget', '7'], capture_output=True,
                       text=True, env=e, timeout=120)
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert p.returncode == 0 and len(lines) == 1
    d = json.loads(lines[0])
    assert d['n_gpus'] == 2 and d['extras'].startswith('aborted: ') and 'cpu_baseline' not in d      # cpu_baseline: N = 1 only
