"""bench.py's host-side control flow with every GPU-touching piece replaced by a stand-in (no CUDA in the CPU suite): used by
tests/test_bench_contract_cpu.py to check the ONE-JSON-line contract, the contract keys, a failing optional block and the
--extras-budget deadline.  MOCK_FAIL=1: the training block raises; MOCK_STICKY=1: it raises and every later synchronize raises too (sticky device error);
MOCK_HANG=1: the configs[3] block stalls for 30 s."""
import sys, types, time, json, io, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
# ---- fakes
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda *a, **k: None
_sync_state = {'armed': False}
def _sync(*a, **k):
    if _sync_state['armed']:           # MOCK_STICKY: a device error that every later CUDA call reports again
        raise RuntimeError('CUDA error: an illegal memory access was encountered')
torch.cuda.synchronize = _sync
torch.cuda.empty_cache = lambda: None
_real_device = torch.device
class FakeTensorOps: pass
bench.timed = lambda fn, steps, warmup, dist_on, after=None: 33.0
bench.count_launches = lambda fn: (30, 108, {'k': 1})
bench.relation_kernel_roofline = lambda ops, pk, device, sweep=True: ({'frac': 0.007}, {'module': 45.0}, [{'N': 300}])
bench.cpu_baseline = lambda steps=1: {'value': 1.6}
bench.config2_block = lambda *a, **k: {'images_per_sec': 700}
def fake_cfg3(args, prec, device, world, rank, dist_on, train=True, report=None):
    if report: report({'test': 1})
    if os.environ.get('MOCK_HANG'): time.sleep(30)
    return {'test': 1, 'train': 2}
bench.config3_block = fake_cfg3
def fake_train(args, ts, images, im_info, device, world, rank, dist_on, mode, report=None):
    if report: report({'eager': True})
    if os.environ.get('MOCK_FAIL'): raise RuntimeError('boom')
    if os.environ.get('MOCK_STICKY'):
        _sync_state['armed'] = True
        raise RuntimeError('CUDA error: an illegal memory access was encountered')
    return {'graph': True}
bench.train_block = fake_train
class ClockSampler:
    def __init__(self, i): self.stop_flag = False
    def start(self): pass
    def summary(self): return {'sm_mhz': 1965}
bench.ClockSampler = ClockSampler
bench.require_built = lambda: None
import relnet_b200
from relnet_b200 import ops, pipeline, trunk as TR, train as TN
ops.default_precision = lambda: 'f16'
ops.device_info = lambda: dict(sm100=True, sm_count=148, cc=(10, 0))
ops.proposal = lambda *a, **k: (None, None, torch.tensor([300]))
class FakeHead:
    def __init__(self, *a, **k): self.cfg = {}
    def forward(self, *a): return {}
pipeline.RelationHead = FakeHead
pipeline.init_head_params = lambda *a, **k: {}
class FakeTrunk:
    def __call__(self, im): return (torch.zeros(1), torch.zeros(1), torch.zeros(1))
TR.make_trunk = lambda *a, **k: FakeTrunk()
class FakeGraphed:
    def __init__(self, fn, inputs, warmup=3): self.out = {'learn_nms_sorted_bbox': torch.zeros(100, 80, 4), 'nms_final_score_output': torch.zeros(100, 80)}
    def __call__(self, *a): return self.out
pipeline.GraphedStep = FakeGraphed
pipeline.Detector = lambda *a, **k: (lambda im: {})
class FakeStreamer:
    depth = 2
    def __init__(self, *a, **k): pass
    def submit(self, im): return 0
    def collect(self, t): return None
pipeline.StreamingDetector = FakeStreamer
class FakeTS:
    def __init__(self, *a, **k): pass
TN.TrainStep = FakeTS
# tensors: .to(device) on cuda -> keep on cpu
_orig_to = torch.Tensor.to
def to(self, *a, **k):
    a = tuple(('cpu' if (isinstance(x, torch.device) and x.type == 'cuda') else x) for x in a)
    k = {kk: ('cpu' if (isinstance(v, torch.device) and v.type == 'cuda') else v) for kk, v in k.items()}
    return _orig_to(self, *a, **k)
torch.Tensor.to = to
torch.Tensor.pin_memory = lambda self: self
_orig_randn = torch.randn
torch.randn = lambda *a, **k: _orig_randn(*((8, 8) if a[:2] == (4096, 4096) else a), **{kk: v for kk, v in k.items() if kk != "device"})
if os.environ.get('MOCK_RANK'):        # one rank of a 2-process job, process-group calls replaced (peers are not simulated)
    import torch.distributed as dist
    os.environ.update(WORLD_SIZE='2', RANK=os.environ['MOCK_RANK'], LOCAL_RANK='0')
    dist.init_process_group = lambda *a, **k: None
    dist.barrier = lambda *a, **k: None
    dist.destroy_process_group = lambda *a, **k: None
sys.argv = ['bench.py', '--steps', '4', '--warmup', '3'] + sys.argv[1:]
bench.main()
