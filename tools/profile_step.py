#!/usr/bin/env python
"""torch.profiler view of one dg mode cycle of bench.py's workload: GPU time by kernel and the
wall time per training step (to see what the hot-path kernels leave on the table)."""
import sys, time
from pathlib import Path
import torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench
from dgod_b200.dg import DGFRCNN

dev = torch.device("cuda")
torch.backends.cudnn.benchmark = True
torch.manual_seed(0)
B = 8
model = DGFRCNN(9, B, "dg", bench.REG_WEIGHTS, 2).to(dev).train().to(memory_format=torch.channels_last)
res = [bench.to_device(b, dev) for b in bench.synthetic_batches(4, B, 2, 0)]
bench.calibrate(model.detector, res[0][0])
if "--eager" not in sys.argv:          # bench.py's default host-side setup: folded frozen BN + graphed backbone
    from dgod_b200.utils import fold_frozen_bn
    fold_frozen_bn(model.detector.backbone)
    with torch.no_grad():
        shape = model.detector.transform([i for i in res[0][0]], None)[0].tensors.shape
    model.detector.backbone = torch.cuda.make_graphed_callables(model.detector.backbone, (torch.rand(shape, device=dev),), num_warmup_iters=3)
opt = model.configure_optimizer(lr=bench.BENCH_LR)
_head_forward = model.detector.rpn.head.forward


def _ranged_head_forward(x):          # the RPN head's forward as one range in the table ("rpn_head_forward")
    with torch.profiler.record_function("rpn_head_forward"):
        return _head_forward(x)


model.detector.rpn.head.forward = _ranged_head_forward

def step(b):
    loss = model.training_step(b)
    opt.zero_grad(set_to_none=True)
    loss.backward()
    opt.step()

for _ in range(2):
    for s in range(8):
        step(res[(s // 2) % 4])
torch.cuda.synchronize()
for s in range(8):
    mode = model.mode
    t0 = time.perf_counter(); step(res[(s // 2) % 4]); torch.cuda.synchronize()
    print(f"mode {mode}: {1e3 * (time.perf_counter() - t0):7.1f} ms")
torch.cuda.synchronize(); t0 = time.perf_counter()
for s in range(8):
    step(res[(s // 2) % 4])
torch.cuda.synchronize()
print(f"8-step cycle, no syncs in between: {1e3 * (time.perf_counter() - t0):7.1f} ms")
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
    for s in range(8):
        step(res[(s // 2) % 4])
    torch.cuda.synchronize()
from torch.autograd import DeviceType
kern = [e for e in prof.events() if e.device_type == DeviceType.CUDA]
gpu_ms = sum(e.device_time for e in kern) / 1e3
ours = sum(e.device_time for e in kern if e.name.startswith("dgod::") or "dgod::" in e.name) / 1e3
span = (max(e.time_range.end for e in kern) - min(e.time_range.start for e in kern)) / 1e3
print(f"GPU kernels over the 8-step cycle: {len(kern)} launches, {gpu_ms:.1f} ms busy in a {span:.1f} ms span "
      f"({100 * gpu_ms / span:.0f} % busy); dgod_b200 kernels {ours:.2f} ms")
ka = prof.key_averages()
print(prof.key_averages().table(sort_by="self_cuda_time_total", row_limit=-1, max_name_column_width=110))
