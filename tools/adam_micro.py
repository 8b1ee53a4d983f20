"""K7 micro-benchmark: the Adam kernel on 8,018,624 parameters with random and with 'trained-network-like' data (many
tiny gradients), with / without the bf16 shadow."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from acme_b200 import _capi

n = 8_018_624
gen = torch.Generator(device='cuda').manual_seed(0)
step = torch.full((1,), 50, dtype=torch.int64, device='cuda')


def run(name, g, m, v, shadow):
  p = torch.randn(n, device='cuda', generator=gen)
  sh = torch.empty(n, dtype=torch.bfloat16, device='cuda') if shadow else None
  call = lambda: _capi.call('b200rl_adam', n, p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), 1e-3, 0.9,
                            0.999, 1e-8, 0, None, _capi.ptr(sh), _capi.current_stream())
  for _ in range(3):
    call()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(20):
    call()
  e1.record(); torch.cuda.synchronize()
  us = e0.elapsed_time(e1) / 20 * 1e3
  bytes_ = n * (28 + (2 if shadow else 0))
  print(f'{name:46s} shadow={int(shadow)}  {us:6.1f} us  {bytes_ / us / 1e3:7.1f} GB/s')


for shadow in (False, True):
  g = torch.randn(n, device='cuda', generator=gen)
  run('random N(0,1) g, m, |v|', g, torch.randn(n, device='cuda', generator=gen), torch.randn(n, device='cuda', generator=gen).abs_(), shadow)
  gs = g * torch.pow(10.0, -torch.rand(n, device='cuda', generator=gen) * 12)        # gradients spanning 12 decades
  run('g over 12 decades, m = 0.1 g, v = 0.001 g^2', gs, 0.1 * gs, 0.001 * gs * gs, shadow)
  z = torch.zeros(n, device='cuda')
  gz = g * (torch.rand(n, device='cuda', generator=gen) < 0.3)
  run('70% exactly-zero g, m = v = 0', gz, z.clone(), z.clone(), shadow)
