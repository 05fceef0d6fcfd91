"""H2D/D2H rate of a pinned 8 MB buffer allocated on each NUMA node of the host (A/B on one box)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from of_dis_b200 import numa
torch.cuda.set_device(0)
st = torch.cuda.Stream(); torch.cuda.set_stream(st)
print('gpu bus', numa.gpu_pci_bus_id(0), 'sysfs node/cpus', numa.gpu_numa_cpus(0)[0], len(numa.gpu_numa_cpus(0)[1]))
all_cpus = os.sched_getaffinity(0)
nodes = sorted(int(d[4:]) for d in os.listdir('/sys/devices/system/node') if d.startswith('node') and d[4:].isdigit())
N = 2 * 1024 * 1024
dev = torch.empty(N, dtype=torch.float32, device='cuda')
def t(fn, n=40):
    for _ in range(10): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(n): fn()
    b.record(st); torch.cuda.synchronize()
    return a.elapsed_time(b) / n
bufs = {}
for nd in nodes:
    cpus = numa._parse_cpulist(open('/sys/devices/system/node/node%d/cpulist' % nd).read()) & all_cpus
    if not cpus: continue
    os.sched_setaffinity(0, cpus)
    h = torch.empty(N, dtype=torch.float32, pin_memory=True); h.fill_(1.0)
    bufs[nd] = h
os.sched_setaffinity(0, all_cpus)
for rep in range(3):
    for nd, h in bufs.items():
        ms = t(lambda: dev.copy_(h, non_blocking=True)); ms2 = t(lambda: h.copy_(dev, non_blocking=True))
        print('round %d node %d: H2D %.1f GB/s  D2H %.1f GB/s' % (rep, nd, N * 4 / 1e6 / ms, N * 4 / 1e6 / ms2))
