"""Dry run of bench.py's b200 arm on the CPU (run by tests/test_bench_contract.py in a subprocess): the handful of torch.cuda
calls are stubbed and the library is replaced by the host-compiled build of tests/emu.  It checks that the Python logic of the
bench runs against the current ABI and that the JSON line carries the contract's keys — the numbers mean nothing here."""
import sys, types, runpy, json, io, contextlib
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
torch.cuda.set_device = lambda *a, **k: None
torch.cuda.synchronize = lambda *a, **k: None
_orig_tensor = torch.tensor
torch.tensor = lambda *a, **k: _orig_tensor(*a, **{kk: vv for kk, vv in k.items() if kk != 'device'})
torch.Tensor.pin_memory = lambda self, *a, **k: self
import emu_lib
from serf_b200 import sim
sim._LIB = emu_lib.lib()          # bypass the product loader (which refuses this build) for the dry run only
import shutil
import tempfile
import numpy as np
dump = tempfile.mkdtemp(prefix='bench_dump_')
sys.argv = ['bench.py', '--nodes', '30000', '--steps', '3', '--warmup', '3', '--ref-nodes', '20000', '--dump-outputs', dump]
buf = io.StringIO()
with contextlib.redirect_stdout(buf):
    runpy.run_path(os.path.join(ROOT, 'bench.py'), run_name='__main__')
line = json.loads(buf.getvalue().strip().splitlines()[-1])
# --dump-outputs: every result of the last step as float64 (30 000 nodes: no sampling), consistent with the JSON line
files = sorted(os.listdir(dump))
assert files == sorted(['node_ids.npy', 'lamport_time.npy', 'convergence.npy', 'stats.npy', 'state_hash.npy'] +
                       [f'{v}_slot{s}.npy' for v in ('member_status', 'status_ltime') for s in range(2)]), files
out = {f[:-4]: np.load(os.path.join(dump, f)) for f in files}
assert all(a.dtype == np.float64 for a in out.values()) and sum(os.path.getsize(os.path.join(dump, f)) for f in files) <= 64 << 20
ids = out['node_ids'].astype(np.int64)
assert ids.size == 30000 and (np.diff(ids) > 0).all()
assert out['convergence'][0] == line['ticks_to_convergence'] and out['convergence'][1] == 1
assert out['stats'][2] == line['edge_updates_per_step']
assert (out['member_status_slot0'] == 3).sum() >= ids.size - 8           # the leaver is Left in (nearly) every view
shutil.rmtree(dump)
need = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
        "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"]
missing = [k for k in need if k not in line]
assert not missing, missing
assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and line["roofline"]["bound"] == "hbm"
assert set(line["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and line["e2e"]["d2h_bytes_per_step"] > 0
assert set(line["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"}
assert line["gpu_launches"] > 0 and line["steps"] == 3 and line["n_gpus"] == 1
print("bench dry run ok:", line["metric"], line["config"]["workload"] if "workload" in line["config"] else line["config"])
