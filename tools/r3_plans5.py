"""dhqr_qr_host_f64 at BASELINE config 3: does it matter who wrote the pinned host buffer last (CPU memcpy as in bench.py's e2e leg vs a
device-to-host copy)?  Wall time + upload timeline for both, first upload of 384 / 768 columns."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C
import torch
import dhqr_b200 as D
dev = torch.device("cuda:0"); h = D.default_handle(0)
m, n = 32768, 4096
host = torch.empty((n, m), dtype=torch.float64).pin_memory()
src = torch.empty((n, m), dtype=torch.float64, device=dev)
D.fill_uniform_(src.t(), 0)
pristine = src.cpu()                       # pageable CPU copy, like bench.py's `pristine`
al = torch.empty(n, dtype=torch.float64).pin_memory()
def run(refresh, reps=4):
    ts = []
    for _ in range(reps):
        if refresh == "cpu": host.copy_(pristine)
        else: host.copy_(src)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        D._lib.call("dhqr_qr_host_f64", h.raw, m, n, C.c_void_p(host.data_ptr()), m, C.c_void_p(al.data_ptr()), 0)
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts
run("d2h", 2)
for rnd in range(2):
    for refresh in ("cpu", "d2h"):
        for first, chunk in ((0, 512), (768, 512), (0, 0)):
            h.set_option("host_first", first); h.set_option("host_chunk", chunk)
            ts = run(refresh)
            print(f"buffer last written by {refresh}: first {first:4d} chunk {chunk:4d}: " + " ".join(f"{t:.2f}" for t in ts) + " ms", flush=True)
h.set_option("host_first", 0); h.set_option("host_chunk", 512); h.set_option("host_trace", 1)
print("--- trace, buffer last written by the CPU", flush=True)
run("cpu", 1)
print("--- trace, buffer last written by a device-to-host copy", flush=True)
run("d2h", 1)
