"""Scratch timing of the preamble-search kernel on random device data (developer tool)."""
import os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from softgnss_python_b200 import _native, postnav
n, ms = int(sys.argv[1]) if len(sys.argv) > 1 else 256, 37000
L = _native.lib()
big = torch.randn((n, 13, ms), dtype=torch.float64, device="cuda")
ipv = big.view(n, 13 * ms)[:, 3 * ms:4 * ms]
first = torch.zeros(n, dtype=torch.int32, device="cuda")
bits = torch.zeros((n, 1501), dtype=torch.uint8, device="cuda")
valid = torch.zeros(n, dtype=torch.int32, device="cuda")
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for mode in ("device outputs", "host outputs"):
    ts = []
    for it in range(6):
        flush.fill_(it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if mode == "device outputs":
            L.check(L.dll.sgx_find_preambles(ipv.data_ptr(), 13 * ms, n, ms, first.data_ptr(), bits.data_ptr(), valid.data_ptr(), None))
        else:
            postnav.find_preambles_batch(ipv)
        e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    print(mode, "us per call:", ["%.0f" % t for t in ts], "-> %.0f GB/s" % (n * ms * 8 / (min(ts) * 1e-6) / 1e9))
