"""Speed-of-light table for fast_kernel (VERDICT r01 item 3a): the same launch timed with the kernel cut off after
   mode 1: TMA tile load only   mode 2: + packed reject and pixel queue   mode 3: + exact pixel scores (no NMS / emit)
   mode 0: full kernel
on the bench input (KITTI-shaped 1242x375 stereo pairs, 64 images per launch, 4 rotating batches > L2).  The stage time is the
CUDA-event time of the `fast_nms` stage on the library's stream (borb_set_timing), mean over --steps launches.
usage: python tools/fast_ablation.py [--pairs 32] [--steps 40]  -> one JSON line."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                                  # noqa: E402  (device buffers only)
from orb_slam2_b200 import _lib, synth                                         # noqa: E402
from orb_slam2_b200.extractor import ORBextractor                              # noqa: E402

W, H, LEVEL_PIXELS = 1242, 375, 1441432


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=32)
    ap.add_argument("--steps", type=int, default=40)
    a = ap.parse_args()
    lib = _lib.load()
    B, NBUF = a.pairs, 4
    host = np.empty((NBUF, 2 * B, H, W), np.uint8)
    for p in range(B):
        l, r, _ = synth.stereo_pair(2024, 0, p, W, H)
        for j in range(NBUF):
            host[j, 2 * p] = np.roll(l, 37 * j, axis=0)
            host[j, 2 * p + 1] = np.roll(r, 37 * j, axis=0)
    d_in = torch.from_numpy(host).cuda()
    x = ORBextractor(2000)
    x.reserve(W, H, 2 * B)
    cap = x.capacity(W, H)
    nl = torch.zeros(B, dtype=torch.int32).pin_memory(); nr = torch.zeros(B, dtype=torch.int32).pin_memory()
    bf, b = 386.1448, float(np.float32(386.1448) / np.float32(718.856))

    def step(k):
        _lib.check(lib.borb_stereo_frames_device_enqueue(x._h, d_in[k % NBUF].data_ptr(), B, W, H, W, W * H, bf, b, nl.data_ptr(), nr.data_ptr(),
                                                         None, None, cap), "enqueue")

    out = {}
    names = {1: "tma_only", 2: "tma_reject", 3: "tma_reject_score", 0: "full"}
    for mode in (1, 2, 3, 0):
        _lib.check(lib.borb_debug_set_fast_mode(x._h, mode), "set_fast_mode")
        for k in range(4):
            step(k)
        _lib.check(lib.borb_sync(x._h), "sync")
        x.set_timing(True)
        for k in range(a.steps):
            step(k)
        _lib.check(lib.borb_sync(x._h), "sync")
        tot = (C.c_double * 8)(); n = C.c_uint64()
        _lib.check(lib.borb_stage_times_total(x._h, tot, C.byref(n)), "stage_times_total")
        x.set_timing(False)
        ms = tot[2] / max(n.value, 1)
        out[names[mode]] = {"fast_ms": ms, "GBps": LEVEL_PIXELS * 2 * B / (ms * 1e-3) / 1e9}
    peak = 6574.1
    pk = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        peak = float(json.load(open(pk))["hbm_gbs"])
    for v in out.values():
        v["frac_of_hbm_peak"] = v["GBps"] / peak
    print(json.dumps({"what": "fast_kernel ablation, 64 images (32 KITTI-shaped stereo pairs) per launch", "images_per_launch": 2 * B,
                      "algorithmic_bytes_per_launch": LEVEL_PIXELS * 2 * B, "hbm_peak_GBps": peak, "modes": out}))


if __name__ == "__main__":
    main()
