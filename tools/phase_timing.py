"""Build a -DCPT_PHASE_TIMING copy of the library and print where the cycles of a frame go (GPU box).

usage: python tools/phase_timing.py [clips] [frames] [single]   (single = 1: the single persistent kernel, else the split plan)"""
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = os.path.join(ROOT, "classifier-pipeline_b200")


def main(clips=148, frames=300, single=0):
    import torch
    from classifier_pipeline_b200 import native

    dbg = os.path.join(PKG, "libcptrack_timing.so")
    srcs = [os.path.join(PKG, "csrc", f) for f in sorted(os.listdir(os.path.join(PKG, "csrc"))) if f.endswith(".cu")]
    subprocess.run(["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-DCPT_PHASE_TIMING",
                    "-Xcompiler", "-fPIC", "-shared", "-o", dbg] + srcs, check=True)
    native.LIB_PATH = dbg
    from classifier_pipeline_b200.batch import BatchExtractor, linear_clips
    from classifier_pipeline_b200.synthetic import MODELS, make_clips_torch

    ex = BatchExtractor(device=0, max_regions=16)
    slots = [ex.ctx.weight_table(m[3], max_frames=2048) for m in MODELS]
    d_frames, models = make_clips_torch(clips, frames, torch.device("cuda", 0))
    cl = linear_clips([frames] * clips, np.array([MODELS[m][2] for m in models]), np.array([slots[m] for m in models]))
    out = {}
    if single:
        native.check(ex.ctx.lib.cpt_debug_force_single_kernel(ex.ctx._h, 1))
    ex.extract_device(d_frames, cl, out=out)
    torch.cuda.synchronize()
    buf = (ctypes.c_longlong * 32)()
    native.check(ex.ctx.lib.cpt_debug_phase_cycles(ex.ctx._h, buf, 1))
    ex.extract_device(d_frames, cl, out=out)
    torch.cuda.synchronize()
    native.check(ex.ctx.lib.cpt_debug_phase_cycles(ex.ctx._h, buf, 0))
    total = clips * frames
    if not single:
        # frame_regions_kernel, thread 0 of every CTA (cycles include the waits at the CTA's barriers)
        names = {7: "header + info", 15: "quad bytes -> hot rows", 4: "band record + work lists", 5: "normalise", 8: "blur + threshold",
                 9: "components (close .. labels)"}
        for i, n in names.items():
            print("{:28s} {:9.0f} cycles/frame".format(n, buf[i] / total))
        print("lists: normalise {:.1f} groups/frame, blur {:.1f}; frames that reach the components stage {:.4f}".format(
            buf[28] / total, buf[29] / total, buf[30] / total))
        return
    names = {14: "S fused sweep", 5: "S  of which: waiting for staged rows", 6: "S wait scalars + ballots", 2: "S message",
             8: "producer: wait free stage", 9: "producer: issue copies",
             7: "M wait sweep", 16: "M scalars thread 0", 3: "M scalars bar", 15: "M quad maxima -> hot rows", 4: "M marks+lists",
             11: "C wait mask", 12: "C components",
             20: "C  close+reset+bar", 21: "C  run starts+bar", 22: "C  unions+bar", 23: "C  roots+bar", 24: "C  run stats+bar",
             25: "C  rank+bar", 26: "C  label writes", 27: "C  variance+bar"}
    for i, n in names.items():
        print("{:22s} {:9.0f} cycles/frame".format(n, buf[i] / total))
    print("lists: normalise {:.1f} groups/frame, blur {:.1f}; dense frames {:.4f}, no-foreground frames {:.4f}".format(
        buf[28] / total, buf[29] / total, buf[30] / total, buf[31] / total))
    print("S total {:.0f} cycles/frame, M total {:.0f}, C total {:.0f}".format(
        sum(buf[i] for i in (14, 6, 2)) / total, sum(buf[i] for i in (7, 16, 3, 15, 4, 5, 8, 9)) / total, (buf[11] + buf[12]) / total))


if __name__ == "__main__":
    main(*[int(x) for x in sys.argv[1:]])
