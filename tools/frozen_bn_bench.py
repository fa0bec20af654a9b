"""Device-timed student step with frozen BatchNorm: DistillStep (2-cell student + 3 frozen teachers, bf16, lockstep
launches, captured into a CUDA graph) at B = 32 with 96 x 96 P3 (the bench.py shape), every student BatchNorm layer in
eval() against every layer in train().  Prints one JSON line per arm and a summary line with the card's name and power
limit.    python tools/frozen_bn_bench.py [--batch 32] [--steps 200] [--repeats 3]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mm_distillnet_b200 as mmd  # noqa: E402

CC = [48, 120, 352]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def make_step(frozen, B, dev):
    torch.manual_seed(0)
    student = mmd.BiFPNStack(*[mmd.BiFPN(112, CC, first_time=(i == 0)) for i in range(2)]).to(dev).train()
    if frozen:
        for m in student.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.eval()
    teachers = []
    for k in range(3):
        torch.manual_seed(10 + k)
        teachers.append(mmd.BiFPNStack(*[mmd.BiFPN(112, CC, first_time=(i == 0)) for i in range(2)]).to(dev).eval())
    gen = torch.Generator().manual_seed(1)
    xs = [[torch.randn(B, c, 96 >> i, 96 >> i, generator=gen).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
           for i, c in enumerate(CC)] for _ in range(4)]
    step = mmd.DistillStep(student, teachers)
    step.capture(tuple(xs[0]), [tuple(x) for x in xs[1:]], warmup=3)
    return step


def time_step(step, n):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(10):
        step.replay()
    torch.cuda.synchronize()
    start.record()
    for _ in range(n):
        step._graph.replay()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frozen_bn_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    steps = {"train": make_step(False, a.batch, dev), "frozen": make_step(True, a.batch, dev)}
    res = {k: [] for k in steps}
    for _ in range(a.repeats):          # alternate the arms so that clock / neighbour drift hits both
        for k, s in steps.items():
            res[k].append(time_step(s, a.steps))
    for k, v in res.items():
        print(json.dumps({"arm": k, "batch": a.batch, "ms_per_step": v, "min_ms": min(v)}))
    print(json.dumps({"card": card(), "frozen_over_train": min(res["frozen"]) / min(res["train"])}))


if __name__ == "__main__":
    main()
