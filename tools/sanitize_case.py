"""A small end-to-end pass of every product kernel family for compute-sanitizer (memcheck / racecheck):
bf16 stack forward + backward (tcgen05 / bulk-copy kernels, poolfuse, projections), fp32 stack forward + backward (the
generic kernels), MTA forward + backward.    compute-sanitizer --tool memcheck python tools/sanitize_case.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mm_distillnet_b200 as mmd  # noqa: E402

dev = torch.device("cuda", 0)
CC = [48, 120, 352]
torch.manual_seed(0)
for dtype in (torch.bfloat16, torch.float32):
    stack = mmd.BiFPNStack(*[mmd.BiFPN(112, CC, first_time=(i == 0)) for i in range(2)]).to(dev).train()
    xs = [torch.randn(1, c, 48 >> i, 48 >> i, device=dev).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
          for i, c in enumerate(CC)]
    out = stack(tuple(xs))
    crit = mmd.MTALoss()
    teachers = [[o.detach().flip(0) * 0.5 for o in out] for _ in range(2)]
    kd = crit.forward_each(list(out), teachers) if dtype == torch.bfloat16 else torch.stack([crit(list(out), t) for t in teachers])
    (0.005 * kd.sum() + sum(o.float().mean() for o in out)).backward()
    stack.eval()
    with torch.no_grad():
        stack(tuple(x.detach() for x in xs))
    torch.cuda.synchronize()
    print(dtype, "ok", float(kd.sum()))

# detection heads (node kernels with one input, header halves, gather / scatter / act glue) and the detection loss
import numpy as np  # noqa: E402
for dtype in (torch.bfloat16, torch.float32):
    reg, cls = mmd.Regressor(112, 9, 3).to(dev).train(), mmd.Classifier(112, 9, 20, 3).to(dev).train()
    feats = [torch.randn(1, 112, max(48 >> i, 1), max(48 >> i, 1), device=dev).to(dtype).requires_grad_(True) for i in range(5)]
    r, ar = reg(feats)
    c, ac = cls(feats)
    N = r.shape[1]
    xy = torch.rand(N, 2, device=dev) * 300
    anchors = torch.cat([xy, xy + 20 + torch.rand(N, 2, device=dev) * 100], dim=1).unsqueeze(0)
    ann = [np.array([[20, 30, 200, 180, 3], [100, 90, 260, 300, 7]], dtype=np.float32)]
    lr, lc = mmd.YetAnotherFocalLoss()((c, r, anchors), ann)
    (lr + lc + ar.float().mean() + ac.float().mean()).sum().backward()
    reg.eval()
    with torch.no_grad():
        reg([f.detach() for f in feats])
    torch.cuda.synchronize()
    print(dtype, "heads + focal ok", float(lr), float(lc))

# pseudo-label generation (score / compact / NMS / merge kernels) feeding the detection loss on device-made labels
from mm_distillnet_b200 import pseudo as PS  # noqa: E402
for dtype in (torch.bfloat16, torch.float32):
    B, K, T = 2, 20, 2
    ys, xs_ = torch.meshgrid(torch.arange(4, 128, 8.0), torch.arange(4, 128, 8.0), indexing="ij")
    ctr = torch.stack([ys.reshape(-1), xs_.reshape(-1)], dim=1).repeat_interleave(3, dim=0)
    half = torch.tensor([16.0, 20.0, 26.0]).repeat(ctr.shape[0] // 3).unsqueeze(1)
    anchors = torch.cat([ctr - half, ctr + half], dim=1).unsqueeze(0).to(dev)          # [1, 768, 4] (y1, x1, y2, x2)
    N = anchors.shape[1]
    preds = []
    for t in range(T):
        c = 0.02 + 0.1 * torch.rand(B, N, K, device=dev)
        hot = torch.randint(0, N, (B, 40), device=dev)
        for b in range(B):
            c[b, hot[b], torch.randint(0, K, (40,), device=dev)] = 0.4 + 0.5 * torch.rand(40, device=dev)
        preds.append((c.to(dtype), (0.1 * torch.randn(B, N, 4, device=dev)).to(dtype), anchors))
    vcd = {"predictions_txt2i": {"c%d" % i: i for i in range(0, K, 2)}, "predictions_i2txt": {i: "c%d" % i for i in range(0, K, 2)},
           "labels_txt2i": {"c%d" % i: i // 2 for i in range(0, K, 2)}}
    cfg = {"conf_threshold": "0.3", "nms_threshold": "0.5", "image_size": "128", "ignore_labels": "4"}
    labels = PS.teacher_pseudo_labels(preds, vcd, cfg, cap=512, max_rows=64, max_labels=64)
    cs = torch.rand(B, N, K, device=dev).to(dtype).requires_grad_(True)
    rs = torch.randn(B, N, 4, device=dev).to(dtype).requires_grad_(True)
    lr, lc = mmd.YetAnotherFocalLoss()((cs, rs, anchors), labels)
    (lr + lc).sum().backward()
    torch.cuda.synchronize()
    print(dtype, "pseudo-labels + focal ok", labels.counts.tolist(), float(lr), float(lc))

# the one-launch optimizer step over a flat gradient buffer (adam.cu)
ps = [torch.nn.Parameter(torch.randn(*s, device=dev)) for s in ((112,), (112, 112, 1, 1), (3,), (1025,))]
flat = torch.randn(sum(p.numel() for p in ps) + 8, device=dev)
o = 0
for p in ps:
    p.grad = flat[o:o + p.numel()].view(p.shape)
    o += p.numel() + 2
opt = mmd.FlatAdam(ps, lr=1e-3, weight_decay=1e-2, decoupled_weight_decay=True)
for _ in range(3):
    opt.step(flat)
torch.cuda.synchronize()
print("adam ok", int(opt.step_count), float(ps[1].abs().mean()))

# frozen BatchNorm: every other node's BatchNorm in eval() inside a training stack (frozen vector written by the prep
# launch, no statistics, constant-coefficient BatchNorm backward), plus a frozen head level
for dtype in (torch.bfloat16, torch.float32):
    stack = mmd.BiFPNStack(*[mmd.BiFPN(112, CC, first_time=(i == 0)) for i in range(2)]).to(dev).train()
    bns = [m for m in stack.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for m in bns[::2]:
        m.eval()
    xs = [torch.randn(1, c, 48 >> i, 48 >> i, device=dev).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
          for i, c in enumerate(CC)]
    out = stack(tuple(xs))
    reg = mmd.Regressor(112, 9, 3).to(dev).train()
    for m in reg.bn_list[2]:
        m.eval()
    r, ar = reg(out)
    (sum(o.float().mean() for o in out) + r.float().mean() + ar.float().mean()).backward()
    torch.cuda.synchronize()
    print(dtype, "frozen BatchNorm ok", int(bns[0].num_batches_tracked), int(bns[1].num_batches_tracked))
