"""Data-parallel distillation step over the hot path (one process per GPU).

Mirrors what the reference's step wrapper + driver do around the BiFPN/MTA path
(ModelWithNMSLossAugmented.forward, src/optimization/train_methods.py:310-358: student forward with grad, every
teacher forward under no_grad in eval mode, `criterion_kd(features_s, features_t)` per teacher;
train_traditional, src/optimization/traditional.py:171-182: loss = w_kd * sum(stack(kd_losses)), backward) and
replaces the cfg's DataParallel / DDP gradient exchange (train_methods.py:944-961) by ONE NCCL all-reduce of the
student's flat fp32 gradient buffer (mean over ranks = DDP semantics; BatchNorm statistics stay per rank, MTA's
'batchmean' is over the local batch, teachers are replicated: no other cross-GPU traffic).
"""
import torch
import torch.distributed as dist

from .bifpn import BiFPN, BiFPNStack, forward_multi, forward_multi_heads, mark_state_changed
from .mta import MTALoss


def _flat_channels_last(like, device):
    """(flat uint8 buffer, views): one channels_last view per tensor of `like` (same logical [B,C,H,W] shape and dtype),
    laid out back to back at 256-byte aligned offsets of ONE allocation."""
    offs, total = [], 0
    for x in like:
        offs.append(total)
        total += (x.numel() * x.element_size() + 255) // 256 * 256
    flat = torch.empty(max(total, 256), dtype=torch.uint8, device=device)
    views = []
    for x, off in zip(like, offs):
        B, C, H, W = x.shape
        v = flat[off:off + x.numel() * x.element_size()].view(x.dtype).view(B, H, W, C).permute(0, 3, 1, 2)
        views.append(v)
    return flat, views


class DistillStep:
    """step(student_inputs, teacher_inputs) -> detached fp32 tensor [n_teachers, n_levels] of MTA losses.

    `student` is a BiFPNStack / BiFPN in train mode, `teachers` a list of BiFPNStack / BiFPN in eval mode.
    Inputs may live on the host (ideally pinned): they are copied to the device inside the call.  After the call
    every student parameter's `.grad` is a view into `self.flat_grad` (already averaged over the process group).
    """

    def __init__(self, student, teachers, criterion=None, w_kd=0.005, process_group=None, device=None,
                 batch_networks=True, kd_mode="each", optimizer=None):
        if not isinstance(student, (BiFPN, BiFPNStack)):
            raise TypeError("DistillStep drives mm_distillnet_b200 BiFPN / BiFPNStack modules")
        self.student, self.teachers = student, list(teachers)
        self.criterion = criterion if criterion is not None else MTALoss()
        self.w_kd = float(w_kd)
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        self.device = device if device is not None else next(student.parameters()).device
        self.flat_grad = None
        # optional mm_distillnet_b200.FlatAdam over the student's parameters: its one-launch step runs right behind the
        # gradient all-reduce, inside the call (and therefore inside a captured graph) — optimizer.step() of
        # src/optimization/traditional.py:190
        self.optimizer = optimizer
        self.batch_networks = bool(batch_networks)
        # "each": criterion_kd(features_s, features_t) per teacher, the shipped ModelWithNMSLossAugmented wrapper
        #         (train_methods.py:351-358) -> losses [n_teachers, n_levels];
        # "product": ONE call criterion_kd(features_s, [features_t1, features_t2, ...]) against the product of the
        #         teachers' attention maps, the ModelWithNMSKDListLoss wrapper (train_methods.py:165-262, KD term :256-261;
        #         MTALoss.forward list-of-lists branch, MTALoss.py:20-34) -> losses [1, n_levels]
        if kd_mode not in ("each", "product"):
            raise ValueError("DistillStep: kd_mode must be 'each' or 'product'")
        self.kd_mode = kd_mode
        # multi-stream fallback (stacks that cannot share launches): the frozen teachers and the student are independent until the MTA loss: each teacher stack runs on its own
        # CUDA stream so the small pyramid levels (P5-P7: fewer CTAs than SMs) of different networks overlap
        self.streams = [torch.cuda.Stream(device=self.device) for _ in self.teachers] if self.device.type == "cuda" else []
        student._runner.grad_sink = self._on_flat_grad
        for t in self.teachers:
            t.eval()
            for p in t.parameters():
                p.requires_grad_(False)     # train_methods.py:891-893

    def _on_flat_grad(self, flat):
        """Called from the student's backward with the single contiguous fp32 gradient buffer."""
        if self.world > 1:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.pg)
            flat.mul_(1.0 / self.world)
        self.flat_grad = flat

    def _to_device(self, xs):
        return tuple(x if x.device == self.device else x.to(self.device, non_blocking=True) for x in xs)

    def _batchable(self, xs, xts):
        stacks = [self.student] + self.teachers
        if len(stacks) > 4 or not all(isinstance(m, BiFPNStack) and m.fusable() for m in stacks):
            return False
        return all(x.dtype == torch.bfloat16 for x in xs) and all(x.dtype == torch.bfloat16 for t in xts for x in t) and \
            all(t[0].shape[0] == xs[0].shape[0] for t in xts)

    def _kd(self, feats_s, feats_t_all):
        """criterion_kd(features_s, features_t) per teacher (train_methods.py:351-358) -> Tensor[n_teachers, n_levels]."""
        teachers = [[f.detach() for f in ft] for ft in feats_t_all]
        if self.kd_mode == "product":
            return self.criterion(feats_s, teachers if len(teachers) > 1 else teachers[0]).unsqueeze(0)
        if isinstance(self.criterion, MTALoss) and 1 <= len(teachers) <= 4:
            return self.criterion.forward_each(feats_s, teachers)      # one set of launches for all teachers
        return torch.stack([self.criterion(feats_s, t) for t in teachers])

    def __call__(self, student_inputs, teacher_inputs):
        xs = self._to_device(student_inputs)
        xts = [self._to_device(t) for t in teacher_inputs]
        if self.batch_networks and self._batchable(xs, xts):
            # one lockstep pass: the same node of the student and of every teacher shares a launch
            outs = forward_multi([(self.student, xs)] + [(t, x) for t, x in zip(self.teachers, xts)])
            feats_s, feats_t_all = outs[0], outs[1:]
            kd = self._kd(feats_s, feats_t_all)                                                  # :351-358
        else:
            main = torch.cuda.current_stream(self.device)
            feats_t_all = []
            for teacher, tin, st in zip(self.teachers, xts, self.streams):   # train_methods.py:320-336
                st.wait_stream(main)
                with torch.cuda.stream(st), torch.no_grad():
                    feats_t = teacher(tin)
                    for f in feats_t:
                        f.record_stream(main)
                feats_t_all.append(feats_t)
            feats_s = self.student(xs)                                   # :318
            for st in self.streams:
                main.wait_stream(st)
            kd = self._kd(feats_s, feats_t_all)                          # :351-358
        # loss = w_kd * sum(stack(kd_losses)); loss.backward()  (traditional.py:171-182, KD term): d loss / d kd[t, l] is
        # the constant w_kd, so the backward starts from that constant instead of three scalar kernels (sum, mul, expand)
        g = getattr(self, "_kd_grad", None)
        if g is None or g.shape != kd.shape or g.device != kd.device:
            g = self._kd_grad = torch.full_like(kd.detach(), self.w_kd)
        torch.autograd.backward([kd], [g])
        if self.optimizer is not None:
            self.optimizer.step(self.flat_grad)
        return kd.detach()

    # ---- CUDA-graph replay of the whole step -----------------------------------------------------------------------
    def _capture_set(self, student_inputs, teacher_inputs, warmup):
        """One static input set (channels_last views of ONE flat buffer) + the step captured over it."""
        dev = self.device
        srcs = list(student_inputs) + [x for xs in teacher_inputs for x in xs]
        flat, views = _flat_channels_last(srcs, dev)
        with torch.no_grad():
            for v, x in zip(views, srcs):
                v.copy_(x.detach())
        ns = len(student_inputs)
        g_xs = [v.requires_grad_(bool(x.requires_grad)) for v, x in zip(views[:ns], student_inputs)]
        g_xt, k = [], ns
        for xs in teacher_inputs:
            g_xt.append(views[k:k + len(xs)])
            k += len(xs)
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):      # plans, arenas and packed blocks exist before the capture starts
                for x in g_xs:
                    x.grad = None
                self(g_xs, g_xt)
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        for x in g_xs:
            x.grad = None
        if self._want_master and self._flat_master is None:
            self._flat_master = torch.zeros_like(self.flat_grad)
        try:   # the static inputs' AccumulateGrad nodes were created on another stream than the capture stream
            torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
        except AttributeError:
            pass
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):   # the stream the warm-up ran on (autograd leaf streams match)
            out = self(g_xs, g_xt)
            if self._flat_master is not None:
                # double-buffered capture: every graph leaves the averaged gradient in the SAME buffer (2.8 MB copy),
                # which is what the parameters' .grad view, whichever graph ran last
                self._flat_master.copy_(self.flat_grad)
        return {"flat": flat, "xs": g_xs, "xt": g_xt, "graph": graph, "out": out}

    def capture(self, student_inputs, teacher_inputs, warmup=3, double_buffer=False):
        """Capture one full step (teacher forwards on their side streams, student forward, MTA, backward, gradient
        all-reduce) into a CUDA graph over static device copies of the inputs.  The step is ~400 kernel launches of a
        few microseconds each: replaying it as one graph takes the host (and any driver contention, e.g. a clock
        monitor) out of the critical path.  Returns self; use replay().

        The graph keeps the BatchNorm modes of the student's layers as they were at capture time (frozen BatchNorm:
        layers in eval() inside the train-mode student); after switching a layer between train() and eval(), call
        capture() again — replays do not check the modes.

        `double_buffer=True` captures the step TWICE over two static input sets: prefetch() fills the set the running
        graph does not read and replay_prefetched() replays that set's graph, so the pipelined feed needs no
        staging-to-static copy (2 x 236 MB of HBM traffic per step at B = 32).  Both graphs leave the averaged gradient
        in one buffer (`flat_grad`, viewed by every parameter's .grad)."""
        self._flat_master, self._want_master = None, bool(double_buffer)
        self._sets = [self._capture_set(student_inputs, teacher_inputs, warmup)]
        if double_buffer:
            self._sets.append(self._capture_set(student_inputs, teacher_inputs, warmup))
            flat = self.flat_grad
            for p in self.student.parameters():
                if p.requires_grad and p.grad is not None:
                    off = p.grad.storage_offset() - flat.storage_offset()
                    p.grad = self._flat_master[off:off + p.grad.numel()].view(p.grad.shape)
            self.flat_grad = self._flat_master
        self._cur = 0
        self._bind(0)
        self._stage_xs = None
        self._fill = 0
        return self

    def _bind(self, k):
        """The legacy single-set attribute names follow the set whose graph ran last."""
        st = self._sets[k]
        self._cur = k
        self._flat_static, self._g_xs, self._g_xt, self._graph, self._g_out = st["flat"], st["xs"], st["xt"], st["graph"], st["out"]

    def replay(self, student_inputs=None, teacher_inputs=None):
        """Copy new inputs (host or device tensors; pinned host memory makes the copies asynchronous) into the static
        buffers and replay the captured step.  Returns the static [n_teachers, n_levels] loss tensor; the student's
        parameter gradients are in `flat_grad` / `.grad`, input gradients in `graph_inputs()[i].grad`."""
        if getattr(self, "_graph", None) is None:
            raise RuntimeError("DistillStep.replay() needs capture() first")
        if student_inputs is not None:
            for d, x in zip(self._g_xs, student_inputs):
                d.detach().copy_(x, non_blocking=True)
        if teacher_inputs is not None:
            for ds, xs in zip(self._g_xt, teacher_inputs):
                for d, x in zip(ds, xs):
                    d.copy_(x, non_blocking=True)
        self._graph.replay()
        self._after_replay()
        return self._g_out

    def _after_replay(self):
        """A replay updates running statistics (and, with an optimizer, the parameters) on the device only: bump the cells'
        state epoch so that eval-mode plans of the student re-fold their packed blocks on next use."""
        mark_state_changed(list(self.student) if isinstance(self.student, BiFPNStack) else [self.student])

    # ---- pipelined input feed for replay(): the host->device copy of step i+1 overlaps the replay of step i -----------
    def prefetch(self, student_inputs, teacher_inputs):
        """Start copying the NEXT step's inputs (host tensors, ideally pinned) into a device input set on a side stream:
        a staging set (single-buffered capture) or the static set of the graph that is not running (double_buffer).
        The copy waits until the set's previous consumer is done, so one call per step is safe; it never blocks the host
        for pinned inputs."""
        if getattr(self, "_graph", None) is None:
            raise RuntimeError("DistillStep.prefetch() needs capture() first")
        dev = self.device
        double = len(self._sets) == 2
        if getattr(self, "_stage_xs", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._ev_ready = [torch.cuda.Event(), torch.cuda.Event()]
            self._ev_consumed = [torch.cuda.Event(), torch.cuda.Event()]
            for e in self._ev_consumed:
                e.record(torch.cuda.current_stream(dev))
            if double:
                self._stage_xs = True
            else:
                self._flat_stage, views = _flat_channels_last([x.detach() for x in self._g_xs] + [x for xs in self._g_xt for x in xs], dev)
                ns = len(self._g_xs)
                self._stage_xs, self._stage_xt, k = views[:ns], [], ns
                for xs in self._g_xt:
                    self._stage_xt.append(views[k:k + len(xs)])
                    k += len(xs)
        if double:
            k = self._fill
            dst_xs, dst_xt = [x.detach() for x in self._sets[k]["xs"]], self._sets[k]["xt"]
        else:
            k = 0
            dst_xs, dst_xt = self._stage_xs, self._stage_xt
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._ev_consumed[k])
            for d, x in zip(dst_xs, student_inputs):
                d.copy_(x, non_blocking=True)
            for ds, xs in zip(dst_xt, teacher_inputs):
                for d, x in zip(ds, xs):
                    d.copy_(x, non_blocking=True)
            self._ev_ready[k].record(self._copy_stream)
        self._pending = k
        if double:
            self._fill ^= 1
        self._prefetched = True

    def replay_prefetched(self):
        """Replay the captured step on the inputs of the last prefetch(): waits for that copy, then either moves the staging
        set into the graph's static inputs (device-to-device) and replays, or — double_buffer — replays the graph that was
        captured over the set the copy went into."""
        if not getattr(self, "_prefetched", False):
            raise RuntimeError("DistillStep.replay_prefetched() needs prefetch() first")
        cur = torch.cuda.current_stream(self.device)
        k = self._pending
        cur.wait_event(self._ev_ready[k])
        if len(self._sets) == 2:
            self._bind(k)
            self._graph.replay()
            self._ev_consumed[k].record(cur)     # the first-cell projections' backward reads the inputs at the very end
        else:
            with torch.no_grad():
                self._flat_static.copy_(self._flat_stage)       # one copy: both sets share the flat layout
            self._ev_consumed[k].record(cur)
            self._graph.replay()
        self._prefetched = False
        self._after_replay()
        return self._g_out

    def graph_inputs(self):
        return self._g_xs


def lockstep_detection_forward(student, teachers, student_feats, teacher_feats):
    """YetAnotherEfficientDet.forward behind the backbone (src/YetAnotherEfficientDet.py:667-675: features = bifpn(p3, p4, p5);
    regression = regressor(features); classification = classifier(features)) for the student AND its frozen teachers in
    lockstep: three mmd_bifpn_run_multi calls (stacks, regressors, classifiers) instead of 3 x (1 + n_teachers) op lists, the
    same node of every network sharing a launch.  `student` / every teacher: a module with `.bifpn` (BiFPNStack),
    `.regressor`, `.classifier` (mm_distillnet_b200 modules, e.g. a patched YetAnotherEfficientDet); `student_feats` /
    `teacher_feats[i]`: that network's backbone features (C3, C4, C5).  At most 3 teachers, bf16, equal batch sizes.
    Returns [(classification, regression, features)] — student first; the teachers' entries are computed under no_grad in
    whatever mode the modules are in (eval), the student's carry their autograd nodes."""
    nets = [student] + list(teachers)
    feats = [tuple(student_feats)] + [tuple(f) for f in teacher_feats]
    if len(nets) > 4 or len(nets) != len(feats):
        raise ValueError("lockstep_detection_forward: one student + at most 3 teachers, one feature tuple each")
    stacks = forward_multi([(n.bifpn, f) for n, f in zip(nets, feats)])
    pyramids = [stacks[0]] + [tuple(t.detach() for t in o) for o in stacks[1:]]
    regs = forward_multi_heads([(n.regressor, p) for n, p in zip(nets, pyramids)])
    clss = forward_multi_heads([(n.classifier, p) for n, p in zip(nets, pyramids)])
    return [(c[0], r[0], f) for c, r, f in zip(clss, regs, pyramids)]
