"""CUDA-graph replay of the GMW training step (GMW/main.py:453-465) for fixed batch shapes.

At the reference's batch size (-b 8, README.md:74-79) the step is ~80 kernel launches of 10-80 us each: launch latency,
not arithmetic, bounds it.  Every entry point of libdcd_b200.so is capture-safe (stream-ordered, no allocation, no
synchronisation), so the whole forward + loss + backward is captured once into a torch.cuda.CUDAGraph and replayed with one
launch per step.  Gradients land in the model's parameter blobs' .grad exactly as in the eager step.

    step = GraphedGmwStep(model, batch=8, n=73)              # model: dcd_b200.GMW
    loss = step(kpts_2d, kpts_3d, pred_rot, gt_depth)        # == eager: compute_z -> model -> losses -> backward
    optimizer.step()

With cls_weight != 0 the step adds the correspondence loss (GMW/main.py:455-457), taken from GMW.transport_terms +
correspondence_loss instead of the [b,E,E] plan edge_P: the same gradients bit for bit as through edge_P, and no E x E
tensor but the Sinkhorn kernel K is allocated (not the plan, the loss's [b,E,E] temporaries or a dense dL/dP).  With
cls_weight == 0 the Sinkhorn branch does not run, whatever the model's with_edge_P says.
"""
from __future__ import annotations

import torch

from . import ops


class GraphedGmwStep:
    def __init__(self, model: "ops.GMW", batch: int, n: int = 73, cls_weight: float = 0.0, reg_weight: float = 1.0,
                 warmup: int = 3):
        p = model.params4
        if not p.is_cuda:
            raise RuntimeError("GraphedGmwStep needs the model on a CUDA device")
        dev = p.device
        self.model = model
        self.cls_weight, self.reg_weight = float(cls_weight), float(reg_weight)
        self.k2 = torch.zeros((batch, n, 2), device=dev)
        self.k3 = torch.zeros((batch, n, 3), device=dev)
        self.rot = torch.zeros((batch, 1), device=dev)
        self.gt = torch.zeros((batch,), device=dev)
        self.loss = None
        self.pred_depth = None
        self._graph = None
        self._warmup = warmup
        self._primed = False

    def _eager(self):
        model = self.model
        Z, idx = ops.compute_z(self.k2, self.k3, self.rot)
        if self.cls_weight != 0.0:
            w, terms = model.transport_terms(self.k2, self.k3)
        else:
            w, terms = model._edge_branch(None, self.k2, self.k3, model.params4, model.params6)
        reg, zsel = ops.compute_reg_loss(Z, w, self.gt, idx)
        loss = self.reg_weight * reg
        if terms is not None:
            loss = loss + self.cls_weight * ops.correspondence_loss(terms)
        loss.backward()
        return loss.detach(), zsel.detach()

    def _capture(self):
        model = self.model
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                            # warm-up off the capturing stream (allocator, lazy attributes)
            for _ in range(self._warmup):
                model.zero_grad(set_to_none=True)
                self._eager()
        torch.cuda.current_stream().wait_stream(s)
        model.zero_grad(set_to_none=True)                     # .grad is (re)allocated from the graph's private pool
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self.loss, self.pred_depth = self._eager()

    def __call__(self, kpts_2d, kpts_3d, pred_rot, gt_depth):
        self.k2.copy_(kpts_2d)
        self.k3.copy_(kpts_3d)
        self.rot.copy_(pred_rot.reshape(self.rot.shape))
        self.gt.copy_(gt_depth.reshape(self.gt.shape))
        if self._graph is None:
            self._capture()
        # (.grad was None at capture, so the captured backward ASSIGNS the static gradient tensors: nothing accumulates
        #  across replays; an optimizer may read / zero them freely, but must not set them to None)
        self._graph.replay()
        return self.loss
