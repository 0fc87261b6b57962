"""Training engine for the sequential 3x3-conv CNNs on the hand-written sm_100a kernels.

Replaces Keras' ``model.fit`` compute path (FLPyfhelin.py:118-136, :193) for the medical CNN:

  input     preprocess_u8 (uint8 -> bf16 NHWC [P,16], 1/255, Philox affine augmentation; layer-1 input
            carries pixels w, w+1, w+2 in its channels) into one of two X0 slots — the trainer stages
            batch i+1 on a side stream while step i runs
  forward   6 x conv_fwd_pool  (TMA-fed tcgen05 tap GEMMs, bias + ReLU + 2x2 max-pool + 3-bit
                                arg-max/active code fused in the TMEM epilogue; only pooled tensors
                                reach HBM; layer 1 on the pair-row variant: the whole pooling window
                                in one TMEM lane)
            head_forward_backward (Dense 128-64-C + softmax CE, forward AND backward, one launch on a
                                   cluster of 8 CTAs)
  backward  unpool_relu / conv_dgrad chain on the main stream (layers 6..2),
            conv_wgrad (tcgen05, MN-major operands, split-K partials summed in a fixed order) on a side stream,
            layer 1: wgrad0_gather straight from the pooled gradient (no un-pool, no dY tensor): four
                     masked GEMMs on the tensor cores (wgrad0_mma.cu), FP32-pipe gather as the fallback
  update    conv_grad_finalize + Adam + conv_weight_relayout: layers 2..6 and the head on the side
            stream under the layer-1 kernel, the 896 layer-1 parameters in the tail (``opt`` hooks)

All buffers are allocated once; a step is CUDA-graph capturable (one graph per input slot); every
kernel uses programmatic dependent launch (csrc/nn/launch.cuh).
"""
from __future__ import annotations

import os

import math
from typing import List, Optional

import torch
import torch.nn.functional as F

from .. import _ext
from ..config import FLConfig
from ..models.pack import ParamPack


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


class MedCNNEngine:
    def __init__(self, model, pack: ParamPack, cfg: FLConfig, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("the tcgen05 engine needs a CUDA device (sm_100a)")
        self.ops = _ext.ops()
        self.ops.set_head_cluster(0 if os.environ.get("HEFL_HEAD_CLUSTER", "1") == "0" else 1)
        self.ops.set_pdl(0 if os.environ.get("HEFL_PDL", "1") == "0" else 1)   # programmatic dependent launch
        self.model, self.pack, self.cfg, self.device = model, pack, cfg, device
        B, S = cfg.batch_size, cfg.image_size
        if cfg.in_channels != 3:
            raise ValueError("engine expects 3-channel uint8 images")
        self.B = B
        convs = list(model.convs)
        self.n = len(convs)
        offs = {k: o for k, _, o, _ in pack.entries}
        keys = [k for k in pack.keras_order_keys()]
        conv_keys = [(f"c_{2 * i}_0", f"c_{2 * i}_1") for i in range(self.n)]
        self.H: List[int] = []
        self.Ci: List[int] = []
        self.CK: List[int] = []
        self.Co: List[int] = []
        h = S
        for i, c in enumerate(convs):
            ci, co = c.in_channels, c.out_channels
            ck = 16 if i == 0 else ci
            if ck not in (16, 32, 64) or co not in (32, 64, 128):
                raise ValueError(f"unsupported conv shape ({ci}->{co}) for the tcgen05 engine")
            self.H.append(h)
            self.Ci.append(ci)
            self.CK.append(ck)
            self.Co.append(co)
            h = (h - 2) // 2
        self.H.append(h)                 # feature map side
        # layer-1 input carries pixels (w, w+1, w+2) in its 16 channels: 3 tap-GEMMs instead of 9 (conv_tcgen05.cu TS=1)
        self.spack0 = (os.environ.get("HEFL_SPACK0", "1") != "0" and self.Ci[0] == 3 and self.CK[0] == 16
                       and self.Co[0] == 32)
        # un-pool inside the dgrad epilogue: correct (bit-exact test) but measured 10 us/step SLOWER than the
        # separate un-pool kernels (the epilogue is issue-bound; 4x the stores), so off by default
        # pair-row forward kernel (both columns of a pooling window in one TMEM lane, conv_tcgen05.cu G1b): on by
        # default for layer 1, where it reads the same s-packed input and issues the same three MMAs per accumulator
        # as the tap-GEMM forward (bit-identical outputs, tests). On the small layers it is slower (one 128-window
        # tile per pooled row: 20.3 vs 16.8 us, 16.2 vs 11.6 us), so HEFL_FWD_PAIR=all is only for experiments.
        mode = os.environ.get("HEFL_FWD_PAIR", "1")
        self.fwd_pair = {"0": 0, "1": 1, "all": self.n}.get(mode, 0)      # number of leading layers that may use it
        self.fuse_unpool = os.environ.get("HEFL_FUSE_UNPOOL", "0") != "0"
        self.fuse_from = int(os.environ.get("HEFL_FUSE_UNPOOL_FROM", "0"))     # fuse only into layers >= this index
        # layer-1 weight gradient by gather from the pooled gradient (csrc/nn/wgrad_gather.cu)
        self.gather_wgrad0 = (os.environ.get("HEFL_GATHER_WGRAD0", "1") != "0" and self.Co[0] == 32
                              and self.CK[0] == 16 and self.H[0] <= 256)
        bf = dict(dtype=torch.bfloat16, device=device)
        self.P = [B * self.H[l] * self.H[l] for l in range(self.n + 1)]
        # activations / gradients (all NHWC bf16 viewed as [pixels, channels])
        # layer-1 input with 8 pixels of slack: its wgrad reads 4-pixel windows (overlapping TMA rows)
        # two copies: batch i+1 is pre-processed into the other slot while step i trains (fl/trainer.py)
        self._x0_bufs = [torch.zeros(self.P[0] + 8, 16, **bf) for _ in range(2)]
        self.X0 = [b[: self.P[0]] for b in self._x0_bufs]
        self._x0_base = self._x0_bufs[0]
        self.X = [self.X0[0]]
        self.amax, self.dY, self.gX = [], [], [None]
        for l in range(self.n):
            hp = self.H[l + 1]
            self.X.append(torch.zeros(B * hp * hp, self.Co[l], **bf))
            self.amax.append(torch.zeros(B * hp * hp, self.Co[l], dtype=torch.uint8, device=device))
            # layer 1 normally takes the gather path (no conv-grid gradient at all): allocate lazily
            self.dY.append(None if l == 0 else torch.zeros(self.P[l], self.Co[l], **bf))
            self.gX.append(torch.zeros(B * hp * hp, self.Co[l], **bf))
        # weights
        wf_off, wd_off, dw_off = [0], [0], [0]
        for l in range(self.n):
            wf_off.append(wf_off[-1] + 9 * self.Co[l] * self.CK[l])
            wd_off.append(wd_off[-1] + 9 * self.Ci[l] * self.Co[l])
            dw_off.append(dw_off[-1] + (9 * self.CK[l] + 1) * self.Co[l])
        self.wf_off, self.wd_off, self.dw_off = wf_off, wd_off, dw_off
        self.Wf = torch.zeros(wf_off[-1], **bf)
        self.Wd = torch.zeros(wd_off[-1], **bf)
        self.dW32 = torch.zeros(dw_off[-1], dtype=torch.float32, device=device)
        self.shadow = torch.zeros(pack.n_trainable, **bf)
        rows = []
        self.b_off = []
        for l, (kw, kb) in enumerate(conv_keys):
            rows.append([self.Ci[l], self.CK[l], self.Co[l], offs[kw], offs[kb], wf_off[l], wd_off[l], dw_off[l]])
            self.b_off.append(offs[kb])
        self.table = torch.tensor(rows, dtype=torch.int64)
        self.bias = [pack.flat[self.b_off[l]: self.b_off[l] + self.Co[l]] for l in range(self.n)]
        # flat parameters [0, p0) belong to layer 1 (weights then bias come first in the pack)
        self.p0 = max(offs[conv_keys[0][0]] + 9 * self.Ci[0] * self.Co[0], self.b_off[0] + self.Co[0])
        if self.n > 1 and not (self.p0 <= offs[conv_keys[1][0]] and self.p0 <= self.b_off[1]):
            self.p0 = 0          # unexpected parameter order: never split the update
        # dense head: fused kernels when it is the reference's 3-layer shape, else PyTorch autograd
        fcs = list(model.fcs)
        self.fused_head = len(fcs) == 3 and B <= 32 and B % 2 == 0
        if self.fused_head:
            nfc = self.n * 2 + 1
            self.head_offs = []
            for i in range(3):
                self.head_offs += [offs[f"c_{nfc + i}_0"], offs[f"c_{nfc + i}_1"]]
            self.F, self.H1, self.H2, self.C = fcs[0].in_features, fcs[0].out_features, fcs[1].out_features, fcs[2].out_features
            self.h1_buf = torch.zeros(B * self.H1, dtype=torch.float32, device=device)
            self.dh1_buf = torch.zeros(B * (self.H1 + self.H2), dtype=torch.float32, device=device)
            self.dfeat = torch.zeros(B, self.F, **bf)
        # one-launch parameter update needs the fused head (it owns the step increment) and the dense
        # parameters as one contiguous tail of the flat buffer
        self.dense_off = min(self.head_offs) if self.fused_head else 0
        # measured: 43 us fused (scattered m/v/flat accesses) vs 24 us for finalize+Adam+relayout -> off by default
        self.fused_step = os.environ.get("HEFL_FUSED_STEP", "0") == "1" and self.fused_head
        self.theta = torch.zeros(B, 2, 3, dtype=torch.float32, device=device)
        self.aug_seed = (cfg.seed * 2654435761 + 12345) & 0x7FFFFFFFFFFFFFFF or 1
        self.prep_count = 0          # augmented batches pre-processed so far (keys the in-kernel Philox draw)
        # weight gradients run on a side stream, concurrently with the dgrad / un-pool chain
        self.side = torch.cuda.Stream(device)
        self.two_streams = True
        self.step_ref: Optional[torch.Tensor] = None     # device step counter (set by the trainer)
        self.after_restore()

    # ------------------------------------------------------------------ weights
    def after_update(self) -> None:
        """Called after Adam wrote the bf16 shadow: rebuild the tensor-core weight layouts."""
        self.ops.conv_weight_relayout(self.shadow, self.table, self.Wf, self.Wd, 0, -1, self.spack0)

    def after_restore(self) -> None:
        self.shadow.copy_(self.pack.trainable())
        self.after_update()

    def _wf(self, l):
        return self.Wf[self.wf_off[l]: self.wf_off[l + 1]]

    def _wd(self, l):
        return self.Wd[self.wd_off[l]: self.wd_off[l + 1]]

    def _dw(self, l):
        return self.dW32[self.dw_off[l]: self.dw_off[l + 1]]

    # ------------------------------------------------------------------ forward
    def _make_theta(self, shear=0.2, zoom=0.2) -> torch.Tensor:
        B, dev = self.B, self.device
        r = torch.rand(B, 4, device=dev)
        sh = (r[:, 0] * 2 - 1) * shear * (math.pi / 180.0)
        zx = 1.0 + (r[:, 1] * 2 - 1) * zoom
        zy = 1.0 + (r[:, 2] * 2 - 1) * zoom
        flip = torch.where(r[:, 3] < 0.5, -1.0, 1.0)
        th = self.theta
        th.zero_()
        th[:, 0, 0] = zx * flip
        th[:, 0, 1] = -torch.sin(sh) * zx
        th[:, 1, 1] = torch.cos(sh) * zy
        return th

    def preprocess(self, x_u8: torch.Tensor, slot: int, train: bool, augment: bool) -> None:
        """uint8 NHWC batch -> bf16 [P,16] layer-1 input of ``slot`` (1/255 rescale + Keras-style random
        affine, FLPyfhelin.py:80-86). Augmentation parameters are drawn inside the kernel from Philox
        keyed by (seed, number of augmented batches so far, sample): reproducible and independent of
        which stream or slot the batch is staged on."""
        seed = 0
        if train and augment:
            seed = (self.aug_seed + 0x9E3779B97F4A7C15 * (self.prep_count + 1)) & 0x7FFFFFFFFFFFFFFF or 1
            self.prep_count += 1
        self.ops.preprocess_u8(x_u8, None, self.X0[slot], seed, None, self.spack0)

    def forward_convs(self, slot: int, train: bool) -> torch.Tensor:
        x = self.X0[slot]
        for l in range(self.n):
            h = self.H[l]
            if l < self.fwd_pair and h % 2 == 0 and (h - 2) // 2 <= 128 and self.CK[l] <= 32 and self.Co[l] <= 64:
                self.ops.conv_fwd_pool_pair(x if l else self._x0_bufs[slot], self._wf(l), self.bias[l], self.X[l + 1],
                                            self.amax[l] if train else None, self.B, h, h, self.CK[l], self.Co[l],
                                            self.spack0 and l == 0)
                x = self.X[l + 1]
                continue
            self.ops.conv_fwd_pool(x, self._wf(l), self.bias[l], self.X[l + 1],
                                   self.amax[l] if train else None, self.B, h, h, self.CK[l], self.Co[l],
                                   self.spack0 and l == 0)
            x = self.X[l + 1]
        return self.X[self.n]

    def features(self, x_u8: torch.Tensor, train: bool, augment: bool, slot: int = 0) -> torch.Tensor:
        self.preprocess(x_u8, slot, train, augment)
        return self.forward_convs(slot, train)

    def _head(self, feat: torch.Tensor) -> torch.Tensor:
        x = feat
        fcs = self.model.fcs
        for fc in fcs[:-1]:
            x = F.relu(fc(x))
        return fcs[-1](x)

    # ------------------------------------------------------------------ steps
    def train_step(self, x_u8: torch.Tensor, y: torch.Tensor, out: torch.Tensor, augment: bool = True, opt=None) -> None:
        self.preprocess(x_u8, 0, True, augment)
        self.train_step_staged(0, y, out, opt)

    def train_step_staged(self, slot: int, y: torch.Tensor, out: torch.Tensor, opt=None) -> None:
        """Forward + backward on the already pre-processed batch in ``slot`` (CUDA-graph body).

        ``opt`` (optional) applies the parameter update: ``opt.bump()`` advances the step counter and
        ``opt.apply(lo, hi)`` runs Adam on flat parameters [lo, hi). With two streams, everything but
        layer 1 is updated on the side stream while layer 1's weight-gradient kernel still runs; only
        the 896 layer-1 parameters are left for the tail of the step."""
        feat_bf = self.forward_convs(slot, True)
        if self.fused_head:
            self.ops.head_forward_backward(feat_bf, self.pack.flat, self.pack.grad, self.head_offs, y, self.dfeat,
                                           self.h1_buf, self.dh1_buf, out, self.step_ref if self.fused_step else None,
                                           self.B, self.F, self.H1, self.H2, self.C, True)
            g = self.dfeat.view_as(feat_bf)
        else:
            feat = feat_bf.view(self.B, -1).float().requires_grad_(True)
            logits = self._head(feat)
            loss = F.cross_entropy(logits, y)
            loss.backward()
            out[0] = loss.detach()
            out[1] = (logits.argmax(1) == y).sum()
            g = feat.grad.to(torch.bfloat16).view_as(feat_bf).contiguous()
        main = torch.cuda.current_stream(self.device)
        split = False
        dy_ready = False
        for l in range(self.n - 1, -1, -1):
            h = self.H[l]
            if l == 0 and self.gather_wgrad0:
                if opt is not None and self.two_streams and not self.fused_step and self.n > 1 and self.p0 > 0:
                    split = True
                    ev = torch.cuda.Event()
                    ev.record(main)                     # dgrad of layer 2 (last reader of Wd) is enqueued
                    with torch.cuda.stream(self.side):
                        self.side.wait_event(ev)
                        opt.bump()
                        self.ops.conv_grad_finalize(self.dW32, self.table, self.pack.grad, 1, self.n)
                        opt.apply(self.p0, self.pack.n_trainable)
                        self.ops.conv_weight_relayout(self.shadow, self.table, self.Wf, self.Wd, 1, self.n)
                # 3-channel layer: weight gradient gathered straight from the pooled gradient
                self.ops.wgrad0_gather(self._x0_bufs[slot], g, self.amax[0], self._dw(0), self.B, h, h, self.spack0)
                break
            xin = self.X0[slot] if l == 0 else self.X[l]
            if self.dY[l] is None:
                self.dY[l] = torch.zeros(self.P[l], self.Co[l], dtype=torch.bfloat16, device=self.device)
            if not dy_ready:
                self.ops.unpool_relu(g, self.amax[l], self.X[l + 1], self.dY[l], self.B, h, h, self.Co[l])
            dy_ready = False
            if self.two_streams and l > 0:
                # wgrad(l) only needs X[l] and dY[l]; dgrad(l) -> unpool(l-1) -> ... proceeds meanwhile
                self.side.wait_stream(main)
                with torch.cuda.stream(self.side):
                    self.ops.conv_wgrad(xin, self.dY[l], self._dw(l), self.B, h, h, self.CK[l], self.Co[l])
            else:
                self.ops.conv_wgrad(xin, self.dY[l], self._dw(l), self.B, h, h, self.CK[l], self.Co[l])
            if l > 0:
                # dgrad(l) scatters its result straight into the conv-grid gradient of layer l-1 (un-pool fused
                # into the epilogue) unless that layer takes the gather path, which wants the pooled gradient
                if self.fuse_unpool and l - 1 >= self.fuse_from and not (l == 1 and self.gather_wgrad0):
                    if self.dY[l - 1] is None:
                        self.dY[l - 1] = torch.zeros(self.P[l - 1], self.Co[l - 1], dtype=torch.bfloat16, device=self.device)
                    self.ops.conv_dgrad(self.dY[l], self._wd(l), self.dY[l - 1], self.B, h, h, self.Co[l], self.Ci[l],
                                        self.amax[l - 1], self.H[l - 1])
                    dy_ready = True
                else:
                    self.ops.conv_dgrad(self.dY[l], self._wd(l), self.gX[l], self.B, h, h, self.Co[l], self.Ci[l])
                    g = self.gX[l]
        if self.two_streams:
            main.wait_stream(self.side)
        if self.fused_step:
            return
        if opt is None:
            self.ops.conv_grad_finalize(self.dW32, self.table, self.pack.grad)
        elif split:
            self.ops.conv_grad_finalize(self.dW32, self.table, self.pack.grad, 0, 1)
            opt.apply(0, self.p0)
            self.ops.conv_weight_relayout(self.shadow, self.table, self.Wf, self.Wd, 0, 1, self.spack0)
        else:
            opt.bump()
            self.ops.conv_grad_finalize(self.dW32, self.table, self.pack.grad)
            opt.apply(0, self.pack.n_trainable)
            self.after_update()

    def fused_update(self, m: torch.Tensor, v: torch.Tensor, step: torch.Tensor, lr_scale: torch.Tensor, cfg) -> None:
        """finalize + Adam + bf16 shadow + tensor-core weight layouts + dW32 clear, one launch."""
        self.ops.fused_update(self.dW32, self.table, self.pack.flat, self.pack.grad, m, v, self.shadow, self.Wf, self.Wd,
                              step, lr_scale, cfg.lr, cfg.lr_decay, 0.9, 0.999, 1e-7, self.dense_off,
                              self.pack.n_trainable)
        if self.spack0:
            self.ops.conv_weight_relayout(self.shadow, self.table, self.Wf, self.Wd, 0, 1, True)

    def eval_step(self, x_u8: torch.Tensor, y: torch.Tensor, out: torch.Tensor) -> None:
        self.preprocess(x_u8, 0, False, False)
        self.eval_step_staged(0, y, out)

    def eval_step_staged(self, slot: int, y: torch.Tensor, out: torch.Tensor) -> None:
        feat_bf = self.forward_convs(slot, False)
        if self.fused_head:
            self.ops.head_forward_backward(feat_bf, self.pack.flat, self.pack.grad, self.head_offs, y, self.dfeat,
                                           self.h1_buf, self.dh1_buf, out, None, self.B, self.F, self.H1, self.H2, self.C, False)
            return
        feat = feat_bf.view(self.B, -1).float()
        logits = self._head(feat)
        out[0] = F.cross_entropy(logits, y)
        out[1] = (logits.argmax(1) == y).sum()
