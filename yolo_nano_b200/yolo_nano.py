"""Drop-in for the reference detector class `models.yolo_nano.YOLONano`.

Same constructor arguments, same mutable attributes, same `forward(x) ->
(bboxes, scores, cls_inds)` contract and the same `state_dict` layout as
`/root/reference/models/yolo_nano.py:12-376`; but `forward` never runs a torch
operator: the `nn.Conv2d` / `nn.BatchNorm2d` objects below are parameter
containers only (so `state_dict`, `load_state_dict`, `deepcopy`, `parameters()`
and the reference's own `fuse_conv_bn` keep working), and the computation is
done by the sm_100a engine behind `include/yolonano_b200.h`.

Batch semantics: the reference's eval branch decodes image 0 only
(`models/yolo_nano.py:365-367`).  `forward` keeps exactly that contract;
`detect(x)` is the batched extension (one result triple per image, each identical
to calling the reference once per image).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .engine import Engine, EngineError
from .topology import (ACT_LEAKY, STAGE_CHANNELS, STAGE_REPEATS, NECK_CHANNELS, STRIDES,
                       conv_table, head_channels)


class _Container(nn.Module):
    """Holds parameters under reference names; computing through it is a bug."""

    def forward(self, *a, **k):  # pragma: no cover - guard
        raise RuntimeError("parameter container: the forward path runs in the CUDA engine, "
                           "there is no PyTorch fallback")


class Conv(_Container):
    """Parameter layout of the reference `Conv` (utils/modules.py:8-18):
    `convs.0` = Conv2d(with bias), `convs.1` = BatchNorm2d, `convs.2` = LeakyReLU(0.1)."""

    def __init__(self, c1, c2, k, s=1, p=0, d=1, g=1, leaky=True):
        super().__init__()
        self.convs = nn.Sequential(
            nn.Conv2d(c1, c2, k, stride=s, padding=p, dilation=d, groups=g),
            nn.BatchNorm2d(c2),
            nn.LeakyReLU(0.1, inplace=True) if leaky else nn.Identity(),
        )


def _pw(cin, cout):
    return nn.Conv2d(cin, cout, kernel_size=1, stride=1, padding=0, bias=False)


def _dw(c, stride):
    return nn.Conv2d(c, c, kernel_size=3, stride=stride, padding=1, bias=False, groups=c)


class ShuffleV2Block(_Container):
    """Parameter layout of one ShuffleNetV2 unit (backbone/shufflenetv2.py:31-67)."""

    def __init__(self, inp, oup, stride):
        super().__init__()
        if stride not in (1, 2):
            raise ValueError("illegal stride value")
        half = oup // 2
        if stride == 1 and inp != 2 * half:
            raise ValueError("stride-1 unit needs inp == oup")
        self.stride = stride
        # registration order (branch1 before branch2) fixes both the state_dict order and
        # the RNG consumption order of the default initialisers
        self.branch1 = nn.Sequential() if stride == 1 else nn.Sequential(
            _dw(inp, stride), nn.BatchNorm2d(inp), _pw(inp, half), nn.BatchNorm2d(half),
            nn.ReLU(inplace=True))
        self.branch2 = nn.Sequential(
            _pw(inp if stride > 1 else half, half), nn.BatchNorm2d(half), nn.ReLU(inplace=True),
            _dw(half, stride), nn.BatchNorm2d(half),
            _pw(half, half), nn.BatchNorm2d(half), nn.ReLU(inplace=True))


class ShuffleNetV2(_Container):
    """Parameter layout + initialisation of the 1.0x backbone
    (backbone/shufflenetv2.py:81-154)."""

    def __init__(self, model_size="1.0x"):
        super().__init__()
        if model_size != "1.0x":
            raise NotImplementedError("only the 1.0x backbone is on the YOLO-Nano path")
        self.model_size = model_size
        self.stage_repeats = list(STAGE_REPEATS)
        c = STAGE_CHANNELS[0]
        self.conv1 = nn.Sequential(nn.Conv2d(3, c, 3, 2, 1, bias=False), nn.BatchNorm2d(c),
                                   nn.ReLU(inplace=True))
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1)
        for idx, (rep, cout) in enumerate(zip(STAGE_REPEATS, STAGE_CHANNELS[1:])):
            units = [ShuffleV2Block(c, cout, 2)] + [ShuffleV2Block(cout, cout, 1) for _ in range(rep - 1)]
            setattr(self, f"stage{idx + 2}", nn.Sequential(*units))
            c = cout
        self._initialize_weights()

    def _initialize_weights(self):
        # same draws, in the same module order, as backbone/shufflenetv2.py:131-154:
        # conv ~ N(0, 1/weight.shape[1]), BN weight 1 / bias 1e-4 / running_mean 0
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.normal_(m.weight, 0, 1.0 / m.weight.shape[1])
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0.0001)
                nn.init.constant_(m.running_mean, 0)


def _head(num_out):
    n = NECK_CHANNELS
    return nn.Sequential(Conv(n, n, k=3, p=1, g=n), Conv(n, n, k=1),
                         Conv(n, n, k=3, p=1, g=n), Conv(n, n, k=1),
                         nn.Conv2d(n, num_out, 1))


class YOLONano(nn.Module):
    """B200-native YOLO-Nano-1.0x detector, API-compatible with the reference class."""

    def __init__(self, device, input_size=None, num_classes=20, trainable=False,
                 conf_thresh=0.001, nms_thresh=0.50, anchor_size=None, backbone="1.0x",
                 diou_nms=False, gemm_mode: Optional[int] = None):
        super().__init__()
        self.device = device
        self.input_size = input_size
        self.num_classes = num_classes
        self.trainable = trainable
        self.conf_thresh = conf_thresh
        self.nms_thresh = nms_thresh
        self.diou_nms = bool(diou_nms)
        self.bk = backbone
        self.stride = list(STRIDES)
        self.anchor_size = torch.tensor(anchor_size).view(3, len(anchor_size) // 3, 2)
        self.num_anchors = self.anchor_size.size(1)
        if self.num_anchors != 3:
            raise NotImplementedError("the engine is built for 3 anchors per level")
        self.gemm_mode = _lib.GEMM_TC_3XTF32 if gemm_mode is None else int(gemm_mode)

        if self.bk != "1.0x":
            # the reference prints a message and calls exit(0) (models/yolo_nano.py:35-37)
            raise SystemExit("For YOLO-Nano, we only support <1.0x> as our backbone !!")
        print("Use backbone: shufflenetv2_1.0x")
        self.backbone = ShuffleNetV2(self.bk)
        c3, c4, c5 = STAGE_CHANNELS[1:]
        n = NECK_CHANNELS
        self.conv1x1_0 = Conv(c3, n, k=1)
        self.conv1x1_1 = Conv(c4, n, k=1)
        self.conv1x1_2 = Conv(c5, n, k=1)
        self.smooth_0 = Conv(n, n, k=3, p=1)
        self.smooth_1 = Conv(n, n, k=3, p=1)
        self.smooth_2 = Conv(n, n, k=3, p=1)
        self.smooth_3 = Conv(n, n, k=3, p=1)
        nout = head_channels(self.num_classes, self.num_anchors)
        self.head_det_1 = _head(nout)
        self.head_det_2 = _head(nout)
        self.head_det_3 = _head(nout)
        if self.trainable:
            self.init_bias()

        # engine state lives outside nn.Module bookkeeping (deepcopy / state_dict safe)
        object.__setattr__(self, "_engine", None)
        object.__setattr__(self, "_engine_key", None)
        object.__setattr__(self, "_weights_key", None)
        object.__setattr__(self, "_wt_cache", None)
        object.__setattr__(self, "_out_cache", None)
        object.__setattr__(self, "_train_step", None)

    # ---- reference API ---------------------------------------------------------------
    def init_bias(self):
        """Objectness-logit bias = -log(99) (models/yolo_nano.py:77-83)."""
        init_prob = 0.01
        bias_value = -torch.log(torch.tensor((1.0 - init_prob) / init_prob))
        for head in (self.head_det_1, self.head_det_2, self.head_det_3):
            nn.init.constant_(head[-1].bias[..., : self.num_anchors], bias_value)

    def set_grid(self, input_size):
        """models/yolo_nano.py:115-117.  The grid is analytic inside the kernels; this
        only records S (the engine re-plans its workspace lazily)."""
        self.input_size = input_size

    def create_grid(self, input_size):
        """Grid tensors of the reference (models/yolo_nano.py:86-112), built on demand for
        callers that inspect them; the engine does not use tables."""
        g, st, an = [], [], []
        for lvl, s in enumerate(self.stride):
            n = input_size // s
            ys, xs = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
            g.append(torch.stack([xs, ys], -1).float().view(1, n * n, 1, 2))
            st.append(torch.full((1, n * n, self.num_anchors, 2), float(s)))
            an.append(self.anchor_size[lvl].repeat(n * n, 1, 1))
        dev = self.device
        return (torch.cat(g, 1).to(dev), torch.cat(st, 1).to(dev), torch.cat(an, 0).to(dev).unsqueeze(0))

    @property
    def grid_cell(self):
        return self.create_grid(self.input_size)[0]

    @property
    def stride_tensor(self):
        return self.create_grid(self.input_size)[1]

    @property
    def all_anchors_wh(self):
        return self.create_grid(self.input_size)[2]

    # ---- weights -> engine -------------------------------------------------------------
    def fused_weights(self):
        """(W, b) per conv with BatchNorm folded exactly like utils/fuse_conv_bn.py:6-22.
        Works on the unfused module and after `fuse_conv_bn` (BN slots are Identity)."""
        out = {}
        with torch.no_grad():
            for spec in conv_table(self.num_classes, self.num_anchors):
                conv = self.get_submodule(spec.name)
                w = conv.weight
                b = conv.bias
                bn = self.get_submodule(spec.bn) if spec.bn is not None else None
                if isinstance(bn, nn.modules.batchnorm._BatchNorm):
                    if b is None:
                        b = torch.zeros_like(bn.running_mean)
                    factor = bn.weight / torch.sqrt(bn.running_var + bn.eps)
                    w = w * factor.reshape([conv.out_channels, 1, 1, 1])
                    b = (b - bn.running_mean) * factor + bn.bias
                elif b is None:
                    b = torch.zeros(conv.out_channels, dtype=w.dtype, device=w.device)
                out[spec.name] = (w, b)
        return out

    def _weight_tensors(self):
        """The 469 (154 after fuse_conv_bn) tensors the engine weights are derived from.  The list is cached
        together with every (`_modules` / `_parameters` / `_buffers` dict, key, object) slot of the module tree
        and rebuilt as soon as one slot holds another object: fuse_conv_bn replaces modules, and
        `load_state_dict(assign=True)` and dtype / device conversions put new tensor objects in place, whose
        changes the fingerprint of the old objects would never see.  The check is identity only (~30 us)."""
        c = self._wt_cache
        if c is None or not all(d.get(k) is v for d, k, v in c[0]):
            slots = [(d, k, v) for m in self.modules() for d in (m._modules, m._parameters, m._buffers)
                     for k, v in d.items() if v is not None]
            object.__setattr__(self, "_wt_cache", (slots, list(self.state_dict(keep_vars=True).values())))
        return self._wt_cache[1]

    def _weights_fingerprint(self):
        # (storage, in-place version) of every tensor: changes on load_state_dict / optimizer steps / .to()
        return tuple((t.data_ptr(), t._version) for t in self._weight_tensors())

    def mark_weights_dirty(self):
        """Force a re-pack of the engine weights on the next forward (for writers that bypass autograd's
        version counters, e.g. the fused ModelEMA / SGD kernels)."""
        object.__setattr__(self, "_weights_key", None)

    def _device(self) -> torch.device:
        p = next(self.parameters())
        return p.device

    def engine(self, batch: int = 1) -> Engine:
        """The engine for the current device / S / class count, with current weights."""
        dev = self._device()
        if dev.type != "cuda":
            raise EngineError("YOLONano (B200) needs its parameters on a CUDA device: "
                              "there is no CPU fallback")
        eng = self._engine
        key = (dev, self.num_classes, tuple(self.anchor_size.flatten().tolist()), self.gemm_mode)
        if eng is None or self._engine_key[:4] != key or self._engine_key[4] < batch:
            if eng is not None:
                eng.close()
            mb = max(batch, self._engine_key[4] if self._engine_key else 1)
            eng = Engine(dev, self.input_size, self.num_classes, self.anchor_size.view(-1, 2).tolist(),
                         self.conf_thresh, self.nms_thresh, self.diou_nms, self.gemm_mode, mb)
            object.__setattr__(self, "_engine", eng)
            object.__setattr__(self, "_engine_key", key + (mb,))
            object.__setattr__(self, "_weights_key", None)
        if eng.input_size != self.input_size:
            eng.set_grid(self.input_size)
        eng.set_thresholds(self.conf_thresh, self.nms_thresh, self.diou_nms)
        fp = self._weights_fingerprint()
        if fp != self._weights_key:
            eng.load_weights(self.fused_weights())
            object.__setattr__(self, "_weights_key", fp)
        return eng

    def __deepcopy__(self, memo):
        # ModelEMA deep-copies the model (utils/misc.py:70): the copy gets its own engine lazily
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_engine", "_engine_key", "_weights_key", "_wt_cache", "_out_cache", "_train_step"):
                object.__setattr__(new, k, None)
            else:
                object.__setattr__(new, k, copy.deepcopy(v, memo))
        return new

    # ---- the path ------------------------------------------------------------------------
    @torch.no_grad()
    def detect(self, x: torch.Tensor) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        """Batched extension: one (bboxes [K,4] f32, scores [K] f32, cls_inds [K] i64)
        triple per image, each what the reference returns for that image alone."""
        nb = int(x.shape[0])
        eng = self.engine(nb)
        # device outputs are reused between calls (same addresses -> the engine replays its CUDA graph)
        oc_ = self._out_cache
        if oc_ is None or oc_[0] is not eng or oc_[1] != (nb, eng.num_boxes):
            oc_ = (eng, (nb, eng.num_boxes), eng.alloc_outputs(nb))
            object.__setattr__(self, "_out_cache", oc_)
        boxes, scores, cls, counts = eng.forward_detect(x, oc_[2])
        counts_h = counts.cpu().numpy()                       # the one synchronising copy (the reference's .to('cpu'))
        kmax = int(counts_h.max()) if nb else 0
        # rows [0, max count) of every image: three copies per call, not three per image
        bh = boxes[:, :kmax].cpu().numpy()
        sh = scores[:, :kmax].cpu().numpy()
        ch = cls[:, :kmax].cpu().numpy()
        res = []
        for b in range(nb):
            k = int(counts_h[b])
            # owned, writable host arrays: callers rescale boxes in place
            # (evaluator/cocoapi_evaluator.py:85-87, test.py:133-135)
            res.append((np.array(bh[b, :k], dtype=np.float32, copy=True),
                        np.array(sh[b, :k], dtype=np.float32, copy=True),
                        ch[b, :k].astype(np.int64)))
        return res

    def detect_images(self, canvases, rects=None) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        """`detect` for uint8 BGR images [B,S,S,3] already resized / letterboxed to the grid size on the
        host (`rects` int32 [B,4] = x0, y0, w, h of the content; None = whole canvas): Normalize +
        ToTensor of the reference's ValTransforms (data/transforms.py:445-458) run on the device and
        the images cross PCIe as bytes.  Same results as `detect(ValTransforms(...)(img))`."""
        canvases = torch.as_tensor(canvases)
        if canvases.dtype != torch.uint8 or canvases.dim() != 4 or canvases.shape[-1] != 3:
            raise ValueError("detect_images wants uint8 [B,S,S,3]")
        b = canvases.shape[0]
        eng = self.engine(b)
        if rects is not None:
            rects = torch.as_tensor(rects, dtype=torch.int32).contiguous()
        out = eng.alloc_outputs(b, pinned_host=True)
        eng.submit_host_u8(0, canvases.contiguous(), out, rects)
        eng.wait_host(0)
        boxes, scores, cls, counts = out
        res = []
        for i in range(b):
            k = int(counts[i])
            res.append((np.array(boxes[i, :k].numpy(), dtype=np.float32, copy=True),
                        np.array(scores[i, :k].numpy(), dtype=np.float32, copy=True),
                        cls[i, :k].numpy().astype(np.int64)))
        return res

    def detect_raw_images(self, images) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        """The evaluators' per-image loop (evaluator/cocoapi_evaluator.py:70-87, vocapi_evaluator.py) for a list of
        ORIGINAL uint8 BGR images of any shapes: ValTransforms (letterbox resize + normalisation) on the device, the
        detector, and the inverse box mapping `bboxes = (bboxes - offset) / scale * [w, h, w, h]` on the NMS output —
        returns boxes in pixels of each original image."""
        nb = len(images)
        eng = self.engine(nb)
        x, maps = eng.preprocess_images(images)
        boxes, scores, cls, counts = eng.forward_detect(x)
        eng.map_boxes(boxes, counts, maps)
        counts_h = counts.cpu().numpy()
        kmax = int(counts_h.max()) if nb else 0
        bh, sh, ch = boxes[:, :kmax].cpu().numpy(), scores[:, :kmax].cpu().numpy(), cls[:, :kmax].cpu().numpy()
        return [(np.array(bh[b, :int(counts_h[b])], dtype=np.float32, copy=True),
                 np.array(sh[b, :int(counts_h[b])], dtype=np.float32, copy=True),
                 ch[b, :int(counts_h[b])].astype(np.int64)) for b in range(nb)]

    def evaluate_voc(self, images, gt, batch_size: int = 64, use_07_metric: bool = True, ovthresh: float = 0.5,
                     capacity: Optional[int] = None):
        """`VOCAPIEvaluator.evaluate` + `do_python_eval` (evaluator/vocapi_evaluator.py) on the device: `images` is an
        iterable of ORIGINAL uint8 BGR images, `gt` one (boxes [G,4], labels [G], difficult [G]) per image in
        voc_eval's coordinates.  Per batch: ValTransforms, detection, the inverse box mapping and the det-file lines
        stay on the device; the host waits once, for the APs.  Returns (aps float64 [C], mAP).  `capacity` bounds
        the detection lines (default: every anchor box of every image, which cannot overflow)."""
        from .voc_eval import VOCDetections
        if batch_size < 1:
            raise ValueError("batch_size must be positive")
        eng = self.engine(batch_size)
        if capacity is None:
            capacity = len(gt) * eng.num_boxes
        dets = VOCDetections(eng.device, self.num_classes, capacity)
        batch = []

        def run(batch):
            eng = self.engine(len(batch))
            x, maps = eng.preprocess_images(batch)
            boxes, scores, cls, counts = eng.forward_detect(x)
            eng.map_boxes(boxes, counts, maps)
            dets.add(boxes, scores, cls, counts)

        for im in images:
            batch.append(im)
            if len(batch) == batch_size:
                run(batch)
                batch = []
        if batch:
            run(batch)
        return dets.evaluate(gt, ovthresh=ovthresh, use_07_metric=use_07_metric)

    def forward(self, x, target=None):
        if self.trainable:
            # training branch (models/yolo_nano.py:333-358).  The returned losses are plain device scalars WITHOUT a
            # grad_fn — there is no autograd graph on this path.
            #   model.train():  BatchNorm on batch statistics; the SAME call also runs the backward chain through
            #     all 77 convolutions (train_step.TrainStep) and leaves d(sum of the four losses)/d(parameter) in
            #     `model.gradients` {name: tensor} — what train.py:229's `total_loss.backward()` leaves in `.grad`.
            #     `train_step.Trainer` is the loop body of train.py (SGD / all-reduce / EMA on top of this).
            #   model.eval():   running statistics folded into the convs; losses + `model.head_gradients`
            #     (d/d raw head maps) from the inference engine.
            if self.training:
                if target is None:
                    raise ValueError("trainable forward needs target [B, N, 11] (tools.multi_gt_creator)")
                from .train_step import TrainStep
                if self._train_step is None:
                    object.__setattr__(self, "_train_step", TrainStep(self))
                dev = self._device()
                losses, grads = self._train_step.forward_backward(
                    x.to(dev, torch.float32), target.to(dev, torch.float32))
                object.__setattr__(self, "gradients", grads)
                return losses[0], losses[1], losses[2], losses[3]
            if target is None:
                raise ValueError("trainable forward needs target [B, N, 11] (tools.multi_gt_creator)")
            eng = self.engine(int(x.shape[0]))
            dev = eng.device
            losses, self.head_gradients = eng.forward_train_loss(
                x.to(dev, torch.float32), target.to(dev, torch.float32).contiguous())
            return losses[0], losses[1], losses[2], losses[3]
        # eval: the reference decodes image 0 only (models/yolo_nano.py:365-367)
        return self.detect(x[:1])[0]
