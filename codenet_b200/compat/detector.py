"""Detector entry points mirror: lib/detectors/base_detector.py:20-155 and lib/detectors/ctdet.py:26-74.

`CtdetDetector(opt)` builds the network, quantises it, loads the checkpoint (`opt.load_model`, reference key space),
freezes the activation ranges and runs forward + decode through the compiled int8 engine.  `run()` returns the same
dict as the reference (`results` keyed by 1-based class id and the stage timers test.py prints, test.py:76-79).
Only what differs from the reference lives here: engine construction, process / process_u8, the device-side box transform,
run()'s multi-scale path (all test scales of an image in one engine batch, merge_outputs on the device: cdn_ctdet_merge) and
run_batch() (many raw frames per engine step, their warpAffine in one cdn_warp_affine_u8_batch launch per step, or for the
unquantised model one cdn_warp_affine_u8_f32_batch launch that also normalises).
pre_process, merge_outputs and run keep the reference's contract (same inputs, outputs and timer keys) in this package's own
decomposition (input_geometry / _Stages / group_by_class); INTEGRATION.md section 2 shows the patch for users who keep the reference's BaseDetector.
"""
import time
from types import SimpleNamespace

import numpy as np
import torch

from .nms import soft_nms
from .decode import ctdet_decode
from .quantize_model import quantize_shufflenetv2_dcn, freeze_ranges
from .shufflenetv2_dcn import PoseShuffleNetV2


def default_opt(**kw):
    """The fields of lib/opts.py that reach the hot path, with the reference's defaults for ctdet / shufflenetv2."""
    o = SimpleNamespace(
        gpus=[0], arch="shufflenetv2", heads={"hm": 20, "wh": 2, "reg": 2}, head_conv=64, num_classes=20,
        resume_quantize=True, w_bit=4, a_bit=8, wt_percentile=False, act_percentile=False, w2=False, maxpool=False,
        load_model="", mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225], test_scales=[1.0], fix_res=True,
        input_h=512, input_w=512, pad=31, down_ratio=4, flip_test=False, reg_offset=True, cat_spec_wh=False, K=100,
        nms=False, debug=0, offset_mode="bilinear", max_batch=1)
    o.__dict__.update(kw)
    return o


# ---- affine helpers (lib/utils/image.py:14-61) restated with numpy only --------------------------------------------
def _third_point(a, b):
    d = a - b
    return b + np.array([-d[1], d[0]], dtype=np.float32)


def _solve_affine(src, dst):
    """2x3 matrix mapping three src points to three dst points (what cv2.getAffineTransform computes)."""
    A = np.hstack([src.astype(np.float64), np.ones((3, 1))])
    return np.linalg.solve(A, dst.astype(np.float64)).T


def get_affine_transform(center, scale, rot, output_size, shift=np.array([0, 0], dtype=np.float32), inv=0):
    if not isinstance(scale, (np.ndarray, list)):
        scale = np.array([scale, scale], dtype=np.float32)
    scale = np.asarray(scale, dtype=np.float32)
    src_w, dst_w, dst_h = scale[0], output_size[0], output_size[1]
    rad = np.pi * rot / 180
    sn, cs = np.sin(rad), np.cos(rad)
    src_dir = np.array([-(src_w * -0.5) * sn, (src_w * -0.5) * cs], dtype=np.float32)
    dst_dir = np.array([0, dst_w * -0.5], np.float32)
    src = np.zeros((3, 2), np.float32); dst = np.zeros((3, 2), np.float32)
    src[0] = center + scale * shift
    src[1] = center + src_dir + scale * shift
    dst[0] = [dst_w * 0.5, dst_h * 0.5]
    dst[1] = np.array([dst_w * 0.5, dst_h * 0.5], np.float32) + dst_dir
    src[2] = _third_point(src[0], src[1]); dst[2] = _third_point(dst[0], dst[1])
    return _solve_affine(dst, src) if inv else _solve_affine(src, dst)


def transform_preds(coords, center, scale, output_size):
    t = get_affine_transform(center, scale, 0, output_size, inv=1)
    pts = np.concatenate([coords[:, 0:2].astype(np.float32), np.ones((coords.shape[0], 1), np.float32)], 1)
    return (pts.astype(np.float64) @ t.T)


def boxes_to_image_space(dets, center, scale, out_w, out_h):
    """Both corners of every box [N,6] through the inverse of the network-input affine (what ctdet_post_process,
    lib/utils/post_process.py:86-103, does corner by corner): one 2x3 matrix, one matrix product per corner set."""
    t = get_affine_transform(center, scale, 0, (out_w, out_h), inv=1)
    d = np.array(dets, dtype=np.float32, copy=True)
    corners = d[:, :4].reshape(-1, 2).astype(np.float32)
    homog = np.concatenate([corners, np.ones((corners.shape[0], 1), np.float32)], 1).astype(np.float64)
    d[:, :4] = (homog @ t.T).reshape(-1, 4)
    return d


def group_by_class(dets, num_classes):
    """[N,6] (x1,y1,x2,y2,score,class) -> {1-based class id: float32 [n,5]} in detection order."""
    cls = dets[:, 5].astype(np.int64)
    return {j + 1: np.ascontiguousarray(dets[cls == j, :5], dtype=np.float32).reshape(-1, 5) for j in range(num_classes)}


def ctdet_post_process(dets, c, s, h, w, num_classes):
    """Host restatement used by the tests (the detector itself transforms on the device): per image, boxes back to image
    coordinates and grouped per 1-based class."""
    return [group_by_class(boxes_to_image_space(dets[i], c[i], s[i], w, h), num_classes) for i in range(dets.shape[0])]


class _Stages:
    """Wall-clock accounting of run(): the keys test.py prints (test.py:76-79)."""
    KEYS = ("load", "pre", "net", "dec", "post", "merge")

    def __init__(self):
        self.t = dict.fromkeys(self.KEYS, 0.0)
        self.start = self.mark = time.time()

    def lap(self, key, now=None):
        now = time.time() if now is None else now
        self.t[key] += now - self.mark
        self.mark = now

    def result(self, results):
        out = {"results": results, "tot": time.time() - self.start}
        out.update(self.t)
        return out


class CtdetDetector:
    def __init__(self, opt):
        if opt.gpus[0] < 0 or not torch.cuda.is_available():
            raise RuntimeError("codenet_b200 has no CPU execution path: CtdetDetector needs a B200 (opt.gpus >= 0)")
        opt.device = torch.device("cuda", opt.gpus[0])
        self.opt = opt
        self.float_model = not opt.resume_quantize
        self.mean = np.array(opt.mean, dtype=np.float32).reshape(1, 1, 3)
        self.std = np.array(opt.std, dtype=np.float32).reshape(1, 1, 3)
        self.max_per_image = 100
        self.num_classes = opt.num_classes
        self.scales = opt.test_scales
        if self.float_model:
            # the unquantised model (test.py without --resume-quantize): its state dict in the reference's key space feeds
            # engine_f32.EngineF32 (fp32 NCHW kernels; opt.f32_gemm = "fp32" | "tf32x3" selects the 1x1-conv arithmetic)
            sd = getattr(opt, "state_dict", None)
            if getattr(opt, "load_model", ""):
                ck = torch.load(opt.load_model, map_location="cpu")
                sd = ck["state_dict"] if "state_dict" in ck else ck
            if sd is None:
                raise RuntimeError("float CtdetDetector needs opt.load_model or opt.state_dict")
            self._f32_state = {(k[7:] if k.startswith("module.") else k): v for k, v in sd.items()}
            self._f32_engines = {}
            self.model = None
            return
        self.model = PoseShuffleNetV2(opt.heads, opt.head_conv, w2=opt.w2, maxpool=opt.maxpool)
        quantize_shufflenetv2_dcn(self.model, quant_conv=opt.w_bit, quant_bn=None, quant_act=opt.a_bit,
                                  wt_quant_mode='symmetric', act_quant_mode='asymmetric', wt_per_channel=True,
                                  wt_percentile=opt.wt_percentile, act_percentile=opt.act_percentile,
                                  deform_backbone=False, w2=opt.w2, maxpool=opt.maxpool)
        if getattr(opt, "load_model", ""):
            self.load_model(opt.load_model)
        elif getattr(opt, "state_dict", None) is not None:
            self.load_state_dict(opt.state_dict)
        self.model.offset_mode = getattr(opt, "offset_mode", "bilinear")
        self.model.eval()
        freeze_ranges(self.model)
        self.mean = np.array(opt.mean, dtype=np.float32).reshape(1, 1, 3)
        self.std = np.array(opt.std, dtype=np.float32).reshape(1, 1, 3)
        self.max_per_image = 100
        self.num_classes = opt.num_classes
        self.scales = opt.test_scales
        self.opt = opt
        self.pause = True

    # -- checkpoint ingestion (lib/models/model.py:35-88: strips 'module.', tolerates the optimizer entry) ------------
    def load_state_dict(self, sd):
        sd = {(k[7:] if k.startswith("module.") else k): (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v)))
              for k, v in sd.items()}
        own = self.model.state_dict()
        for k, v in sd.items():
            if k in own and tuple(own[k].shape) != tuple(v.shape):
                v = v.reshape(own[k].shape) if v.numel() == own[k].numel() else own[k]
                sd[k] = v
        missing, unexpected = self.model.load_state_dict(sd, strict=False)
        # the stage-shared QuantAct appears under every unit's name (all aliases of ONE module): a key is only missing
        # if none of its aliases was provided
        live = self.model.state_dict(keep_vars=True)
        given = {id(live[k]) for k in sd if k in live}
        missing = [k for k in missing if not k.endswith("num_batches_tracked") and id(live[k]) not in given]
        if missing:
            raise RuntimeError("checkpoint lacks %d tensors of the quantised CoDeNet graph, e.g. %s" % (len(missing), missing[:4]))
        return unexpected

    def load_model(self, path):
        ck = torch.load(path, map_location="cpu")
        return self.load_state_dict(ck["state_dict"] if "state_dict" in ck else ck)

    # -- geometry of the network input -------------------------------------------------------------------------------------
    def input_geometry(self, height, width, scale):
        """(input height, input width, centre, scale) of base_detector.py:48-60: fixed resolution -> the longer side is
        mapped onto the input width; otherwise the scaled image is padded up to the next multiple of pad + 1."""
        sh, sw = int(height * scale), int(width * scale)
        if self.opt.fix_res:
            return (sh, sw), (self.opt.input_h, self.opt.input_w), np.array([sw / 2., sh / 2.], np.float32), float(max(height, width))
        ih, iw = (sh | self.opt.pad) + 1, (sw | self.opt.pad) + 1
        return (sh, sw), (ih, iw), np.array([sw // 2, sh // 2], np.float32), np.array([iw, ih], np.float32)

    def _meta(self, c, s, ih, iw):
        r = self.opt.down_ratio
        return {'c': c, 's': s, 'out_height': ih // r, 'out_width': iw // r}

    def pre_process(self, image, scale, meta=None):
        """uint8 HWC image -> normalised fp32 [1|2,3,H,W] tensor + meta, cv2 resize / warpAffine as in the reference."""
        import cv2
        (sh, sw), (ih, iw), c, s = self.input_geometry(image.shape[0], image.shape[1], scale)
        warped = cv2.warpAffine(cv2.resize(image, (sw, sh)), get_affine_transform(c, s, 0, [iw, ih]), (iw, ih), flags=cv2.INTER_LINEAR)
        chw = self._normalize_host(warped).transpose(2, 0, 1)[None]
        if self.opt.flip_test:
            chw = np.concatenate([chw, chw[..., ::-1]], 0)
        return torch.from_numpy(np.ascontiguousarray(chw)), self._meta(c, s, ih, iw)

    def _normalize_host(self, warped):
        """pre_process's normalisation (base_detector.py:66-68) of uint8 HWC pixels: numpy float64, rounded once to fp32."""
        return ((warped / 255. - self.mean) / self.std).astype(np.float32)

    def _normalize_device(self, images):
        """_process_float's normalisation of uint8 [..., 3] CUDA pixels (pre_process_device's layout): torch fp32 on the device."""
        mean = torch.as_tensor(self.mean.reshape(3), device=images.device)
        std = torch.as_tensor(self.std.reshape(3), device=images.device)
        return (images.float() / 255.0 - mean) / std

    def _device_table(self, scale):
        """Which normalisation run() gives test scale `scale` of a uint8 HWC frame in the unquantised model: True for
        _normalize_device (pre_process_device: scale 1 with opt.device_pre_process), False for pre_process's _normalize_host."""
        return scale == 1 and bool(getattr(self.opt, "device_pre_process", True))

    def _table_index(self, scales, frames):
        """cdn_warp_affine_u8_f32_batch's table index of every descriptor of `frames` frames (frame-major, scale-minor): 0 for
        the device normalisation, 1 for the host one (_device_table, _norm_tables)."""
        return np.tile(np.array([0 if self._device_table(s) else 1 for s in scales], np.int32), frames)

    def _host_table(self):
        """_normalize_host of the 256 byte values in every channel: numpy fp32 [3, 256]."""
        return np.ascontiguousarray(self._normalize_host(np.repeat(_BYTES[:, None], 3, 1)[None])[0].T)

    def _norm_tables(self, dev):
        """The tables of cdn_warp_affine_u8_f32_batch, fp32 [2, 3, 256] on `dev`: [0] = _normalize_device and [1] =
        _normalize_host of the 256 byte values in every channel, each computed by the helper itself.  Both normalisations are
        elementwise functions of a byte and its channel, so a lookup in these tables gives exactly what they give."""
        on_dev = self._normalize_device(torch.from_numpy(np.repeat(_BYTES[:, None], 3, 1)).to(dev)).t()
        return torch.stack([on_dev, torch.from_numpy(self._host_table()).to(dev)]).contiguous()

    def pre_process_device(self, image, scale=1, meta=None):
        """pre_process for a raw uint8 HWC image at test scale 1 ON THE DEVICE: the frame is uploaded as it is and
        cdn_warp_affine_u8 (bit-identical to the cv2.warpAffine call of base_detector.py:61-65; at scale 1 the cv2.resize in
        front of it is the identity) writes the network-sized uint8 image, mirrored copy included for --flip_test.  The
        normalisation then happens inside the stem kernel.  Returns (uint8 CUDA tensor [1|2, H, W, 3], meta)."""
        import ctypes as C
        from .. import _lib
        if scale != 1 or image.dtype != np.uint8 or image.ndim != 3 or image.shape[2] != 3:
            raise ValueError("pre_process_device takes a uint8 HWC image at test scale 1")
        (sh, sw), (ih, iw), c, s = self.input_geometry(image.shape[0], image.shape[1], 1)
        M = np.ascontiguousarray(get_affine_transform(c, s, 0, [iw, ih]), dtype=np.float64)
        src = torch.from_numpy(np.ascontiguousarray(image)).to(self.opt.device)
        n = 2 if self.opt.flip_test else 1
        dst = torch.empty((n, ih, iw, 3), dtype=torch.uint8, device=self.opt.device)
        with torch.cuda.device(self.opt.device):
            _lib.check(_lib.load().cdn_warp_affine_u8(C.c_void_p(src.data_ptr()), sh, sw, C.c_void_p(M.ctypes.data), C.c_void_p(dst.data_ptr()),
                                                      ih, iw, n - 1, C.c_void_p(torch.cuda.current_stream(self.opt.device).cuda_stream)))
        return dst, self._meta(c, s, ih, iw)

    def _is_identity_input(self, image, scale):
        """True when resize + warpAffine leave the image untouched: uint8, already input-sized, landscape or square (for a
        portrait image the longer side is the height, so the affine scales by input_w / height and pads)."""
        return (scale == 1 and self.opt.fix_res and not self.opt.flip_test and image.dtype == np.uint8 and
                image.shape[:2] == (self.opt.input_h, self.opt.input_w) and image.shape[1] >= image.shape[0])

    def _engine_for(self, H, W, batch, device):
        eng = self.model.compile_engine(H, W, max(batch, getattr(self.opt, "max_batch", 1)), device=device, K=self.opt.K)
        if not getattr(eng, "_norm", False):
            eng.set_normalization(self.mean.reshape(3), self.std.reshape(3))
        return eng

    def process_u8(self, images_u8, return_time=False):
        """Fast path of run(): uint8 [B,H,W,3] images already at the network's input size (then the reference's
        resize + warpAffine of pre_process are the identity and only the normalisation is left, which the stem kernel
        applies).  CUDA tensor in, same outputs as process()."""
        if self.float_model:
            return self._process_float(images_u8, return_time)
        B, H, W, _ = images_u8.shape
        dev = images_u8.device.index if images_u8.device.index is not None else torch.cuda.current_device()
        out = self._engine_for(H, W, B, dev).run(images_u8.contiguous(), maps=True, dets=True)
        torch.cuda.synchronize(images_u8.device)
        forward_time = time.time()
        output = {h: out[h] for h in self.opt.heads}
        return (output, out["dets"], forward_time) if return_time else (output, out["dets"])

    def _process_float(self, images, return_time):
        """process() for the unquantised model: EngineF32 forward (logits), hm.sigmoid_() as ctdet.py:32, decode on the device."""
        if images.dtype == torch.uint8:                              # pre_process_device's layout: normalise as base_detector.py:66-68
            images = self._normalize_device(images).permute(0, 3, 1, 2)
        x = images.contiguous().float()
        output, dets = self._forward_float(x)
        torch.cuda.synchronize(x.device)
        forward_time = time.time()
        return (output, dets, forward_time) if return_time else (output, dets)

    def _forward_float(self, x):
        """_process_float without the synchronisation: enqueues EngineF32 (detect, or forward + the flip average + decode with
        --flip_test) on the current stream and returns (output, dets).  x: contiguous CUDA fp32 [B,3,H,W]."""
        from ..arch import NetConfig
        from ..engine_f32 import EngineF32
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        eng = self._f32_engines.get(dev)
        if eng is None:
            cfg = NetConfig(num_classes=int(self.opt.heads["hm"]), w2=bool(self.opt.w2), maxpool=bool(self.opt.maxpool))
            eng = self._f32_engines[dev] = EngineF32(cfg, self._f32_state, device=dev, K=self.opt.K,
                                                     gemm=getattr(self.opt, "f32_gemm", "fp32"))
        if not self.opt.flip_test and self.opt.reg_offset:
            dets, _, v = eng.detect(x)
            hm, wh, reg = v["hm"].sigmoid(), v["wh"], v.get("reg")
        else:
            v = eng.forward(x)
            hm, wh, reg = v["hm"].sigmoid(), v["wh"].contiguous(), (v.get("reg") if self.opt.reg_offset else None)
            if self.opt.flip_test:
                hm = (hm[0::2] + torch.flip(hm[1::2], [3])) / 2
                wh = (wh[0::2] + torch.flip(wh[1::2], [3])) / 2
                reg = reg[0::2] if reg is not None else None
            dets = ctdet_decode(hm, wh, reg=reg, cat_spec_wh=self.opt.cat_spec_wh, K=self.opt.K)
        output = {"hm": hm, "wh": wh}
        if reg is not None:
            output["reg"] = reg
        return output, dets

    def process(self, images, return_time=False):
        """images: CUDA fp32 [B,3,H,W] (the reference's tensor) or uint8 [B,H,W,3] (pre_process_device).
        Returns (output {'hm' (post-sigmoid), 'wh', 'reg'}, dets [B|1,K,6][, time])."""
        if not images.is_cuda:
            raise RuntimeError("codenet_b200 has no CPU execution path: process() needs CUDA images")
        if self.float_model:
            return self._process_float(images, return_time)
        x = images.contiguous() if images.dtype == torch.uint8 else images.contiguous().float()
        marks = []

        def mark():                                  # the network's outputs are complete: the forward time of run()'s "net"
            torch.cuda.synchronize(images.device)
            marks.append(time.time())
        output, dets = self._forward(x, mark=mark)
        return (output, dets, marks[0]) if return_time else (output, dets)

    def _forward(self, x, out=None, maps=True, mark=None):
        """process() of the quantised model without a synchronisation: enqueues the engine and the decode on the current stream
        and returns (output, dets).  x: contiguous CUDA uint8 [B,H,W,3] or fp32 [B,3,H,W].  `out`: Engine.run's output
        buffers, kept by the caller so that the engine replays one graph (at least B images each); `maps=False` leaves the head
        maps out where the detections do not need them.  `mark()`, if given, is called once the network's outputs are
        enqueued, before the host-side decode steps."""
        B = x.shape[0]
        H, W = (x.shape[1], x.shape[2]) if x.dtype == torch.uint8 else (x.shape[2], x.shape[3])
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        eng = self._engine_for(H, W, B, dev)
        if not self.opt.flip_test:
            # forward + sigmoid + decode in one graph replay; `hm` comes back post-sigmoid like output['hm'].sigmoid_()
            out = eng.run(x, maps=maps or not self.opt.reg_offset, dets=True, out=out)
            if mark is not None:
                mark()
            output = {h: out[h][:B] for h in self.opt.heads if h in out}
            dets = out["dets"][:B] if self.opt.reg_offset else ctdet_decode(out["hm"][:B], out["wh"][:B], reg=None, K=self.opt.K)
        else:
            # image + mirrored image: average hm and wh with the mirror flipped back (ctdet.py:35-38), on the device
            import ctypes as C
            from .. import _lib
            out = eng.run(x, maps=True, dets=False, out=out)
            output = {h: out[h][:B] for h in self.opt.heads}
            pairs = B // 2
            hm = torch.empty((pairs,) + tuple(out["hm"].shape[1:]), dtype=torch.float32, device=x.device)
            wh = torch.empty((pairs,) + tuple(out["wh"].shape[1:]), dtype=torch.float32, device=x.device)
            with torch.cuda.device(x.device):
                _lib.check(_lib.load().cdn_ctdet_flip_merge(
                    C.c_void_p(out["hm"].data_ptr()), C.c_void_p(out["wh"].data_ptr()), pairs, hm.shape[1], hm.shape[2], hm.shape[3],
                    C.c_void_p(hm.data_ptr()), C.c_void_p(wh.data_ptr()),
                    C.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)))
            reg = out["reg"][0:B:2].contiguous() if self.opt.reg_offset else None     # the unflipped image of every pair
            if mark is not None:
                mark()
            dets = ctdet_decode(hm, wh, reg=reg, cat_spec_wh=self.opt.cat_spec_wh, K=self.opt.K)
        return output, dets

    def post_process(self, dets, meta, scale=1):
        """dets [1|B,K,6] in output-map coordinates -> {class: [n,5]} in image coordinates.  The affine runs on the device
        (cdn_ctdet_post_affine); the grouping per class is a view operation on the K rows that come back."""
        import ctypes as C
        from .. import _lib
        d = torch.as_tensor(dets, dtype=torch.float32, device=self.opt.device).detach().reshape(1, -1, 6).contiguous().clone()
        t = np.ascontiguousarray(get_affine_transform(meta['c'], meta['s'], 0, (meta['out_width'], meta['out_height']), inv=1),
                                 dtype=np.float64).reshape(1, 6)
        g = torch.empty_like(d)
        counts = torch.empty((1, self.num_classes), dtype=torch.int32, device=d.device)
        with torch.cuda.device(d.device):
            st = C.c_void_p(torch.cuda.current_stream(d.device).cuda_stream)
            L = _lib.load()
            _lib.check(L.cdn_ctdet_post_affine(C.c_void_p(d.data_ptr()), 1, d.shape[1], C.c_void_p(t.ctypes.data), st))
            _lib.check(L.cdn_ctdet_group_by_class(C.c_void_p(d.data_ptr()), 1, d.shape[1], self.num_classes, C.c_void_p(g.data_ptr()),
                                                  C.c_void_p(counts.data_ptr()), st))
        rows, cnt = g[0].cpu().numpy(), counts[0].cpu().numpy()
        ends = np.cumsum(cnt)
        out = {j + 1: np.ascontiguousarray(rows[ends[j] - cnt[j]:ends[j], :5], dtype=np.float32).reshape(-1, 5)
               for j in range(self.num_classes)}
        if scale != 1:
            for v in out.values():
                v[:, :4] /= scale
        return out

    def merge_outputs(self, detections):
        """Per class: all scales stacked; soft-NMS when several scales were run or --nms is set; then the max_per_image best
        scores overall survive (lib/detectors/ctdet.py:59-74)."""
        classes = range(1, self.num_classes + 1)
        merged = {j: np.ascontiguousarray(np.vstack([d[j] for d in detections]), dtype=np.float32) for j in classes}
        if len(self.scales) > 1 or self.opt.nms:
            for j in classes:
                soft_nms(merged[j], Nt=0.5, method=2)
        total = sum(len(merged[j]) for j in classes)
        if total > self.max_per_image:
            cut = np.partition(np.concatenate([merged[j][:, 4] for j in classes]), total - self.max_per_image)[total - self.max_per_image]
            merged = {j: v[v[:, 4] >= cut] for j, v in merged.items()}
        return merged

    def _image_of(self, src):
        """ndarray | path | pre-processed dict of the prefetching loader (test.py:62-72) -> (image, pre-processed dict or None)"""
        if isinstance(src, np.ndarray):
            return src, None
        if isinstance(src, str):
            import cv2
            return cv2.imread(src), None
        return src['image'][0].numpy(), src

    def _frame_layout(self, height, width, scales):
        """[(source height, source width, forward matrix, meta)] of `scales` for an height x width frame: the source of a scale is
        the image pre_process hands to cv2.warpAffine (the frame itself at scale 1, its cv2.resize otherwise)."""
        layout = []
        for scale in scales:
            (sh, sw), (ih, iw), c, s = self.input_geometry(height, width, scale)
            layout.append((sh, sw, get_affine_transform(c, s, 0, [iw, ih]), self._meta(c, s, ih, iw)))
        return layout

    def _pack_frame(self, image, layout, scales, pool, offsets, desc, slot0):
        """Writes the source image of every scale of one uint8 HWC frame into the byte pool at `offsets` (the frame at scale 1,
        pre_process's host cv2.resize otherwise: DESIGN.md section 9) and fills its warp descriptors: slot0 + k for scale k, or
        slot0 + 2k with the --flip_test mirror in slot0 + 2k + 1."""
        import cv2
        n = 2 if self.opt.flip_test else 1
        for k, ((sh, sw, M, _), scale, off) in enumerate(zip(layout, scales, offsets)):
            src = image if scale == 1 else cv2.resize(image, (sw, sh))
            pool[off:off + sh * sw * 3] = np.ascontiguousarray(src).reshape(-1)
            slot = slot0 + n * k
            desc[k] = (off, sh, sw, np.asarray(M, np.float64).reshape(6), slot, slot + 1 if n == 2 else -1)

    def _warp(self, pool, desc, dst):
        """cdn_warp_affine_u8_batch on the current stream: the descriptors `desc` (_lib.WARP_DESC) from the device byte pool into
        the uint8 CUDA batch dst [slots, H, W, 3]."""
        import ctypes as C
        from .. import _lib
        st = C.c_void_p(torch.cuda.current_stream(dst.device).cuda_stream)
        _lib.check(_lib.load().cdn_warp_affine_u8_batch(C.c_void_p(pool.data_ptr()), C.c_void_p(desc.ctypes.data), len(desc),
                                                         C.c_void_p(dst.data_ptr()), dst.shape[0], dst.shape[1], dst.shape[2], st))

    def _warp_f32(self, pool, desc, table, tables, dst):
        """cdn_warp_affine_u8_f32_batch on the current stream: the descriptors `desc` from the device byte pool into the fp32 CUDA
        batch dst [slots, 3, H, W], descriptor i normalised with tables[table[i]] (_norm_tables)."""
        import ctypes as C
        from .. import _lib
        st = C.c_void_p(torch.cuda.current_stream(dst.device).cuda_stream)
        table = np.ascontiguousarray(table, dtype=np.int32)
        _lib.check(_lib.load().cdn_warp_affine_u8_f32_batch(
            C.c_void_p(pool.data_ptr()), C.c_void_p(desc.ctypes.data), C.c_void_p(table.ctypes.data), len(desc),
            C.c_void_p(tables.data_ptr()), tables.shape[0], C.c_void_p(dst.data_ptr()), dst.shape[0], dst.shape[2], dst.shape[3], st))

    def _slots_u8(self, image, scales, ih, iw):
        """The network images of `scales` of one uint8 HWC frame as one uint8 CUDA batch [slots, ih, iw, 3] (scale-major, the
        mirror after its image): the frame and its host cv2.resize copies (scales other than 1) go to the device in one byte pool
        and one cdn_warp_affine_u8_batch launch writes every slot, mirrors included.  Returns (batch, metas)."""
        from .._lib import WARP_DESC
        n = 2 if self.opt.flip_test else 1
        dev = self.opt.device
        layout = self._frame_layout(image.shape[0], image.shape[1], scales)
        (_, offsets, nbytes), = plan_frame_steps([[sh * sw * 3 for sh, sw, _, _ in layout]], n * len(scales), 1)
        pool = np.empty(nbytes, np.uint8)
        desc = np.empty(len(scales), WARP_DESC)
        self._pack_frame(image, layout, scales, pool, offsets[0], desc, 0)
        dst = torch.empty((n * len(scales), ih, iw, 3), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            self._warp(torch.from_numpy(pool).to(dev), desc, dst)
        return dst, [m for _, _, _, m in layout]

    def _merge_on_device(self, dets, metas, clock, tail=None):
        """post_process of every scale + merge_outputs for the detections [F*S, K, 6] of F images' S test scales (image-major,
        scale-minor; metas likewise): one post-affine with the per-slot transforms, one grouping, one cdn_ctdet_merge over the F
        images and one copy back.  Returns the F results.  When S x K exceeds the device merge's segment limit the per-scale
        post_process and the host merge_outputs take over, image by image.  `tail` (a device int32 tensor) comes back in the
        same copy: then (results, tail as numpy) is returned."""
        import ctypes as C
        from .. import _lib
        S, K, nc = len(self.scales), dets.shape[1], self.num_classes
        F = dets.shape[0] // S
        if S * K > MERGE_MAX_ROWS:
            results = []
            for f in range(F):
                per_scale = [self.post_process(dets[f * S + i:f * S + i + 1], metas[f * S + i], scale) for i, scale in enumerate(self.scales)]
                clock.lap("post")
                results.append(self.merge_outputs(per_scale))
                clock.lap("merge")
            return results if tail is None else (results, tail.cpu().numpy())
        d = dets.detach().to(self.opt.device, torch.float32).contiguous().clone()
        t = np.ascontiguousarray(np.stack([get_affine_transform(m['c'], m['s'], 0, (m['out_width'], m['out_height']), inv=1).reshape(6)
                                           for m in metas]), dtype=np.float64)
        g = torch.empty_like(d)
        counts = torch.empty((F * S, nc), dtype=torch.int32, device=d.device)
        R = S * K * 5                                                               # merged rows of one image
        extra = 0 if tail is None else tail.numel()
        buf = torch.empty(F * (R + nc) + extra, dtype=torch.float32, device=d.device)   # rows, the class counts (int32), tail
        divisors = np.ascontiguousarray(self.scales, dtype=np.float32)
        with torch.cuda.device(d.device):
            st = C.c_void_p(torch.cuda.current_stream(d.device).cuda_stream)
            L = _lib.load()
            _lib.check(L.cdn_ctdet_post_affine(C.c_void_p(d.data_ptr()), F * S, K, C.c_void_p(t.ctypes.data), st))
            _lib.check(L.cdn_ctdet_group_by_class(C.c_void_p(d.data_ptr()), F * S, K, nc, C.c_void_p(g.data_ptr()),
                                                  C.c_void_p(counts.data_ptr()), st))
            clock.lap("post")
            _lib.check(L.cdn_ctdet_merge(C.c_void_p(g.data_ptr()), C.c_void_p(counts.data_ptr()), F, S, K, nc,
                                         C.c_void_p(divisors.ctypes.data), int(bool(self.opt.nms)), self.max_per_image,
                                         C.c_void_p(buf.data_ptr()), C.c_void_p(buf[F * R:].data_ptr()), st))
            if extra:
                buf[F * (R + nc):].view(torch.int32).copy_(tail)
        host = buf.cpu().numpy()
        cnts = host[F * R:F * (R + nc)].view(np.int32).reshape(F, nc)
        results = []
        for f in range(F):
            rows, cnt = host[f * R:(f + 1) * R].reshape(-1, 5), cnts[f]
            ends = np.cumsum(cnt)
            results.append({j + 1: rows[ends[j] - cnt[j]:ends[j]] for j in range(nc)})
        clock.lap("merge")
        return results if tail is None else (results, host[F * (R + nc):].view(np.int32).copy())

    def _run_float(self, image, prepared, clock):
        """run() of the unquantised model: one network call per scale as before (its uint8 normalisation runs in torch fp32,
        which is not what pre_process computes at scales other than 1), then the device merge."""
        dets, metas = [], []
        for scale in self.scales:
            if prepared is not None:
                images = prepared['images'][scale][0]
                meta = {k: (v.numpy()[0] if torch.is_tensor(v) else v) for k, v in prepared['meta'][scale].items()}
            elif image.dtype == np.uint8 and image.ndim == 3 and self._device_table(scale):
                images, meta = self.pre_process_device(image, scale)
            else:
                images, meta = self.pre_process(image, scale)
            images = images.to(self.opt.device)
            torch.cuda.synchronize()
            clock.lap("pre")
            _, d, t_forward = self.process(images, return_time=True)
            torch.cuda.synchronize()
            clock.lap("net", t_forward)
            clock.lap("dec")
            dets.append(d[:1])
            metas.append(meta)
        return self._merge_on_device(torch.cat(dets, 0), metas, clock)[0]

    def run(self, image_or_path_or_tensor, meta=None):
        """All test scales of the image that share one network input size (all of them with fix_res) go through the engine as
        one batch, scale-major with every mirror right after its image; then one post-affine, grouping and merge on the device
        for all scales and one copy back (merge_outputs on the host only when scales x K exceeds the device merge's limit)."""
        clock = _Stages()
        image, prepared = self._image_of(image_or_path_or_tensor)
        clock.lap("load")
        if self.float_model:
            return clock.result(self._run_float(image, prepared, clock))
        if prepared is not None:
            sizes = [tuple(int(v) for v in prepared['images'][scale][0].shape[-2:]) for scale in self.scales]
        else:
            sizes = [self.input_geometry(image.shape[0], image.shape[1], scale)[1] for scale in self.scales]
        u8 = (prepared is None and image.dtype == np.uint8 and image.ndim == 3 and image.shape[2] == 3 and
              (getattr(self.opt, "device_pre_process", True) or all(self._is_identity_input(image, s) for s in self.scales)))
        dets, metas = [None] * len(self.scales), [None] * len(self.scales)
        for (ih, iw), idx in plan_scale_batches(sizes):
            scales = [self.scales[i] for i in idx]
            if prepared is not None:
                images = torch.cat([prepared['images'][scale][0] for scale in scales], 0)
                ms = [{k: (v.numpy()[0] if torch.is_tensor(v) else v) for k, v in prepared['meta'][scale].items()} for scale in scales]
            elif u8:
                images, ms = self._slots_u8(image, scales, ih, iw)
            else:
                pre = [self.pre_process(image, scale) for scale in scales]
                images, ms = torch.cat([p[0] for p in pre], 0), [p[1] for p in pre]
            images = images.to(self.opt.device)
            torch.cuda.synchronize()
            clock.lap("pre")
            _, d, t_forward = self.process(images, return_time=True)
            torch.cuda.synchronize()
            clock.lap("net", t_forward)
            clock.lap("dec")
            for k, i in enumerate(idx):
                dets[i], metas[i] = d[k:k + 1], ms[k]
        return clock.result(self._merge_on_device(torch.cat(dets, 0), metas, clock)[0])

    def run_batch(self, frames):
        """run() for many frames: frames is a list of uint8 HWC 3-channel arrays, image paths and/or encoded images (bytes,
        bytearray, memoryview, 1-D uint8 arrays).  Returns one dict per frame in run()'s format; element i's results are
        run(frames[i])'s (run() reads a path with cv2.imread), and the stage timers are the call's totals divided evenly across
        its frames (summed over frames they give the wall time).  Paths are read as bytes: the file read is the "load" timer.

        Engine steps of max(opt.max_batch, slots of one frame) slots hold whole frames, frame-major, every frame's slots
        scale-major with each --flip_test mirror right after its image (plan_frame_steps).  Per step the raw frames and their
        host cv2.resize copies (scales other than 1) are packed into a pinned staging buffer, sent with one copy on a copy
        stream, and one cdn_warp_affine_u8_batch launch writes every slot; then the engine, the flip merge and decode.  The
        unquantised model takes the same steps with one cdn_warp_affine_u8_f32_batch launch instead, which writes normalised
        fp32 NCHW slots through the 3 x 256 table run() uses for each scale (_device_table, _norm_tables), then EngineF32
        eagerly (_forward_float).  When
        the one test scale is 1 and a step holds at least JPEG_DEVICE_MIN_FRAMES frames, the JPEG streams the device takes
        (cdn_jpeg_parse) go up compressed in the same staging copy,
        with their descriptors, and one cdn_jpeg_decode_batch call decodes them into the device pool the warp reads; other
        encoded inputs are decoded by cv2 on the host first.  Two staging buffers, kept on the detector, let the packing and
        copy of step n + 1 overlap the compute of step n.  After the last step one post-affine, grouping, cdn_ctdet_merge over
        all frames and one copy back (_merge_on_device), which also brings the decode status of every device-decoded frame:
        a frame the device flagged (corrupt data) is decoded by cv2 and re-run through run().
        Needs fix_res (the engine is compiled for one input size; run() is the path for keep_res); prefetched dicts go through
        run().  JPEGs of the unquantised model are decoded by cv2 on the host."""
        from .. import jpeg
        clock = _Stages()
        items = self._batch_frames(frames)
        if not items:
            return []
        clock.lap("load")
        opt, dev = self.opt, self.opt.device
        n = 2 if opt.flip_test else 1
        S, F, ih, iw = len(self.scales), len(items), opt.input_h, opt.input_w
        spf = n * S
        shapes = [im.shape[:2] if im is not None else (int(d[0]["height"]), int(d[0]["width"])) for im, _, d in items]
        layouts = [self._frame_layout(h, w, self.scales) for h, w in shapes]
        metas = [m for layout in layouts for _, _, _, m in layout]
        max_batch = getattr(opt, "max_batch", 1)
        # a JPEG stream is staged after the raw sources of its step (device decoding implies one test scale)
        steps = plan_frame_steps([[0] if items[f][0] is None else [sh * sw * 3 for sh, sw, _, _ in layouts[f]] for f in range(F)],
                                 spf, max_batch)
        step_slots = max(int(max_batch), spf)
        on_dev = [f for f in range(F) if items[f][0] is None]
        rank = {f: k for k, f in enumerate(on_dev)}
        from .._lib import WARP_DESC
        with torch.cuda.device(dev):
            dev_index = torch.cuda.current_device()
            eng = None if self.float_model else self._engine_for(ih, iw, step_slots, dev_index)
            st = self._batch_state(dev_index, step_slots, ih, iw, eng)
            compute, copy = torch.cuda.current_stream(dev_index), st["copy"]
            dets = torch.empty((F * S, opt.K, 6), dtype=torch.float32, device=dev)
            status = torch.empty(len(on_dev), dtype=torch.int32, device=dev)
            h2d_done, warp_done = [None, None], [None, None]
            for i, (fr, offsets, nbytes) in enumerate(steps):
                b = i % 2
                if h2d_done[b] is not None:
                    h2d_done[b].synchronize()                  # staging buffer b is free again
                jf = [f for f in fr if items[f][0] is None]
                staged = pool_bytes = nbytes
                if jf:
                    # staged: raw sources, the descriptor table, the streams; the device pool goes on with the decoded frames
                    table = -(-nbytes // jpeg.WS_ALIGN) * jpeg.WS_ALIGN
                    desc = np.concatenate([items[f][2] for f in jf])
                    soffs, staged, out_end, ws_bytes = jpeg.layout(desc, table + desc.nbytes, [items[f][1].size for f in jf], 0)
                    out_base = -(-staged // jpeg.WS_ALIGN) * jpeg.WS_ALIGN
                    desc["out_offset"] += out_base
                    pool_bytes = out_base + out_end
                stage, pool, grown = self._staging(st, b, staged, pool_bytes)
                host = stage.numpy()
                wdesc = np.empty(len(fr) * S, WARP_DESC)
                for k, f in enumerate(fr):
                    image, data, _ = items[f]
                    if image is not None:
                        self._pack_frame(image, layouts[f], self.scales, host, offsets[k], wdesc[k * S:(k + 1) * S], k * spf)
                    else:
                        j = jf.index(f)
                        host[soffs[j]:soffs[j] + data.size] = data
                        (sh, sw, M, _), = layouts[f]
                        wdesc[k] = (desc[j]["out_offset"], sh, sw, np.asarray(M, np.float64).reshape(6), k * spf,
                                    k * spf + 1 if n == 2 else -1)
                if jf:
                    host[table:table + desc.nbytes] = desc.view(np.uint8)
                if grown:
                    # a new pool may reuse memory the compute stream freed with work still queued (e.g. the flip merge's maps)
                    copy.wait_stream(compute)
                elif warp_done[b] is not None:
                    copy.wait_event(warp_done[b])              # the warp of step i - 2 has read device pool b
                with torch.cuda.stream(copy):
                    pool[:staged].copy_(stage[:staged], non_blocking=True)
                    h2d_done[b] = torch.cuda.Event()
                    h2d_done[b].record(copy)
                compute.wait_event(h2d_done[b])
                B = len(fr) * spf
                if jf:
                    ws = self._jpeg_workspace(st, ws_bytes)
                    jpeg.decode_batch(pool.data_ptr(), pool.numel(), desc, pool.data_ptr() + table, ws.data_ptr(), ws.numel(),
                                      pool.data_ptr(), pool.numel(), status[rank[jf[0]]:].data_ptr(), compute.cuda_stream)
                if self.float_model:
                    self._warp_f32(pool, wdesc, self._table_index(self.scales, len(fr)), st["tables"], st["dst"])
                else:
                    self._warp(pool, wdesc, st["dst"])
                warp_done[b] = torch.cuda.Event()
                warp_done[b].record(compute)
                clock.lap("pre")
                if self.float_model:
                    _, d = self._forward_float(st["dst"][:B])
                else:
                    _, d = self._forward(st["dst"][:B], out=st["out"], maps=False)
                clock.lap("net")
                dets[fr.start * S:fr.stop * S].copy_(d)
                clock.lap("dec")
            results, bad = self._merge_on_device(dets, metas, clock, tail=status)
        for k in np.flatnonzero(bad):
            # corrupt data the device flagged: what cv2.imread + run() give for the frame
            f = on_dev[k]
            redo = self.run(jpeg.imdecode_host(items[f][1]))
            results[f] = redo["results"]
            for key in _Stages.KEYS:
                clock.t[key] += redo[key]
            clock.mark = time.time()
        out = clock.result(None)
        return [dict(out, results=r, **{k: out[k] / F for k in ("tot",) + _Stages.KEYS}) for r in results]

    def _batch_frames(self, frames):
        """run_batch's inputs checked and loaded -> [(image, encoded bytes, JPEG descriptor)]: uint8 HWC 3-channel arrays as
        they are (image, None, None); paths (read as bytes) and encoded images as (None, bytes, descriptor) when the device
        decodes them (the quantised model, test_scales == [1], at least JPEG_DEVICE_MIN_FRAMES frames per engine step,
        cdn_jpeg_parse accepts the stream), else decoded by cv2.imdecode, which is what cv2.imread does after reading the file
        (image, None, None)."""
        from .. import jpeg
        if not self.opt.fix_res:
            raise ValueError("run_batch needs fix_res: without it every input size compiles its own engine; use run() for keep_res")
        for f in frames:
            if isinstance(f, np.ndarray):
                if f.dtype != np.uint8 or not (f.ndim == 1 or (f.ndim == 3 and f.shape[2] == 3)):
                    raise ValueError("run_batch takes uint8 HWC 3-channel frames or 1-D uint8 encoded images, got %s %s"
                                     % (f.dtype, f.shape))
            elif not isinstance(f, (str, bytes, bytearray, memoryview)):
                raise ValueError("run_batch takes uint8 arrays, image paths or encoded images, not %s (prefetched dicts go "
                                 "through run())" % type(f).__name__)
        # one restart interval decodes serially in one thread, so a device decode call costs about one frame's entropy decode
        # (13-41 ms for 500x375 q75-q95 on a B200) whatever the number of frames: it pays from JPEG_DEVICE_MIN_FRAMES per step
        spf = len(self.opt.test_scales) * (2 if self.opt.flip_test else 1)
        per_step = max(int(getattr(self.opt, "max_batch", 1)), spf) // spf
        device_jpeg = (self.opt.resume_quantize and list(self.opt.test_scales) == [1] and
                       min(per_step, len(frames)) >= JPEG_DEVICE_MIN_FRAMES)
        items = []
        for f in frames:
            if isinstance(f, np.ndarray) and f.ndim == 3:
                items.append((f, None, None))
                continue
            if isinstance(f, str):
                try:
                    with open(f, "rb") as fh:
                        data = np.frombuffer(fh.read(), np.uint8)
                except OSError:
                    raise ValueError("run_batch: cannot read image %r" % f) from None
            else:
                data = jpeg.as_bytes(f)
            if device_jpeg:
                rc, desc = jpeg.parse(data)
                if rc == 0:
                    items.append((None, data, desc))
                    continue
            try:
                items.append((jpeg.imdecode_host(data), None, None))
            except ValueError:
                raise ValueError("run_batch: cannot read image %s" % (repr(f) if isinstance(f, str) else "(%d bytes)" % data.size)) from None
        return items

    def _batch_state(self, dev, step_slots, ih, iw, eng):
        """run_batch's device buffers, kept between calls so the engine replays the same graphs: the warp's destination batch,
        the engine's outputs, the copy stream and the two staging buffers (pinned host + device pool).  The unquantised model
        (eng None) has an fp32 NCHW destination and the normalisation tables instead of engine outputs."""
        key = (dev, step_slots, ih, iw)
        st = getattr(self, "_batch", None)
        if st is None or st["key"] != key:
            f32 = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)
            staging = st["staging"] if st is not None and st["key"][0] == dev else [(None, None), (None, None)]
            st = {"key": key, "copy": torch.cuda.Stream(dev), "staging": staging}
            if self.float_model:
                st.update(dst=f32(step_slots, 3, ih, iw), tables=self._norm_tables(dev))
            else:
                Ho, Wo, cat = eng.plan.out_H, eng.plan.out_W, eng.plan.cat
                st["dst"] = torch.empty((step_slots, ih, iw, 3), dtype=torch.uint8, device=dev)
                st["out"] = {"hm": f32(step_slots, cat, Ho, Wo), "wh": f32(step_slots, 2, Ho, Wo), "reg": f32(step_slots, 2, Ho, Wo),
                             "dets": f32(step_slots, self.opt.K, 6),
                             "inds": torch.empty((step_slots, self.opt.K), dtype=torch.int32, device=dev)}
            self._batch = st
        return st

    def _staging(self, st, b, nbytes, pool_bytes=None):
        """Staging buffer b: pinned host memory of at least nbytes and a device pool of at least pool_bytes (default nbytes; the
        pool also holds what the device writes after the copied bytes, the decoded JPEG frames), each grown by half again when
        too small.  Returns (stage, pool, grown), grown when the device pool is new."""
        pool_bytes = nbytes if pool_bytes is None else pool_bytes
        stage, pool = st["staging"][b]
        if stage is None or stage.numel() < nbytes:
            stage = torch.empty(max(nbytes, (stage.numel() * 3 // 2) if stage is not None else 0), dtype=torch.uint8, pin_memory=True)
        grown = pool is None or pool.numel() < pool_bytes
        if grown:
            size = max(pool_bytes, (pool.numel() * 3 // 2) if pool is not None else 0)
            pool = torch.empty(size, dtype=torch.uint8, device=st["dst"].device)
        st["staging"][b] = (stage, pool)
        return stage, pool, grown

    def _jpeg_workspace(self, st, nbytes):
        """cdn_jpeg_decode_batch's workspace (coefficients, component planes), kept with the staging buffers and grown by half
        again when too small.  Only the compute stream uses it."""
        ws = st.get("jpeg_ws")
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(max(nbytes, (ws.numel() * 3 // 2) if ws is not None else 0), dtype=torch.uint8, device=st["dst"].device)
            st["jpeg_ws"] = ws
        return ws


_BYTES = np.arange(256, dtype=np.uint8)
MERGE_MAX_ROWS = 1024          # CDN_SOFT_NMS_MAX_LEN: test scales x K rows per image that cdn_ctdet_merge takes
# frames per run_batch step from which JPEGs are decoded on the device rather than by cv2 on the host: on one B200 (1000 W) with
# 500x375 4:2:0 files the device decode lost at 16 frames per step and at 32 frames at q95, and won from 64 frames per step
# (profiles/r04_jpeg_decode.json, run_batch rows "paths_device_decode" against "host_imread_then_arrays")
JPEG_DEVICE_MIN_FRAMES = 48


def plan_scale_batches(sizes):
    """Network input size (h, w) of every test scale -> [((h, w), [scale indices])], one batch per distinct size in the order
    of first appearance, scales in their order inside a batch.  The engine batch is scale-major: slot k (or slots 2k, 2k+1
    with the --flip_test mirror right after its image, the order process() pairs them in) holds the k-th scale of the list."""
    groups = {}
    for i, hw in enumerate(sizes):
        groups.setdefault(tuple(int(v) for v in hw), []).append(i)
    return list(groups.items())



def plan_frame_steps(source_bytes, slots_per_frame, max_batch, align=16):
    """run_batch's engine steps.  source_bytes[i]: the byte sizes of frame i's source images (one per test scale), which take
    slots_per_frame engine slots.  A step holds max(max_batch, slots_per_frame) slots and only whole frames, in frame order;
    inside a step every source image starts at a multiple of `align` bytes of the step's pool.  Returns
    [(frames, offsets, pool_bytes)]: frames a range of frame indices, offsets[k][j] the pool offset of source j of the step's
    k-th frame."""
    per_step = max(int(max_batch), slots_per_frame) // slots_per_frame
    steps = []
    for f0 in range(0, len(source_bytes), per_step):
        frames = range(f0, min(f0 + per_step, len(source_bytes)))
        offsets, end = [], 0
        for i in frames:
            offsets.append([])
            for nb in source_bytes[i]:
                offsets[-1].append(end)
                end += -(-int(nb) // align) * align
        steps.append((frames, offsets, end))
    return steps
