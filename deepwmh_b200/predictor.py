"""Host-side mirror of the nnU-Net v1 predictor surface DeepWMH drives (SURVEY.md section 8b):

    trainer = nnUNetTrainerV2(plans, device=0)            # initialize_network + .cuda()
    trainer.load_checkpoint_ram(checkpoint, train=False)   # state_dict with nnU-Net key names
    seg, softmax = trainer.predict_preprocessed_data_return_seg_and_softmax(data, do_mirroring=True, ...)
    seg, softmax = trainer.network.predict_3D(data, do_mirroring=True, use_sliding_window=True, ...)

Same names, argument meaning, defaults and error behaviour as the reference's un-vendored nnunet
fork (reached from deepwmh/main/predict.py:153-156); all arithmetic runs in libdeepwmh_b200.so
(hand-written sm_100a CUDA).  PyTorch is used only for device memory and streams.  Combinations
the reference supports but this path does not (non-tiled, 2-D, regions_class_order, all_in_gpu's
fp16 buffers) raise NotImplementedError -- there is no CPU fallback by design.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import NetDesc, check

ACT_DTYPES = {"fp16": 0, "float16": 0, "half": 0, "bf16": 1, "bfloat16": 1}


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(device=None) -> C.c_void_p:
    """The caller's current stream ON `device` (a stream handle is only valid on its own device)."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def pad_nd_image(image: np.ndarray, new_shape, mode="constant", kwargs=None):
    """[U:batchgenerators pad_nd_image] (a10): symmetric pad of the trailing axes up to new_shape;
    returns (padded, slicer undoing the pad)."""
    kwargs = kwargs or {"constant_values": 0}
    nd = len(new_shape)
    old = np.array(image.shape[-nd:])
    diff = np.maximum(np.array(new_shape), old) - old
    below, above = diff // 2, diff // 2 + diff % 2
    pad = [[0, 0]] * (image.ndim - nd) + [[int(b), int(a)] for b, a in zip(below, above)]
    res = np.pad(image, pad, mode, **kwargs) if diff.any() else image
    return res, tuple(slice(p[0], res.shape[i] - p[1]) for i, p in enumerate(pad))


def mirror_axes_mask(mirror_axes: Sequence[int]) -> int:
    m = 0
    for a in mirror_axes:
        if a not in (0, 1, 2):
            raise ValueError("mirror axes")
        m |= 1 << int(a)
    return m


class SegmentationNetwork:
    """The `trainer.network` object: Generic_UNet weights resident on one B200 + predict_3D."""

    def __init__(self, plans: Dict, device: int = 0, act_dtype: str = "fp16", max_batch: int = 8,
                 share_workspace_with: "Optional[SegmentationNetwork]" = None):
        """share_workspace_with: another network of the same plans on the same device whose activation buffers this one
        borrows (k resident models of a checkpoint ensemble, dwmh_create_like); the lender must have its weights loaded."""
        if not torch.cuda.is_available():
            raise _lib.DwmhError("deepwmh_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
        self._lib = _lib.load()
        st = plans["plans_per_stage"][max(plans["plans_per_stage"].keys())]
        pools = [list(map(int, p)) for p in st["pool_op_kernel_sizes"]]
        kers = [list(map(int, k)) for k in st["conv_kernel_sizes"]]
        self.patch_size = tuple(int(i) for i in st["patch_size"])
        self.num_classes = int(plans["num_classes"]) + 1
        self.input_channels = int(plans["num_modalities"])
        self.device = torch.device("cuda", device)
        self.do_ds = False
        self.conv_op = "Conv3d"
        self.inference_apply_nonlin = "softmax(dim=1)"   # fused into the head kernel
        d = NetDesc()
        d.in_channels, d.num_classes = self.input_channels, self.num_classes
        d.base_num_features, d.max_num_features = int(plans["base_num_features"]), 320
        d.num_pool = len(pools)
        if d.num_pool > _lib.DWMH_MAX_POOL:
            raise NotImplementedError("more than %d poolings" % _lib.DWMH_MAX_POOL)
        for a in range(3):
            d.patch_size[a] = self.patch_size[a]
        for i, p in enumerate(pools):
            for a in range(3):
                d.pool_op_kernel_sizes[i][a] = p[a]
        for i, k in enumerate(kers):
            for a in range(3):
                d.conv_kernel_sizes[i][a] = k[a]
        d.act_dtype = ACT_DTYPES[act_dtype]
        d.max_batch = int(max_batch)
        d.struct_size = C.sizeof(NetDesc)
        self._desc = d
        self._ctx = C.c_void_p()
        self._lender = share_workspace_with          # keeps the lender alive
        if share_workspace_with is not None:
            check(self._lib.dwmh_create_like(C.byref(self._ctx), share_workspace_with._ctx))
        else:
            check(self._lib.dwmh_create(C.byref(self._ctx), device, C.byref(d)))
        self._weights_loaded = False
        self._gaussian_installed = False

    # ---- life cycle -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.dwmh_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def eval(self):
        return self

    def train(self, mode=True):
        if mode:
            raise NotImplementedError("inference-only network")
        return self

    def load_state_dict(self, state_dict: Dict):
        for k, v in state_dict.items():
            a = np.ascontiguousarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v),
                                     dtype=np.float32)
            shape = (C.c_int64 * max(a.ndim, 1))(*a.shape)
            check(self._lib.dwmh_set_weight(self._ctx, k.encode(), a.ctypes.data_as(C.c_void_p), shape, a.ndim))
        check(self._lib.dwmh_commit_weights(self._ctx))
        self._weights_loaded = True

    def install_scipy_gaussian(self):
        """Use scipy's own filter for the importance map (bit-identical to the reference's
        _get_gaussian) instead of the library's closed form."""
        from scipy.ndimage import gaussian_filter
        tmp = np.zeros(self.patch_size)
        tmp[tuple(i // 2 for i in self.patch_size)] = 1
        g = gaussian_filter(tmp, [i / 8.0 for i in self.patch_size], 0, mode="constant", cval=0)
        g = (g / np.max(g) * 1).astype(np.float32)
        g[g == 0] = np.min(g[g != 0])
        g = np.ascontiguousarray(g)
        check(self._lib.dwmh_set_importance_map(self._ctx, g.ctypes.data_as(C.c_void_p)))
        self._gaussian_installed = True

    def _st(self) -> C.c_void_p:
        return _stream(self.device)

    # ---- device-level pieces (used by the sharded drivers) ---------------------------------------
    def weight_map(self, shape: Sequence[int], step_size: float, use_gaussian: bool, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """wgt [X,Y,Z] of the complete tile set (dwmh_weight_map): data-independent, computed locally by every rank."""
        X, Y, Z = (int(v) for v in shape)
        wgt = out if out is not None else torch.empty((X, Y, Z), dtype=torch.float32, device=self.device)
        check(self._lib.dwmh_weight_map(self._ctx, X, Y, Z, float(step_size), int(bool(use_gaussian)), _ptr(wgt), self._st()))
        return wgt

    def axpy_(self, acc: torch.Tensor, x: torch.Tensor, alpha: float):
        """acc += alpha * x on the device (a13: running mean of the k models' softmax)."""
        assert acc.is_cuda and x.is_cuda and acc.dtype == x.dtype == torch.float32 and acc.is_contiguous() and x.is_contiguous()
        check(self._lib.dwmh_axpy(self._ctx, _ptr(acc), _ptr(x), float(alpha), acc.numel(), self._st()))

    def argmax2(self, softmax: torch.Tensor) -> torch.Tensor:
        seg = torch.empty(tuple(softmax.shape[1:]), dtype=torch.uint8, device=softmax.device)
        check(self._lib.dwmh_argmax2(self._ctx, _ptr(softmax), _ptr(seg), seg.numel(), self._st()))
        return seg

    def argmax(self, softmax: torch.Tensor) -> torch.Tensor:
        """Class map uint8 [x,y,z] of fp32 probabilities [C,x,y,z] on the device; ties go to the lower class (numpy.argmax).
        Two classes take dwmh_argmax2, more take dwmh_argmax."""
        assert softmax.is_cuda and softmax.dtype == torch.float32 and softmax.is_contiguous()
        if softmax.shape[0] == 2:
            return self.argmax2(softmax)
        seg = torch.empty(tuple(softmax.shape[1:]), dtype=torch.uint8, device=softmax.device)
        check(self._lib.dwmh_argmax(self._ctx, _ptr(softmax), int(softmax.shape[0]), _ptr(seg), seg.numel(), self._st()))
        return seg

    def normalize_(self, vol: torch.Tensor, seg: Optional[torch.Tensor] = None, mask_mode: int = 2, return_stats: bool = True):
        """In-place z-score of a device fp32 volume (a2).  mask_mode: 0 all, 1 seg>=0, 2 vol!=0.
        return_stats: (mean, std, count) on the host -- this synchronises the stream; False keeps the call asynchronous."""
        assert vol.is_cuda and vol.dtype == torch.float32 and vol.is_contiguous()
        if not return_stats:
            check(self._lib.dwmh_zscore(self._ctx, _ptr(vol), _ptr(seg), vol.numel(), mask_mode, None, self._st()))
            return None
        stats = (C.c_double * 3)()
        check(self._lib.dwmh_zscore(self._ctx, _ptr(vol), _ptr(seg), vol.numel(), mask_mode, stats, self._st()))
        return tuple(stats)

    def accumulate_tiles(self, vol: torch.Tensor, agg: torch.Tensor, wgt: torch.Tensor, step_size: float,
                         do_mirroring: bool, mirror_axes: Sequence[int], use_gaussian: bool,
                         tile_begin: int = 0, tile_end: int = -1):
        """dwmh_predict_3d on device tensors: vol [M,X,Y,Z] fp32 (or [X,Y,Z] for one modality), agg [C,X,Y,Z], wgt [X,Y,Z]
        (accumulated into)."""
        X, Y, Z = vol.shape[-3:]
        if (vol.shape[0] if vol.dim() == 4 else 1) != self.input_channels or vol.dim() not in (3, 4):
            raise ValueError("vol must be [%d, X, Y, Z]" % self.input_channels)
        if tuple(agg.shape) != (self.num_classes, X, Y, Z):
            raise ValueError("agg must be [%d, X, Y, Z]" % self.num_classes)
        check(self._lib.dwmh_predict_3d(self._ctx, _ptr(vol), X, Y, Z, float(step_size), int(bool(do_mirroring)),
                                        mirror_axes_mask(mirror_axes), int(bool(use_gaussian)), _ptr(agg), _ptr(wgt),
                                        int(tile_begin), int(tile_end), self._st()))

    def finalize(self, agg: torch.Tensor, wgt: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        X, Y, Z = wgt.shape
        seg = torch.empty((X, Y, Z), dtype=torch.uint8, device=agg.device)
        check(self._lib.dwmh_finalize(self._ctx, _ptr(agg), _ptr(wgt), _ptr(agg), _ptr(seg), X, Y, Z, self._st()))
        return seg, agg

    def ensemble_masked_add_(self, acc: torch.Tensor, bg_softmax: torch.Tensor, valid_mask: Optional[torch.Tensor] = None):
        """acc += 1 - m (1 - x): one checkpoint of `_parallel_softmax_masking` + `_parallel_ensembling`
        (deepwmh/pipeline/DCNN_multistage.py:102-117), in place on fp32 device tensors."""
        assert acc.is_cuda and acc.dtype == torch.float32 and acc.is_contiguous() and bg_softmax.shape == acc.shape
        assert bg_softmax.dtype == torch.float32 and bg_softmax.is_contiguous()
        if valid_mask is not None:
            assert valid_mask.dtype == torch.float32 and valid_mask.is_contiguous() and valid_mask.shape == acc.shape
        check(self._lib.dwmh_ensemble_masked_add(self._ctx, _ptr(acc), _ptr(bg_softmax), _ptr(valid_mask), acc.numel(), self._st()))

    def ensemble_refine_(self, acc: torch.Tensor, k: int) -> torch.Tensor:
        """acc /= k in place (the ensembled field) -> uint8 label `field < 0.5` (DCNN_multistage.py:118-119)."""
        label = torch.empty(acc.shape, dtype=torch.uint8, device=acc.device)
        check(self._lib.dwmh_ensemble_refine(self._ctx, _ptr(acc), int(k), _ptr(label), acc.numel(), self._st()))
        return label

    def remove_sparks(self, seg: torch.Tensor, min_volume: int = 3) -> torch.Tensor:
        """`remove_sparks` (deepwmh/analysis/image_ops.py:325-344) on the device: uint8 label map [X,Y,Z] -> uint8 mask of the
        6-connected components with at least min_volume voxels."""
        assert seg.is_cuda and seg.dtype == torch.uint8 and seg.is_contiguous() and seg.dim() == 3
        out = torch.empty_like(seg)
        X, Y, Z = seg.shape
        check(self._lib.dwmh_remove_sparks(self._ctx, _ptr(seg), X, Y, Z, int(min_volume), _ptr(out), self._st()))
        return out

    def remove_3mm_sparks(self, seg: torch.Tensor, voxel_size: Sequence[float]) -> torch.Tensor:
        """`remove_3mm_sparks` (image_ops.py:346-367): the voxel-size rule on the host, the component filter on the device."""
        vs = [float(v) for v in voxel_size]
        if max(vs) / min(vs) > 3.0:
            return self.remove_sparks(seg, 3)
        import numpy as _np
        return self.remove_sparks(seg, max(int(_np.around(3.0 / (vs[0] * vs[1] * vs[2]))), 2))

    def num_tiles(self, shape: Sequence[int], step_size: float) -> int:
        s = _lib.compute_steps(self.patch_size, shape, step_size)
        return len(s[0]) * len(s[1]) * len(s[2])

    def forward_patches(self, patches: torch.Tensor) -> torch.Tensor:
        """softmax(Generic_UNet(x)) for x [n,M,px,py,pz] fp32 on device -> [n,C,px,py,pz] fp32."""
        assert patches.is_cuda and patches.dtype == torch.float32 and patches.is_contiguous()
        n = patches.shape[0]
        if patches.numel() != n * self.input_channels * int(np.prod(self.patch_size)):
            raise ValueError("patches must be [n, %d, %d, %d, %d]" % ((self.input_channels,) + self.patch_size))
        out = torch.empty((n, self.num_classes) + tuple(self.patch_size), dtype=torch.float32, device=patches.device)
        check(self._lib.dwmh_forward_patches(self._ctx, _ptr(patches), n, _ptr(out), self._st()))
        return out

    def layer_output(self, index: int, n: int = 1) -> torch.Tensor:
        """Normalised+activated output of layer `index` for the first n samples of the last forward,
        as fp32 [n, c, d, h, w] (test hook)."""
        dims = (C.c_int32 * 5)()
        check(self._lib.dwmh_debug_layer_output(self._ctx, index, C.c_void_p(0), 0, dims, self._st()))
        per = int(dims[1]) * int(dims[2]) * int(dims[3]) * int(dims[4])
        n = min(n, int(dims[0]))
        buf = torch.empty(n * per, dtype=torch.float32, device=self.device)
        check(self._lib.dwmh_debug_layer_output(self._ctx, index, _ptr(buf), buf.numel(), dims, self._st()))
        return buf.view(n, int(dims[1]), int(dims[2]), int(dims[3]), int(dims[4]))

    def num_layers(self) -> int:
        return int(self._lib.dwmh_num_layers(self._ctx))

    def layer_kernel_kind(self, index: int) -> int:
        return int(self._lib.dwmh_layer_kernel_kind(self._ctx, index))

    def layer_norm_on_load(self, index: int) -> int:
        """1 when the layer's InstanceNorm + LeakyReLU are applied by its consumer's loader warps (no separate pass)."""
        return int(self._lib.dwmh_layer_norm_on_load(self._ctx, index))

    def set_force_generic(self, on: bool):
        check(self._lib.dwmh_set_force_generic(self._ctx, int(on)))

    def counters(self) -> Tuple[int, float]:
        k, f = C.c_int64(), C.c_double()
        check(self._lib.dwmh_get_counters(self._ctx, C.byref(k), C.byref(f)))
        return k.value, f.value

    # ---- a7 ---------------------------------------------------------------------------------------
    def predict_3D(self, x, do_mirroring: bool, mirror_axes: Tuple[int, ...] = (0, 1, 2),
                   use_sliding_window: bool = False, step_size: float = 0.5,
                   patch_size: Tuple[int, ...] = None, regions_class_order: Tuple[int, ...] = None,
                   use_gaussian: bool = False, pad_border_mode: str = "constant", pad_kwargs: dict = None,
                   all_in_gpu: bool = False, verbose: bool = True, mixed_precision: bool = True,
                   return_device_tensors: bool = False):
        """[U:SegmentationNetwork.predict_3D].  x: (M, x, y, z) numpy fp32 or CUDA tensor, M = input modalities.
        Returns (seg int64 [x,y,z], class_probabilities fp32 [classes,x,y,z]) as numpy arrays, or -- additive flag
        return_device_tensors -- (seg uint8, probabilities fp32) as CUDA tensors without the device-to-host copies."""
        assert step_size <= 1, "step_size must be smaller than 1. Otherwise there will be a gap between consecutive predictions"
        assert len(x.shape) == 4, "data must have shape (c,x,y,z)"
        if not self._weights_loaded:
            raise _lib.DwmhError("no weights loaded (call load_checkpoint_ram / load_state_dict first)")
        if pad_kwargs is None:
            pad_kwargs = {"constant_values": 0}
        if len(mirror_axes):
            if max(mirror_axes) > 2:
                raise ValueError("mirror axes")
        if not use_sliding_window:
            raise NotImplementedError("only the tiled (use_sliding_window=True) branch is on DeepWMH's path")
        if regions_class_order is not None:
            raise NotImplementedError("regions_class_order is not used by DeepWMH")
        if patch_size is not None and tuple(int(i) for i in patch_size) != self.patch_size:
            raise NotImplementedError("patch_size must equal the plans' patch size %s" % (self.patch_size,))
        if pad_border_mode != "constant" or pad_kwargs.get("constant_values", 0) != 0:
            raise NotImplementedError("only zero constant padding is supported")
        if x.shape[0] != self.input_channels:
            raise ValueError("expected %d input channel(s)" % self.input_channels)
        with torch.cuda.device(self.device):
            if isinstance(x, torch.Tensor) and x.is_cuda:
                # device input stays on the device: zero padding (a10) with the same below / above split as pad_nd_image
                vol = x.detach().to(device=self.device, dtype=torch.float32)
                diff = [max(p - s, 0) for p, s in zip(self.patch_size, vol.shape[1:])]
                pads = [(d // 2, d // 2 + d % 2) for d in diff]
                if any(diff):
                    vol = torch.nn.functional.pad(vol, (pads[2][0], pads[2][1], pads[1][0], pads[1][1], pads[0][0], pads[0][1]))
                vol = vol.contiguous()
                slicer = (slice(None),) + tuple(slice(b, vol.shape[i + 1] - a) for i, (b, a) in enumerate(pads))
            else:
                if isinstance(x, torch.Tensor):
                    x = x.detach().float().numpy()
                data, slicer = pad_nd_image(np.asarray(x, dtype=np.float32), self.patch_size, pad_border_mode, pad_kwargs)
                vol = torch.from_numpy(np.ascontiguousarray(data)).to(self.device, non_blocking=False)
            X, Y, Z = vol.shape[1:]
            agg = torch.zeros((self.num_classes, X, Y, Z), dtype=torch.float32, device=self.device)
            wgt = torch.zeros((X, Y, Z), dtype=torch.float32, device=self.device)
            self.accumulate_tiles(vol, agg, wgt, step_size, do_mirroring, mirror_axes, use_gaussian)
            seg, probs = self.finalize(agg, wgt)
            sl = tuple(slicer[1:])
            if return_device_tensors:
                return seg[sl], probs[(slice(None),) + sl]
            seg_np = seg[sl].cpu().numpy().astype(np.int64)
            probs_np = probs[(slice(None),) + sl].cpu().numpy()
        return seg_np, probs_np


class nnUNetTrainerV2:
    """The slice of the trainer surface `predict_cases` uses [U:nnUNetTrainerV2.py], B200-backed."""

    def __init__(self, plans: Dict, device: int = 0, act_dtype: str = "fp16", max_batch: int = 8,
                 exact_scipy_gaussian: bool = True, share_workspace_with: "Optional[nnUNetTrainerV2]" = None):
        self.plans = plans
        self.process_plans(plans)
        self.data_aug_params = {"do_mirror": True, "mirror_axes": (0, 1, 2)}
        self.network = SegmentationNetwork(plans, device, act_dtype, max_batch,
                                           share_workspace_with.network if share_workspace_with is not None else None)
        if exact_scipy_gaussian:
            self.network.install_scipy_gaussian()

    def process_plans(self, plans: Dict):
        stage = max(plans["plans_per_stage"].keys())
        st = plans["plans_per_stage"][stage]
        self.stage = stage
        self.patch_size = np.array(st["patch_size"]).astype(int)
        self.net_num_pool_op_kernel_sizes = st["pool_op_kernel_sizes"]
        self.net_conv_kernel_sizes = st["conv_kernel_sizes"]
        self.base_num_features = plans["base_num_features"]
        self.num_input_channels = plans["num_modalities"]
        self.num_classes = plans["num_classes"] + 1
        self.normalization_schemes = plans.get("normalization_schemes")
        self.use_mask_for_norm = plans.get("use_mask_for_norm")
        self.transpose_forward = plans.get("transpose_forward", [0, 1, 2])
        self.transpose_backward = plans.get("transpose_backward", [0, 1, 2])
        self.threeD = True

    def load_checkpoint_ram(self, checkpoint: Dict, train: bool = False):
        if train:
            raise NotImplementedError("inference only")
        sd = {(k[7:] if k.startswith("module.") else k): v for k, v in checkpoint["state_dict"].items()}
        self.network.load_state_dict(sd)

    def preprocess_patient(self, input_files, as_numpy: bool = True):
        """[U:nnUNetTrainer.preprocess_patient] -> (data [c, x, y, z] fp32, seg [1, x, y, z], properties): crop_to_nonzero,
        transpose_forward, resample to the plans' spacing and z-score (the last two on the device).  as_numpy=False keeps
        data / seg on the device (the predictor accepts CUDA tensors)."""
        from . import preprocess
        d, s, props = preprocess.preprocess_test_case(self.network, self.plans, list(input_files))
        if as_numpy:
            return d.cpu().numpy(), s.cpu().numpy(), props
        return d, s, props

    def predict_preprocessed_data_return_seg_and_softmax(
            self, data, do_mirroring: bool = True, mirror_axes: Tuple[int] = None,
            use_sliding_window: bool = True, step_size: float = 0.5, use_gaussian: bool = True,
            pad_border_mode: str = "constant", pad_kwargs: dict = None, all_in_gpu: bool = False,
            verbose: bool = True, mixed_precision=True, return_device_tensors: bool = False) -> Tuple[np.ndarray, np.ndarray]:
        if pad_border_mode == "constant" and pad_kwargs is None:
            pad_kwargs = {"constant_values": 0}
        if do_mirroring and mirror_axes is None:
            mirror_axes = self.data_aug_params["mirror_axes"]
        if do_mirroring:
            assert self.data_aug_params["do_mirror"], \
                "Cannot do mirroring as test time augmentation when training was done without mirroring"
        ds = self.network.do_ds
        self.network.do_ds = False
        self.network.eval()
        ret = self.network.predict_3D(data, do_mirroring=do_mirroring, mirror_axes=mirror_axes or (),
                                      use_sliding_window=use_sliding_window, step_size=step_size,
                                      patch_size=self.patch_size, regions_class_order=None,
                                      use_gaussian=use_gaussian, pad_border_mode=pad_border_mode,
                                      pad_kwargs=pad_kwargs, all_in_gpu=all_in_gpu, verbose=verbose,
                                      mixed_precision=mixed_precision, return_device_tensors=return_device_tensors)
        self.network.do_ds = ds
        return ret

    # C-ABI host-buffer call (the end-to-end path bench.py times)
    def predict_raw_volume_host(self, vol: np.ndarray, zscore_mask_mode: int = 2, do_mirroring: bool = True,
                                mirror_axes=(0, 1, 2), step_size: float = 0.5, use_gaussian: bool = True,
                                out_softmax: Optional[np.ndarray] = None, out_seg: Optional[np.ndarray] = None,
                                seg_mask: Optional[np.ndarray] = None):
        """raw fp32 [X,Y,Z] (one modality) or [M,X,Y,Z] host volume -> (seg uint8 [X,Y,Z], softmax fp32 [C,X,Y,Z]); z-score
        of every modality, H2D, tiled prediction, finalize and D2H all inside dwmh_predict_volume_host.  seg_mask: nnU-Net's
        crop mask (int8, >= 0 inside) -> normalisation over that mask (dwmh_predict_volume_host_masked)."""
        M = self.network.input_channels
        assert vol.dtype == np.float32 and vol.flags.c_contiguous
        assert (vol.ndim == 3 and M == 1) or (vol.ndim == 4 and vol.shape[0] == M), "vol must be [%d, X, Y, Z]" % M
        X, Y, Z = vol.shape[-3:]
        sm = out_softmax if out_softmax is not None else np.empty((self.network.num_classes, X, Y, Z), dtype=np.float32)
        sg = out_seg if out_seg is not None else np.empty((X, Y, Z), dtype=np.uint8)
        net = self.network
        if seg_mask is not None:
            assert seg_mask.dtype == np.int8 and seg_mask.shape == (X, Y, Z) and seg_mask.flags.c_contiguous
            with torch.cuda.device(net.device):
                check(net._lib.dwmh_predict_volume_host_masked(
                    net._ctx, vol.ctypes.data_as(C.c_void_p), seg_mask.ctypes.data_as(C.c_void_p), X, Y, Z, float(step_size),
                    int(bool(do_mirroring)), mirror_axes_mask(mirror_axes), int(bool(use_gaussian)),
                    sm.ctypes.data_as(C.c_void_p), sg.ctypes.data_as(C.c_void_p), net._st()))
            return sg, sm
        with torch.cuda.device(net.device):
            check(net._lib.dwmh_predict_volume_host(
                net._ctx, vol.ctypes.data_as(C.c_void_p), X, Y, Z, int(zscore_mask_mode), float(step_size),
                int(bool(do_mirroring)), mirror_axes_mask(mirror_axes), int(bool(use_gaussian)),
                sm.ctypes.data_as(C.c_void_p), sg.ctypes.data_as(C.c_void_p), net._st()))
        return sg, sm
