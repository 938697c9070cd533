"""Host side of the drop-in: `DINOSeg` with the reference's method surface
(`load_from_checkpoint`, `set_resolution`, `predict`, `forward`; reference
dt_segmentation/src/pl_torch_modules.py:141-300), executing on libdinoseg.so.

PyTorch is used for what it is good at here — owning device memory (parameters, workspace,
outputs) and streams.  All arithmetic of the hot path happens inside the CUDA library; there is
no eager / CPU fallback: calling forward on a CPU model raises.
"""
from __future__ import annotations

import ctypes as C
import io
import numbers
import pickle
import types
import warnings
import weakref

import numpy as np
import torch
from torch import nn

from . import _lib
from .synthetic import ARCHS
from .transforms import IMAGENET_MEAN, IMAGENET_STD, get_transforms


# ------------------------------------------------------------------------------------------
# Parameter containers with the reference's state_dict names (vision_transformer.py:163-191).
# They compute nothing themselves: they hold tensors (and give PyTorch's default initialisers, which
# is what the reference relies on for the conv and the head); _Backbone's forward goes to the library.
# ------------------------------------------------------------------------------------------
class _Attention(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)


class _Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Block(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = _Attention(dim)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = _Mlp(dim, hidden)


class _PatchEmbed(nn.Module):
    def __init__(self, dim, patch):
        super().__init__()
        self.patch_size = patch
        self.proj = nn.Conv2d(3, dim, kernel_size=patch, stride=patch)


class _Backbone(nn.Module):
    """Parameters of the truncated DINO ViT (first n_blocks blocks, pl_torch_modules.py:177)."""

    def __init__(self, dim, hidden, num_heads, n_blocks, patch=8, img_size=224):
        super().__init__()
        self.embed_dim = dim
        self.num_heads = num_heads
        self.patch_embed = _PatchEmbed(dim, patch)
        n_pos = (img_size // patch) ** 2
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n_pos + 1, dim))
        self.blocks = nn.ModuleList([_Block(dim, hidden) for _ in range(n_blocks)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)
        self._owner = None            # weakref to the DINOSeg that executes this backbone
        # reference init (vision_transformer.py:188-200); Conv2d keeps its default init
        nn.init.trunc_normal_(self.pos_embed, std=.02)
        nn.init.trunc_normal_(self.cls_token, std=.02)
        self.apply(self._init_weights)

    def _model(self):
        owner = self._owner() if self._owner is not None else None
        if owner is None:
            raise RuntimeError("backbone is not attached to a DINOSeg model")
        return owner

    def forward(self, x):
        """VisionTransformer.forward (vision_transformer.py:237-248) for all tokens: fp32 [B,3,r,r] (normalised, on the
        model's device) -> fp32 [B, N, D], N = (r/8)^2 + 1, CLS token first, after the final norm.  Runs on the GPU
        through DINOSeg.features; the head does not run.  Square frames only, as this method has always required
        (non-square input raises ValueError); for [B,3,H,W] frames get_intermediate_layers(x)[-1] and
        DINOSeg.features(x)[0] return the same tensor."""
        h, w = _frame_hw(x)
        if h != w:
            raise ValueError(f"model.dino(x) takes square frames [B,3,r,r], got {tuple(x.shape)}; for non-square frames "
                             "use model.dino.get_intermediate_layers(x)[-1] or model.features(x)[0]")
        return self._model().features(x, 1)[0]

    def get_intermediate_layers(self, x, n=1):
        """vision_transformer.py:282-290: list of min(n, n_blocks) fp32 [B, N, D] tensors, oldest block first, each the
        final norm of the residual stream after one of the last n blocks (one pass over the blocks).  x: fp32 [B,3,H,W]
        with H and W multiples of 8, N = (H/8)*(W/8) + 1 (CLS, then the patches row by row).  The last element equals
        forward(x) bit for bit."""
        return list(self._model().features(x, n).unbind(0))

    def get_last_selfattention(self, x):
        """Reference vision_transformer.py:273-280 returns the last block's attention [B, H, N, N]; its only caller
        (visualize_attention.py:46-54) reads the CLS row `[0, :, 0, 1:]`.  Here only that row is materialised:
        the result has shape [B, H, 1, N] (the full matrix is 311 MB per frame at 480 px and is never formed)."""
        return self._model().cls_attention(x).unsqueeze(2)

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)


class _MLPHead(nn.Module):
    """pl_torch_modules.py:108-124."""

    def __init__(self, n_classes, input_dim):
        super().__init__()
        self.layer_1 = nn.Linear(input_dim, 200)
        self.layer_2 = nn.Linear(200, 100)
        self.layer_3 = nn.Linear(100, n_classes)


class _LinearHead(nn.Module):
    """pl_torch_modules.py:127-138."""

    def __init__(self, n_classes, input_dim):
        super().__init__()
        self.layer_1 = nn.Linear(input_dim, n_classes)


class _TolerantUnpickler(pickle.Unpickler):
    """PL checkpoints pickle ctor kwargs (optimizer class, loggers...).  Classes from packages
    that are not installed are replaced by inert placeholders instead of failing the load."""

    def find_class(self, module, name):
        try:
            return super().find_class(module, name)
        except Exception:
            return type(name, (), {"__init__": lambda self, *a, **k: None,
                                   "__setstate__": lambda self, s: None})


_tolerant_pickle = types.ModuleType("dino_b200_tolerant_pickle")
_tolerant_pickle.Unpickler = _TolerantUnpickler
_tolerant_pickle.load = lambda f, **kw: _TolerantUnpickler(f, **kw).load()
_tolerant_pickle.__name__ = "pickle"


def _frame_hw(x):
    """(H, W) of device frames fp32 [B,3,H,W]; ValueError for any other layout."""
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"expected frames of shape [B,3,H,W], got {tuple(x.shape)}")
    return int(x.shape[2]), int(x.shape[3])


def _resolution_hw(resolution):
    """`resolution` of the raw-frame entry points: an int r (r x r) or an (H, W) pair."""
    if isinstance(resolution, (tuple, list)):
        if len(resolution) != 2:
            raise ValueError(f"resolution must be an int or an (H, W) pair, got {resolution!r}")
        return int(resolution[0]), int(resolution[1])
    return int(resolution), int(resolution)


class DINOSeg(nn.Module):
    """DINO ViT-S/8 (or ViT-B/8) truncated to `n_blocks` blocks + per-patch MLP head.

    Constructor arguments are the reference's (pl_torch_modules.py:144-147); the training-only
    ones are accepted and stored, nothing else.  `arch` ('vit_small' | 'vit_base') is an
    extension: the reference hard-codes ViT-S (SURVEY.md §0).
    """

    def __init__(self, data_path=None, write_path=None, class_names=None, head='linear', n_blocks=1,
                 batch_size=1, lr=1e-6, optimizer=None, freeze_backbone=True, max_epochs=200, patience=10,
                 grayscale=False, n_classes=7, pretrain_on_sim=False, comet_logger=None, augmented=True,
                 random_init=False, backbone='vit', arch='vit_small'):
        super().__init__()
        if backbone != 'vit':
            raise NotImplementedError("only backbone='vit' is part of the B200 hot path (cnn1/cnn2 are ablations)")
        if head not in ('mlp', 'linear'):
            raise ValueError(f"unknown head {head!r} (reference: 'linear' or 'mlp', pl_torch_modules.py:219-222)")
        if arch not in ARCHS:
            raise ValueError(f"unknown arch {arch!r}")
        self.n_blocks = n_blocks
        self.head = head
        self.batch_size = batch_size
        self.lr = lr
        self.optimizer = optimizer
        self.freeze_backbone = freeze_backbone
        self.max_epochs = max_epochs
        self.patience = patience
        self.grayscale = grayscale
        self.n_classes = n_classes
        self.comet_logger = comet_logger
        self.class_names = class_names
        self.pretrain_on_sim = pretrain_on_sim
        self.augmented = augmented
        self.random_init = random_init
        self.backbone = backbone
        self.arch = arch
        self.hparams = dict(data_path=data_path, write_path=write_path, class_names=class_names, head=head,
                            n_blocks=n_blocks, batch_size=batch_size, lr=lr, freeze_backbone=freeze_backbone,
                            max_epochs=max_epochs, patience=patience, grayscale=grayscale, n_classes=n_classes,
                            pretrain_on_sim=pretrain_on_sim, augmented=augmented, random_init=random_init,
                            backbone=backbone, arch=arch)

        a = ARCHS[arch]
        self.mlp_input_dim = a["embed_dim"]
        self.resolution = 480
        self.transforms = get_transforms(self.resolution)
        # The reference downloads the pretrained DINO weights here (dt_utils.py:19-29).  There is no
        # network: parameters start from the reference's random init and are expected to be
        # overwritten by load_from_checkpoint / load_state_dict.
        self.dino = _Backbone(a["embed_dim"], a["mlp_hidden"], a["num_heads"], n_blocks)
        self.clf = _MLPHead(n_classes, a["embed_dim"]) if head == 'mlp' else _LinearHead(n_classes, a["embed_dim"])
        for p in self.parameters():
            p.requires_grad_(False)

        self.dino._owner = weakref.ref(self)
        self._handle = None
        self._handle_device = None
        self._fingerprint = None
        self._lib_res = None
        self._workspace = None
        self._pending = {}            # ticket -> (frames, out) of predict_batch_async submissions in flight

    # -------------------------------------------------------------------------------------
    # construction from a checkpoint (replaces LightningModule.load_from_checkpoint, README.md:31)
    # -------------------------------------------------------------------------------------
    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location=None, strict=True, **kwargs):
        # Trust: a Lightning checkpoint is a pickle (weights_only=False executes what it contains, exactly like the
        # reference's LightningModule.load_from_checkpoint) - only load checkpoints you would also run as code.
        # Only a class that cannot be resolved (a package of the training environment that is not installed here:
        # pytorch_lightning, comet_ml, ...) triggers the tolerant retry; a corrupt file or any other error surfaces
        # as it is, and if the retry fails too the ORIGINAL error is raised.
        try:
            ckpt = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
        except (ModuleNotFoundError, AttributeError, pickle.UnpicklingError) as first_error:
            try:
                with open(checkpoint_path, "rb") as f:
                    ckpt = torch.load(io.BytesIO(f.read()), map_location="cpu", weights_only=False,
                                      pickle_module=_tolerant_pickle)
            except Exception:
                raise first_error
        hp = dict(ckpt.get("hyper_parameters", {}))
        hp.update(kwargs)
        allowed = cls.__init__.__code__.co_varnames[1:cls.__init__.__code__.co_argcount]
        hp = {k: v for k, v in hp.items() if k in allowed}
        sd = ckpt["state_dict"]
        if "arch" not in hp and "dino.cls_token" in sd:
            hp["arch"] = "vit_base" if sd["dino.cls_token"].shape[-1] == 768 else "vit_small"
        model = cls(**hp)
        model.load_state_dict(sd, strict=strict)
        if map_location is not None:
            model = model.to(map_location)
        return model

    # -------------------------------------------------------------------------------------
    @property
    def device(self):
        return self.dino.cls_token.device

    def set_resolution(self, resolution=480):
        """pl_torch_modules.py:270-274."""
        if resolution % 8 != 0:
            raise ValueError('Resolution should be a multiple of 8.')
        self.transforms = get_transforms(resolution)
        self.resolution = resolution

    # -------------------------------------------------------------------------------------
    # library handle management
    # -------------------------------------------------------------------------------------
    def _cfg(self):
        a = ARCHS[self.arch]
        return _lib.DinosegCfg(a["embed_dim"], a["num_heads"], a["mlp_hidden"], self.n_blocks, 8,
                               int(round((self.dino.pos_embed.shape[1] - 1) ** 0.5)), self.n_classes, 200, 100,
                               0 if self.head == 'mlp' else 1, 1e-6)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError(f"{what} failed: {_lib.last_error(self._handle)}")

    def _release(self):
        if self._handle is not None:
            try:
                if getattr(self, "_pending", None):
                    _lib.load().dinoseg_predict_host_wait(self._handle, 0)
                    self._pending.clear()
                _lib.load().dinoseg_destroy(self._handle)
            except Exception:
                pass
        self._handle = None
        self._fingerprint = None
        self._lib_res = None
        self._workspace = None

    def __del__(self):
        try:
            self._release()
        except Exception:  # interpreter shutdown
            pass

    def _ensure_handle(self):
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("DINOSeg (B200 build) runs on CUDA only: move the model with .to('cuda:N'); "
                               "there is no CPU fallback")
        lib = _lib.load()
        if self._handle is None or self._handle_device != dev:
            self._release()
            h = C.c_void_p()
            cfg = self._cfg()
            idx = dev.index if dev.index is not None else torch.cuda.current_device()
            if lib.dinoseg_create(C.byref(cfg), idx, C.byref(h)) != 0:
                raise RuntimeError("dinoseg_create failed: " + _lib.last_error(None))
            self._handle, self._handle_device = h, dev
        sd = self.state_dict()
        fp = tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        if fp != self._fingerprint:
            stream = self._stream()
            for k, v in sd.items():
                t = v.detach()
                if t.dtype != torch.float32 or not t.is_contiguous():
                    t = t.float().contiguous()
                shape = (C.c_int64 * t.dim())(*t.shape)
                self._check(lib.dinoseg_set_weight(self._handle, k.encode(), t.data_ptr(), shape, t.dim(), stream),
                            f"dinoseg_set_weight({k})")
            torch.cuda.current_stream(dev).synchronize()  # staging copies `t` may be temporaries
            self._fingerprint = fp
            self._lib_res = None
        return lib

    def _ensure_resolution(self, lib, hw):
        """hw: (H, W) in pixels."""
        if self._lib_res != hw:
            rc = lib.dinoseg_set_resolution_hw(self._handle, int(hw[0]), int(hw[1]), self._stream())
            if rc != 0:
                msg = _lib.last_error(self._handle)
                if "multiple of 8" in msg:
                    raise ValueError(msg)
                raise RuntimeError("dinoseg_set_resolution failed: " + msg)
            self._lib_res = hw
            self._workspace = None

    def _ensure_workspace(self, lib, batch):
        need = lib.dinoseg_workspace_bytes(self._handle, batch)
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = None
            raw = torch.empty(need + 1024, dtype=torch.uint8, device=self.device)
            off = (-raw.data_ptr()) % 1024        # the library wants a 1024-byte aligned scratch
            self._workspace = raw[off:off + need]
        return self._workspace

    # -------------------------------------------------------------------------------------
    # inference
    # -------------------------------------------------------------------------------------
    @staticmethod
    def _check_labels_square(hw, want_labels):
        if want_labels and hw[0] != hw[1]:
            raise ValueError(f"label maps (predict's np.kron tail) exist for square frames only, got {hw[0]}x{hw[1]}; "
                             "use the log-probs or the low-res map")

    def _outputs(self, b, hw, want_logprobs, want_lowres, want_labels):
        gh, gw = hw[0] // 8, hw[1] // 8
        dev = self.device
        lp = torch.empty((b * gh * gw, self.n_classes), dtype=torch.float32, device=dev) if want_logprobs else None
        low = torch.empty((b, gh, gw), dtype=torch.uint8, device=dev) if want_lowres else None
        lab = None
        if want_labels:
            p = 480 // gh
            lab = torch.empty((b, gh * p, gh * p), dtype=torch.int64, device=dev)
        return lp, low, lab

    @torch.no_grad()
    def infer(self, x, want_logprobs=True, want_lowres=False, want_labels=False):
        """Run the hot path on device frames x: fp32 [B,3,H,W] (normalised, H and W multiples of 8).

        Returns (logprobs [B*P,C] f32 | None, lowres [B,H/8,W/8] u8 | None, labels [B,g*p,g*p] i64 | None),
        all device tensors; asynchronous on the current stream.  P = (H/8)*(W/8), patches row by row.  Label maps are
        predict()'s output and exist for square frames only (g = H/8 = W/8, p = 480 // g)."""
        lib = self._ensure_handle()
        hw = _frame_hw(x)
        self._check_labels_square(hw, want_labels)
        if x.device != self.device:
            raise ValueError(f"frames are on {x.device}, model on {self.device}")
        x = x.contiguous()
        if x.dtype != torch.float32:
            x = x.float()
        b = int(x.shape[0])
        self._ensure_resolution(lib, hw)
        ws = self._ensure_workspace(lib, b)
        lp, low, lab = self._outputs(b, hw, want_logprobs, want_lowres, want_labels)
        rc = lib.dinoseg_forward(self._handle, x.data_ptr(), b,
                                 lp.data_ptr() if lp is not None else None,
                                 low.data_ptr() if low is not None else None,
                                 lab.data_ptr() if lab is not None else None,
                                 ws.data_ptr(), ws.numel(), self._stream())
        self._check(rc, "dinoseg_forward")
        return lp, low, lab

    @torch.no_grad()
    def half_counts(self, x):
        """Left / right class pixel counts of the label map, the input of the reference's potential-field controller
        (docs/index.html "Controller"; SURVEY.md section 8(f)-4), without shipping the 480x480 int64 maps to the host.

        x: device frames fp32 [B,3,r,r] (runs the forward) or a device uint8 low-res map [B,g,g] (e.g. from infer()).
        Returns a device int32 tensor [B, 2, n_classes]: pixels of each class with x < W/2 (index 0) and x >= W/2
        (index 1) of the (g*p) x (g*p) output map predict() would return.  Square frames / maps only, like predict()."""
        lib = self._ensure_handle()
        if x.dtype == torch.uint8 and x.dim() == 3:
            if x.shape[1] != x.shape[2]:
                raise ValueError(f"half_counts needs a square low-res map [B,g,g], got {tuple(x.shape)}")
            low = x.contiguous()
        else:
            if x.dim() == 4 and x.shape[2] != x.shape[3]:
                raise ValueError(f"half_counts needs square frames [B,3,r,r] (predict's label map), got {tuple(x.shape)}")
            _, low, _ = self.infer(x, want_logprobs=False, want_lowres=True)
        b, g = int(low.shape[0]), int(low.shape[1])
        p = 480 // g
        if p == 0:
            raise ValueError("resolutions above 3840 have an empty label map (480 // g == 0)")
        counts = torch.empty((b, 2, self.n_classes), dtype=torch.int32, device=low.device)
        rc = lib.dinoseg_half_counts(low.data_ptr(), b, g, p, self.n_classes, counts.data_ptr(), self._stream())
        self._check(rc, "dinoseg_half_counts")
        return counts

    @torch.no_grad()
    def cls_attention(self, x):
        """Attention of the CLS query in the last kept block: [B, heads, N] fp32, N = (H/8)*(W/8) + 1, for fp32 frames
        [B,3,H,W] (see _Backbone.get_last_selfattention)."""
        lib = self._ensure_handle()
        hw = _frame_hw(x)
        x = x.to(self.device).contiguous().float()
        b = int(x.shape[0])
        self._ensure_resolution(lib, hw)
        ws = self._ensure_workspace(lib, b)
        n = (hw[0] // 8) * (hw[1] // 8) + 1
        heads = ARCHS[self.arch]["num_heads"]
        out = torch.empty((b, heads, n), dtype=torch.float32, device=self.device)
        rc = lib.dinoseg_cls_attention(self._handle, x.data_ptr(), b, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                       self._stream())
        self._check(rc, "dinoseg_cls_attention")
        return out

    def _frames(self, x, resolution):
        """Validated device frames of features / embeddings -> (contiguous frames, (H, W), raw)."""
        if x.device != self.device:
            raise ValueError(f"frames are on {x.device}, model on {self.device}")
        raw = x.dtype == torch.uint8
        if raw:
            if x.dim() != 4 or x.shape[3] != 3:
                raise ValueError(f"expected uint8 frames of shape [B,H,W,3], got {tuple(x.shape)}")
            hw = _resolution_hw(self.resolution if resolution is None else resolution)
        else:
            hw = _frame_hw(x)
            if resolution is not None and _resolution_hw(resolution) != hw:
                raise ValueError(f"resolution {resolution} given for frames of size {hw[0]}x{hw[1]}")
            x = x.float()
        return x.contiguous(), hw, raw

    @torch.no_grad()
    def embeddings(self, x, n=1, avgpool=False, resolution=None):
        """Image embeddings, one vector per frame, as upstream DINO's k-NN and linear evaluations take them: a device fp32
        tensor, asynchronous on the current stream.  x as in features(): fp32 [B,3,H,W] or uint8 [B,Hs,Ws,3] resized to
        `resolution`.  With L = dino.get_intermediate_layers(x, n) and n_out = min(n, n_blocks):

        - avgpool=False: torch.cat([t[:, 0] for t in L], dim=-1), [B, n_out*D], oldest block first (n = 1: the CLS
          token of model.dino(x), upstream's `model(x)` embedding).  The last block runs for the CLS row only after its
          qkv GEMM, so its slice agrees with features() to the bf16 rounding of the attention and MLP operands; the
          earlier slices equal features() bit for bit.
        - avgpool=True (n_out must be 1): upstream eval_linear's
          torch.cat((cls.unsqueeze(-1), torch.mean(L[-1][:, 1:], dim=1).unsqueeze(-1)), dim=-1).reshape(B, -1),
          [B, 2D] with the CLS token and the patch-token mean interleaved, so that a classifier trained with upstream
          eval_linear applies unchanged.  The last block runs in full and the CLS values equal features() bit for bit."""
        if not isinstance(n, numbers.Integral) or n < 1:
            raise ValueError(f"n must be a positive integer, got {n!r}")
        n = int(n)
        n_out = min(n, self.n_blocks)
        if avgpool and n_out != 1:
            raise ValueError(f"avgpool concatenates the CLS token of one block with its patch mean (upstream eval_linear "
                             f"with n = 1); got n = {n} on a model with {self.n_blocks} blocks")
        lib = self._ensure_handle()
        x, hw, raw = self._frames(x, resolution)
        b = int(x.shape[0])
        self._ensure_resolution(lib, hw)
        ws = self._ensure_workspace(lib, b)
        d = self.mlp_input_dim
        cls = torch.empty((n_out, b, d), dtype=torch.float32, device=self.device)
        mean = torch.empty((b, d), dtype=torch.float32, device=self.device) if avgpool else None
        mean_ptr = mean.data_ptr() if avgpool else None
        if raw:
            mu = (C.c_float * 3)(*IMAGENET_MEAN)
            std = (C.c_float * 3)(*IMAGENET_STD)
            rc = lib.dinoseg_embeddings_u8(self._handle, x.data_ptr(), b, int(x.shape[1]), int(x.shape[2]), mu, std, n,
                                           cls.data_ptr(), mean_ptr, ws.data_ptr(), ws.numel(), self._stream())
            self._check(rc, "dinoseg_embeddings_u8")
        else:
            rc = lib.dinoseg_embeddings(self._handle, x.data_ptr(), b, n, cls.data_ptr(), mean_ptr, ws.data_ptr(),
                                        ws.numel(), self._stream())
            self._check(rc, "dinoseg_embeddings")
        if avgpool:
            return torch.stack((cls[0], mean), dim=-1).reshape(b, -1)
        return cls.permute(1, 0, 2).reshape(b, n_out * d)

    @torch.no_grad()
    def features(self, x, n=1, resolution=None):
        """Backbone features of the last n blocks in one pass (no head): a device fp32 tensor [min(n, n_blocks), B, N, D],
        N = (H/8)*(W/8) + 1 with the CLS token first, then the patches row by row; slice k is the final norm (dino.norm)
        of the residual stream after block n_blocks - min(n, n_blocks) + k (vision_transformer.py:282-290).  x: device
        fp32 [B,3,H,W] (normalised), or device uint8 [B,Hs,Ws,3] raw RGB frames resized to `resolution` (an int r or an
        (H, W) pair; default self.resolution) and normalised as in infer_u8.  Asynchronous on the current stream."""
        if not isinstance(n, numbers.Integral) or n < 1:
            raise ValueError(f"n must be a positive integer, got {n!r}")
        n = int(n)
        lib = self._ensure_handle()
        if x.device != self.device:
            raise ValueError(f"frames are on {x.device}, model on {self.device}")
        raw = x.dtype == torch.uint8
        if raw:
            if x.dim() != 4 or x.shape[3] != 3:
                raise ValueError(f"expected uint8 frames of shape [B,H,W,3], got {tuple(x.shape)}")
            hw = _resolution_hw(self.resolution if resolution is None else resolution)
        else:
            hw = _frame_hw(x)
            if resolution is not None and _resolution_hw(resolution) != hw:
                raise ValueError(f"resolution {resolution} given for frames of size {hw[0]}x{hw[1]}")
            x = x.float()
        x = x.contiguous()
        b = int(x.shape[0])
        self._ensure_resolution(lib, hw)
        ws = self._ensure_workspace(lib, b)
        n_out = min(n, self.n_blocks)
        n_tok = (hw[0] // 8) * (hw[1] // 8) + 1
        out = torch.empty((n_out, b, n_tok, self.mlp_input_dim), dtype=torch.float32, device=self.device)
        if raw:
            mean = (C.c_float * 3)(*IMAGENET_MEAN)
            std = (C.c_float * 3)(*IMAGENET_STD)
            rc = lib.dinoseg_features_u8(self._handle, x.data_ptr(), b, int(x.shape[1]), int(x.shape[2]), mean, std, n,
                                         out.data_ptr(), ws.data_ptr(), ws.numel(), self._stream())
            self._check(rc, "dinoseg_features_u8")
        else:
            rc = lib.dinoseg_features(self._handle, x.data_ptr(), b, n, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                      self._stream())
            self._check(rc, "dinoseg_features")
        return out

    def forward(self, x):
        """pl_torch_modules.py:239-256: [B,3,H,W] -> per-patch log-probabilities [B*P, C], P = (H/8)*(W/8)."""
        return self.infer(x, want_logprobs=True)[0]

    def predict(self, x):
        """Run inference on a single image (pl_torch_modules.py:276-300).

        x : PIL.Image (or HxWx3 uint8 array).  Returns an int64 ndarray of shape
        [g*p, g*p] (480x480 for resolutions 240/480/960).

        The reference's transforms (Resize -> Normalize -> ToTensorV2, :33-41) run on the GPU, fused into the
        patch-embed im2col (bit-exact w.r.t. cv2.resize(INTER_LINEAR) + the fp32 normalisation); `self.transforms`
        stays available for callers that use it directly (visualize_attention.py:45)."""
        img = np.asarray(x)
        if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
            # not a plain RGB uint8 image: host transforms + fp32 path, as the reference does
            t = self.transforms(image=img)['image']
            _, _, lab = self.infer(t.unsqueeze(0).to(self.device), want_logprobs=False, want_labels=True)
            return lab[0].cpu().numpy()
        frames = torch.from_numpy(np.array(img, copy=True)).unsqueeze(0).to(self.device)
        _, _, lab = self.infer_u8(frames, self.resolution, want_logprobs=False, want_labels=True)
        return lab[0].cpu().numpy()

    @torch.no_grad()
    def infer_u8(self, frames_u8, resolution=None, want_logprobs=True, want_lowres=False, want_labels=False):
        """Hot path on RAW device frames: uint8 [B,Hs,Ws,3] RGB (any Hs, Ws) -> resize to `resolution` (an int r for
        r x r, or an (H, W) pair: cv2.resize(img, (W, H)) semantics), normalise (ImageNet), forward.  Returns
        (logprobs, lowres, labels) like infer(); labels only for a square resolution."""
        lib = self._ensure_handle()
        if frames_u8.dim() != 4 or frames_u8.shape[3] != 3 or frames_u8.dtype != torch.uint8:
            raise ValueError(f"expected uint8 frames of shape [B,H,W,3], got {tuple(frames_u8.shape)} {frames_u8.dtype}")
        if frames_u8.device != self.device:
            raise ValueError(f"frames are on {frames_u8.device}, model on {self.device}")
        hw = _resolution_hw(self.resolution if resolution is None else resolution)
        self._check_labels_square(hw, want_labels)
        frames_u8 = frames_u8.contiguous()
        b, sh, sw = int(frames_u8.shape[0]), int(frames_u8.shape[1]), int(frames_u8.shape[2])
        self._ensure_resolution(lib, hw)
        ws = self._ensure_workspace(lib, b)
        lp, low, lab = self._outputs(b, hw, want_logprobs, want_lowres, want_labels)
        mean = (C.c_float * 3)(*IMAGENET_MEAN)
        std = (C.c_float * 3)(*IMAGENET_STD)
        rc = lib.dinoseg_forward_u8(self._handle, frames_u8.data_ptr(), b, sh, sw, mean, std,
                                    lp.data_ptr() if lp is not None else None,
                                    low.data_ptr() if low is not None else None,
                                    lab.data_ptr() if lab is not None else None,
                                    ws.data_ptr(), ws.numel(), self._stream())
        self._check(rc, "dinoseg_forward_u8")
        return lp, low, lab

    # -------------------------------------------------------------------------------------
    # host frames -> host label maps (the library's pipelined host entry points)
    # -------------------------------------------------------------------------------------
    def _host_out(self, b, g, output, out):
        p = 480 // g
        shape, dtype = ((b, g * p, g * p), torch.int64) if output == "labels" else ((b, g, g), torch.uint8)
        if out is None:
            out = torch.empty(shape, dtype=dtype, pin_memory=torch.cuda.is_available())
        elif tuple(out.shape) != shape or out.dtype != dtype or out.device.type != "cpu" or not out.is_contiguous():
            raise ValueError(f"out must be a contiguous CPU tensor of shape {shape} and dtype {dtype}")
        return out

    def _submit_host(self, frames, resolution, output, out):
        """Enqueue one host batch (fp32 [B,3,r,r] normalised, or uint8 [B,H,W,3] raw) -> ticket."""
        if output not in ("labels", "lowres"):
            raise ValueError(output)
        lib = self._ensure_handle()
        if frames.device.type != "cpu":
            raise ValueError("expected CPU frames")
        if isinstance(resolution, (tuple, list)):
            raise ValueError(f"the host entry points take a square resolution (an int), got {resolution!r}")
        if frames.dtype == torch.uint8:
            if frames.dim() != 4 or frames.shape[3] != 3:
                raise ValueError("expected CPU uint8 frames of shape [B,H,W,3]")
            frames = frames.contiguous()
            res = int(self.resolution if resolution is None else resolution)
            b, sh, sw = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
        else:
            if frames.dim() != 4 or frames.shape[1] != 3 or frames.shape[2] != frames.shape[3]:
                raise ValueError(f"expected frames of shape [B,3,r,r], got {tuple(frames.shape)}")
            frames = frames.contiguous().float()
            b, res = int(frames.shape[0]), int(frames.shape[2])
        self._ensure_resolution(lib, (res, res))
        out = self._host_out(b, res // 8, output, out)
        low_ptr = out.data_ptr() if output == "lowres" else None
        lab_ptr = out.data_ptr() if output == "labels" else None
        if frames.dtype == torch.uint8:
            mean = (C.c_float * 3)(*IMAGENET_MEAN)
            std = (C.c_float * 3)(*IMAGENET_STD)
            t = lib.dinoseg_predict_host_submit_u8(self._handle, frames.data_ptr(), b, sh, sw, mean, std, low_ptr, lab_ptr,
                                                   self._stream())
        else:
            t = lib.dinoseg_predict_host_submit(self._handle, frames.data_ptr(), b, low_ptr, lab_ptr, self._stream())
        if t <= 0:
            raise RuntimeError("dinoseg_predict_host_submit failed: " + _lib.last_error(self._handle))
        self._pending[t] = (frames, out)          # the library reads / writes these buffers until predict_wait(t)
        return t

    def predict_batch_async(self, frames, resolution=None, output="labels", out=None):
        """Asynchronous predict_batch for a caller that streams batches (camera, folder of images): enqueue the batch
        and return a ticket at once; `predict_wait(ticket)` returns the numpy result.  Up to 4 batches may be in
        flight; the H2D copy of one overlaps the kernels and the D2H copy of the one before.  frames: CPU fp32
        [B,3,r,r] (normalised) or CPU uint8 [B,H,W,3] (raw; resized to `resolution` and normalised on the GPU);
        `frames` and `out` must not be modified before predict_wait returns."""
        return self._submit_host(frames, resolution, output, out)

    def predict_wait(self, ticket):
        """Wait for a predict_batch_async submission -> numpy result (int64 [B,g*p,g*p] or uint8 [B,g,g])."""
        if ticket not in self._pending:
            raise KeyError(f"unknown ticket {ticket} (already waited for?)")
        rc = _lib.load().dinoseg_predict_host_wait(self._handle, int(ticket))
        _, out = self._pending.pop(ticket)
        self._check(rc, "dinoseg_predict_host_wait")
        return out.numpy()

    def predict_batch_u8(self, frames_u8, resolution=None, output="labels", out=None):
        """Batched predict() on raw HOST frames: uint8 [B,H,W,3] (ideally pinned) -> numpy label maps; resize,
        normalisation, forward, argmax and replication on the GPU, copies pipelined with the kernels."""
        if frames_u8.dtype != torch.uint8 or frames_u8.device.type != "cpu":
            raise ValueError("expected CPU uint8 frames of shape [B,H,W,3]")
        return self.predict_wait(self._submit_host(frames_u8, resolution, output, out))

    def predict_batch(self, frames, output="labels", out=None):
        """Batched counterpart of predict() for already-normalised frames [B,3,r,r].

        Device frames -> device result (asynchronous).  Host frames (ideally pinned) go through
        the library's host entry point, which pipelines H2D copy / kernels / D2H copy over chunks of
        the batch and synchronises -> numpy result.  output: 'labels' (int64 [B,g*p,g*p]) or 'lowres'
        (uint8 [B,g,g]).  out: optional preallocated (pinned) host tensor to receive the result."""
        if output not in ("labels", "lowres"):
            raise ValueError(output)
        if frames.device.type == "cuda":
            _, low, lab = self.infer(frames, want_logprobs=False, want_lowres=output == "lowres",
                                     want_labels=output == "labels")
            return lab if output == "labels" else low
        if frames.dtype == torch.uint8:
            raise ValueError("uint8 frames go through predict_batch_u8")
        return self.predict_wait(self._submit_host(frames, None, output, out))

    def profile_enable(self, on=True, kinds=None):
        """Bracket kernel launches of the following forwards with CUDA events (on the launching
        stream).  kinds: iterable of kernel-kind names to restrict the events to (None = all)."""
        lib = self._ensure_handle()
        mask = 0xffffffff
        if kinds is not None:
            names = [lib.dinoseg_profile_kind_name(i).decode() for i in range(lib.dinoseg_profile_num_kinds())]
            mask = 0
            for k in kinds:
                mask |= 1 << names.index(k)
        self._check(lib.dinoseg_profile_set_mask(self._handle, mask), "dinoseg_profile_set_mask")
        self._check(lib.dinoseg_profile_enable(self._handle, 1 if on else 0), "dinoseg_profile_enable")

    def profile_read(self):
        """-> {kernel kind: (total ms, launches)} accumulated since enable / the last read."""
        lib = self._ensure_handle()
        n = lib.dinoseg_profile_num_kinds()
        ms = (C.c_float * n)()
        cnt = (C.c_int * n)()
        self._check(lib.dinoseg_profile_read(self._handle, ms, cnt, n), "dinoseg_profile_read")
        return {lib.dinoseg_profile_kind_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n) if cnt[i]}

    def profile_gaps(self):
        """-> (span ms, gap ms) of the launches recorded since enable / the last read: first start -> last end, and the part
        of it between launches.  Call BEFORE profile_read (which resets the record)."""
        lib = self._ensure_handle()
        span, gap = C.c_float(0.0), C.c_float(0.0)
        self._check(lib.dinoseg_profile_gaps(self._handle, C.byref(span), C.byref(gap)), "dinoseg_profile_gaps")
        return float(span.value), float(gap.value)

    def last_launch_count(self):
        return _lib.load().dinoseg_last_launch_count(self._handle) if self._handle is not None else 0

    # -------------------------------------------------------------------------------------
    # training side of the reference: out of scope of this build (SURVEY.md §2-2c)
    # -------------------------------------------------------------------------------------
    def fit(self, *a, **k):
        raise NotImplementedError("training is out of scope of the B200 inference build")

    def freeze_bb(self):
        for p in self.dino.parameters():
            p.requires_grad = False

    def unfreeze_bb(self):
        warnings.warn("the B200 build is inference-only; gradients are never computed")
