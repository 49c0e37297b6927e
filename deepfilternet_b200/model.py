"""Host-side mirror of the reference's ``DfNet`` (deepfilternet3.py:334-456, deepfilternet2.py:374-505, deepfilternet.py:232-279).

``DfNet`` keeps the reference module's public surface -- ``forward(spec, feat_erb, feat_spec) ->
(spec_e, m, lsnr, df_coefs | df_alpha)``, ``state_dict()``, ``eval()``, the attributes ``nb_df`` /
``df_order`` / ``df_lookahead`` -- but owns no torch compute: the forward pass runs in the CUDA
kernels of libdfb200.so (csrc/dfb_model.cu) through the C ABI.  torch is used for tensors
(device memory, streams) only.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import re
from typing import Dict, Optional, Tuple, Union

import numpy as np
import torch
from torch import Tensor, nn

from . import _lib
from ._lib import ModelConfigC, TensorC, check
from .config import ModelConfig, load_config
from .libdf import DF
from .weights import pack_state_dict


def _epoch_of(cp: str) -> int:
    return int(os.path.basename(cp).split(".")[0].split("_")[-1])  # checkpoint.py:17-18


def find_checkpoint(dirname: str, epoch: Union[str, int, None] = "best", name: str = "model",
                    extension: str = "ckpt") -> Tuple[Optional[str], Optional[int]]:
    """Checkpoint selection of ``read_cp`` (checkpoint.py:46-75)."""
    checkpoints = []
    if isinstance(epoch, str):
        assert epoch in ("best", "latest")
    if epoch == "best":
        checkpoints = glob.glob(os.path.join(dirname, f"{name}*.{extension}.best"))
    if len(checkpoints) == 0:
        checkpoints = glob.glob(os.path.join(dirname, f"{name}*.{extension}"))
        checkpoints += glob.glob(os.path.join(dirname, f"{name}*.{extension}.best"))
    if len(checkpoints) == 0:
        return None, None
    if isinstance(epoch, int):
        latest = next((x for x in checkpoints if _epoch_of(x) == epoch), None)
        if latest is None:
            raise FileNotFoundError(f"Could not find checkpoint of epoch {epoch}")
    else:
        latest = max(checkpoints, key=_epoch_of)
        epoch = _epoch_of(latest)
    return latest, int(epoch)


def load_state_dict_file(path: str) -> Dict[str, Tensor]:
    sd = torch.load(path, map_location="cpu", weights_only=True)
    return {k.replace("clc", "df"): v for k, v in sd.items()}  # checkpoint.py:78


class DfNet(nn.Module):
    """B200 drop-in for ``df.deepfilternet3.DfNet`` / ``df.deepfilternet2.DfNet`` / ``df.deepfilternet.DfNet``."""

    def __init__(self, cfg: ModelConfig, state_dict: Dict[str, Tensor], df_state: Optional[DF] = None,
                 device: Optional[int] = None, run_df: bool = True):
        super().__init__()
        self.cfg = cfg
        self.nb_df = cfg.nb_df
        self.df_bins = cfg.nb_df
        self.df_order = cfg.df_order
        self.df_lookahead = cfg.df_lookahead
        self.freq_bins = cfg.freq_bins
        self.erb_bins = cfg.nb_erb
        self.run_df = bool(run_df)            # False: init_df(mask_only=True) (checkpoint.py:32)
        self.post_filter = bool(cfg.mask_pf)  # init_df(post_filter=True) sets mask_pf (enhance.py:152-153)
        self.post_filter_beta = float(cfg.pf_beta)
        self._device = 0 if device is None else int(device)
        self.df_state = df_state if df_state is not None else DF(
            cfg.sr, cfg.fft_size, cfg.hop_size, cfg.nb_erb, cfg.min_nb_erb_freqs, device=self._device)
        if self.df_state.device != self._device:
            raise ValueError("df_state lives on a different device than the model")
        if (self.df_state.nb_erb() != cfg.nb_erb or self.df_state.fft_size() != cfg.fft_size
                or self.df_state.hop_size() != cfg.hop_size):
            raise ValueError("df_state was built with a different nb_erb / fft_size / hop_size than the model config")
        if cfg.nb_df > cfg.fft_size // 2 + 1:
            raise _lib.DfbError(_lib.DFB_ERR_INVALID, f"nb_df = {cfg.nb_df} exceeds the {cfg.fft_size // 2 + 1} frequency "
                                                      f"bins of fft_size {cfg.fft_size}")
        self.df_state.norm_alpha = cfg.norm_alpha  # read by df_features (enhance.py:192)
        # keep the reference tensors (state_dict() parity); buffers, not parameters: inference only
        self._sd_names = []
        for k, v in state_dict.items():
            if not torch.is_tensor(v):
                continue
            name = "sd__" + re.sub(r"[^0-9a-zA-Z_]", "__", k)
            self.register_buffer(name, v.detach().clone(), persistent=False)
            self._sd_names.append((k, name))
        packed, derived = pack_state_dict(state_dict, cfg)
        self._packed = packed  # host copies must outlive dfb_model_create only; kept for introspection
        cc = ModelConfigC()
        for k, v in derived.items():
            setattr(cc, k, v)
        cc.norm_alpha = cfg.norm_alpha
        names = [n.encode() for n in packed]
        arr = (TensorC * len(packed))()
        for i, (n, a) in enumerate(packed.items()):
            arr[i].name = names[i]
            arr[i].data = a.ctypes.data_as(C.POINTER(C.c_float))
            arr[i].numel = a.size
        widths = np.ascontiguousarray(self.df_state.erb_widths().astype(np.int64))
        h = C.c_void_p()
        check(_lib.lib().dfb_model_create(C.byref(h), self._device, C.byref(cc), arr, len(packed),
                                          widths.ctypes.data_as(C.POINTER(C.c_int64))))
        self._h = h
        self._derived = derived
        self.set_precision(os.environ.get("DFB_PRECISION", "fp32+gru_tc+proj_tc+conv_tc"))
        check(_lib.lib().dfb_model_set_options(self._h, int(self.post_filter), self.post_filter_beta, int(not self.run_df)))

    def set_precision(self, mode: str) -> None:
        """Arithmetic of the contractions (everything else is always IEEE fp32):
          'fp32'         FFMA everywhere
          'fp32+gru_tc'  the GRU recurrence of H = 256 models on tcgen05 tensor cores with BF16 hi/lo split
                         operands (3 MMAs per product, fp32 accumulate: ~2^-17 relative, 5e-8 RMS end to end)
          'fp32+gru_tc+proj_tc'  plus the GRU input projections on the BF16x3 tcgen05 GEMM
          'fp32+gru_tc+proj_tc+conv_tc'  (default) plus the 1x1 convs of the separable conv blocks (k_dwpw_bx) and
                         the grouped linears (k_gl_bx) on BF16x3 tcgen05 kernels (1e-7 .. 4e-7 RMS end to end)."""
        modes = {"fp32": 0, "fp32+gru_tc": 2, "fp32+gru_tc+proj_tc": 6, "fp32+gru_tc+proj_tc+conv_tc": 14}
        if mode not in modes:
            raise ValueError(f"unknown precision mode {mode!r}; one of {sorted(modes)}")
        check(_lib.lib().dfb_model_set_precision(self._h, modes[mode]))
        self.precision = mode

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                _lib.lib().dfb_model_free(h)
            except Exception:
                pass
            object.__setattr__(self, "_h", None)   # (nn.Module.__setattr__ is unusable during interpreter shutdown)

    # -- nn.Module surface ---------------------------------------------------------------
    def state_dict(self, *args, **kwargs):  # reference tensor names
        return {k: getattr(self, n) for k, n in self._sd_names}

    def to(self, *args, **kwargs):  # weights already live on the B200; keep the reference call working
        return self

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    @property
    def cuda_device(self) -> torch.device:
        return torch.device("cuda", self._device)

    def set_max_workspace(self, nbytes: int) -> None:
        """Cap of the per-call device workspace of enhance(): larger batches are processed in stream groups."""
        check(_lib.lib().dfb_model_set_max_workspace(self._h, int(nbytes)))

    def set_chunking(self, device_chunks: int = 0, host_chunks: int = 4, lanes: int = 2) -> None:
        """Chunk pipeline of enhance(): minimum number of time chunks for long signals (device / host entry point) and
        whether consecutive chunks overlap on two lanes (2) or run back to back (1)."""
        check(_lib.lib().dfb_model_set_chunking(self._h, int(device_chunks), int(host_chunks), int(lanes)))

    def workspace_bytes(self) -> int:
        return int(_lib.lib().dfb_model_workspace_bytes(self._h))

    # -- forward ---------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, spec: Tensor, feat_erb: Tensor, feat_spec: Tensor):
        """Same contract as the reference (deepfilternet3.py:389-456):
        spec [B,1,T,F,2], feat_erb [B,1,T,E], feat_spec [B,1,T,Fd,2] ->
        (spec_e [B,1,T,F,2], m [B,1,T,E], lsnr [B,T,1], df_coefs [B,O,T,Fd,2] | df_alpha [B,T,1])."""
        dev_in = spec.device
        dev = self.cuda_device
        b, _, t, f, _ = spec.shape
        e, fd, o = self.cfg.nb_erb, self.cfg.nb_df, self.cfg.df_order
        if f != self.freq_bins or feat_erb.shape[-1] != e or feat_spec.shape[-2] != fd:
            raise RuntimeError("DF shape error: unexpected feature dimensions")
        sp = spec.to(dev, torch.float32).contiguous()
        fe = feat_erb.to(dev, torch.float32).contiguous()
        fs = feat_spec.to(dev, torch.float32).contiguous()
        spec_e = torch.empty_like(sp)
        m = torch.empty((b, 1, t, e), device=dev, dtype=torch.float32)
        lsnr = torch.empty((b, t, 1), device=dev, dtype=torch.float32)
        coefs = torch.empty((b, t, fd, 2 * o), device=dev, dtype=torch.float32)
        has_alpha = self.cfg.model in ("deepfilternet", "deepfilternet2")   # deepfilternet.py:279, deepfilternet2.py:505
        alpha = torch.empty((b, t, 1), device=dev, dtype=torch.float32) if has_alpha else None
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            check(_lib.lib().dfb_model_forward_full(
                self._h, self.df_state.handle, sp.data_ptr(), fe.data_ptr(), fs.data_ptr(), b, t,
                spec_e.data_ptr(), m.data_ptr(), lsnr.data_ptr(), coefs.data_ptr(),
                alpha.data_ptr() if alpha is not None else None, stream))
        if has_alpha:
            last = alpha if self.run_df else torch.zeros_like(alpha)   # deepfilternet.py:277-278
        else:  # DfOutputReshapeMF, deepfilternet3.py:268-275
            last = coefs.view(b, t, fd, o, 2).permute(0, 3, 1, 2, 4)
        outs = (spec_e, m, lsnr, last)
        if dev_in != dev:
            outs = tuple(x.to(dev_in) for x in outs)
        return outs


def load_model(model_base_dir: str, epoch: Union[str, int, None] = "best", device: int = 0,
               df_state: Optional[DF] = None, env: Optional[dict] = None, post_filter: bool = False,
               mask_only: bool = False) -> Tuple[DfNet, DF, int]:
    """init_model + read_cp for a reference model directory (``config.ini`` + ``checkpoints/``)."""
    cfg = load_config(os.path.join(model_base_dir, "config.ini"), env=env)
    if post_filter:
        cfg.mask_pf = True
    cp_dir = os.path.join(model_base_dir, "checkpoints")
    path, ep = find_checkpoint(cp_dir, epoch)
    if path is not None:
        sd = load_state_dict_file(path)
    else:
        from .onnx_import import state_dict_from_onnx_dir  # _ll ships only as ONNX
        sd = state_dict_from_onnx_dir(model_base_dir, cfg)
        ep = 0
        if sd is None:
            raise FileNotFoundError(f"Could not find a checkpoint in {cp_dir}")
    if df_state is None:
        df_state = DF(cfg.sr, cfg.fft_size, cfg.hop_size, cfg.nb_erb, cfg.min_nb_erb_freqs, device=device)
    model = DfNet(cfg, sd, df_state, device=device, run_df=not mask_only)
    return model, df_state, int(ep)
