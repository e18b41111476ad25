"""Mixed-length (ragged) batches: BASELINE.json config 5.

The reference has no padding masks -- ``DiT.forward`` attends over every frame it is given (src/components/DiT.py:131-148)
and ``SpeechGenerator.__sample_latents`` (src/model/SpeechGenerator.py:150-164) draws ``[1, L_pred, 768]`` per utterance --
so utterances of different length only match it when they run UNPADDED.  A ``RaggedBatch`` sorts the utterances into
groups of equal (frames, text tokens), packs their rows back to back and hands the group list to
``ditto_forward_ragged`` / ``ditto_p_sample_ragged_known`` (include/ditto_b200.h): the row-wise work (LayerNorms, QKV / GLU /
fc2 / projection GEMMs) is ONE launch over all packed rows, only AdaLN modulation, RoPE positions and the two
attentions run per group.  Nothing is padded, so no flop is spent on frames that do not exist.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import DittoError
from .model import DiTTO, _check_text_lengths, _need_cuda_f32, _ptr, _stream
from .sampler import _CapturedStep

__all__ = ["RaggedBatch", "RaggedStepGraph"]


class RaggedBatch:
    """Group list + text contexts + packing order of a mixed-length batch of B utterances.

    ``texts[i]`` is ``[S_i, text_dim]`` (CUDA fp32), ``lengths[i]`` the latent frame count T_i.  With ``guided`` each
    group holds its conditional sequences followed by the unconditional ones (zero text embedding unless
    ``null_texts`` supplies them), sharing the group's latents.  ``text_lengths[i]`` in [1, S_i]: utterance i (and its
    unconditional branch) uses text rows [0, text_lengths[i]) only.  Groups stay keyed on ``texts[i].shape[0]``: padding texts
    to a few widths makes them share groups, and the lengths, being data in the group's context, change no graph."""

    @staticmethod
    def signature(texts, lengths, guided: bool):
        """What a captured step graph depends on: the sorted (frames, tokens) pairs, guidance, device."""
        keys = sorted((int(t), int(x.shape[0])) for t, x in zip(lengths, texts))
        return (tuple(keys), bool(guided), str(texts[0].device) if len(texts) else "")

    def __init__(self, model: DiTTO, texts: Sequence[torch.Tensor], lengths: Sequence[int], guided: bool = False,
                 null_texts: Optional[Sequence[torch.Tensor]] = None, name: str = "ragged",
                 ctx_storage: Optional[List[torch.Tensor]] = None, text_lengths=None):
        if len(texts) == 0 or len(texts) != len(lengths):
            raise DittoError("RaggedBatch needs one text embedding and one length per utterance")
        self.model, self.guided = model, guided
        self.B = len(texts)
        texts = [_need_cuda_f32(f"texts[{i}]", x) for i, x in enumerate(texts)]
        for i, x in enumerate(texts):
            if x.dim() != 2 or x.shape[1] != model.text_dim or x.shape[0] < 1:
                raise DittoError(f"texts[{i}] must be [S, {model.text_dim}] with S >= 1")
        text_lengths = _check_text_lengths(text_lengths, [int(x.shape[0]) for x in texts])
        self.lengths = [int(v) for v in lengths]
        if min(self.lengths) < 1 or max(self.lengths) > model.max_seq_len:
            raise DittoError("every length must be in [1, max_seq_len]")
        self.device = texts[0].device
        keys = [(self.lengths[i], int(texts[i].shape[0])) for i in range(self.B)]
        self.order = sorted(range(self.B), key=lambda i: (keys[i], i))      # packed position -> utterance index
        self.groups = []                                                   # (T, S, [utterance indices])
        for i in self.order:
            if self.groups and self.groups[-1][:2] == keys[i]:
                self.groups[-1][2].append(i)
            else:
                self.groups.append((keys[i][0], keys[i][1], [i]))
        H = model.hidden_dim
        mult = 2 if guided else 1
        self.x_rows = sum(self.lengths)                                     # packed latent rows
        self.n_seq = mult * self.B
        self.seq_rows = mult * self.x_rows
        # per-group text contexts (step-invariant) and the C group table
        self._ctx = []
        arr = (_lib.SeqGroup * len(self.groups))()
        self.x_offset = {}                                                  # utterance -> first packed x row
        row = 0
        for gi, (T, S, idx) in enumerate(self.groups):
            tg = torch.stack([texts[i] for i in idx])
            if guided:
                null = torch.zeros_like(tg) if null_texts is None else torch.stack(
                    [_need_cuda_f32("null_texts", null_texts[i]) for i in idx])
                if null.shape != tg.shape:
                    raise DittoError("null_texts must match texts in shape")
                tg = torch.cat([tg, null], dim=0)
            lens = None
            if text_lengths is not None:
                lens = [text_lengths[i] for i in idx] * (2 if guided else 1)
            ctx = model.text_context(tg, name="ragged_ctx", T_hint=1, text_lengths=lens)
            if ctx_storage is not None:       # buffers a cached step graph reads (same batch signature): refill in place
                store = ctx_storage[gi]
                k = min(store.numel(), ctx.numel())   # both hold at least ditto_text_context_bytes of this group
                store[:k].copy_(ctx[:k])
                ctx = store
            else:
                ctx = ctx.clone()             # owned by this batch (offset-based layout)
            self._ctx.append(ctx)
            arr[gi] = _lib.SeqGroup(n_seq=mult * len(idx), n_x=len(idx), T=T, S=S, ctx=ctx.data_ptr())
            for i in idx:
                self.x_offset[i] = row
                row += T
        self.c_groups = arr
        nbytes = _lib.load().ditto_workspace_bytes_ragged(model.engine(), arr, len(self.groups))
        if nbytes < 0:
            raise DittoError("ditto_workspace_bytes_ragged: bad group list")
        self.ws_bytes = int(nbytes)
        self.H = H

    # -------------------------------------------------------------------------------------- layout helpers
    def workspace(self) -> torch.Tensor:
        return self.model._bufs.get("ws", self.ws_bytes, self.device)

    def pack(self, xs: Sequence[torch.Tensor]) -> torch.Tensor:
        """[T_i, H] per utterance -> packed [sum T, H] in group order."""
        if len(xs) != self.B:
            raise DittoError("one latent per utterance expected")
        out = torch.empty((self.x_rows, self.H), dtype=torch.float32, device=self.device)
        for i, x in enumerate(xs):
            x = _need_cuda_f32(f"x[{i}]", x)
            if tuple(x.shape) != (self.lengths[i], self.H):
                raise DittoError(f"x[{i}] must be [{self.lengths[i]}, {self.H}]")
            out[self.x_offset[i]:self.x_offset[i] + self.lengths[i]] = x
        return out

    def pack_mask(self, masks: Sequence[torch.Tensor]) -> torch.Tensor:
        """[T_i] frame mask per utterance -> packed uint8 [sum T] in group order (one byte per packed latent row)."""
        if len(masks) != self.B:
            raise DittoError("one mask per utterance expected")
        out = torch.empty((self.x_rows,), dtype=torch.uint8, device=self.device)
        for i, q in enumerate(masks):
            if tuple(q.shape) != (self.lengths[i],):
                raise DittoError(f"mask[{i}] must be [{self.lengths[i]}]")
            out[self.x_offset[i]:self.x_offset[i] + self.lengths[i]] = q != 0
        return out

    def pack_seeds(self, seeds: Sequence[int]) -> torch.Tensor:
        """One seed per utterance (checked ints in [0, 2^64)) -> int64 [B] bit patterns in group order, the order of the
        groups' latents (ditto_p_sample_ragged_per_utt)."""
        from .sampler import _seed_tensor
        return _seed_tensor([seeds[i] for i in self.order], self.device)

    def pack_w(self, w: Sequence[float]) -> torch.Tensor:
        """One guidance scale per utterance -> fp32 [B] in group order."""
        return torch.tensor([float(w[i]) for i in self.order], dtype=torch.float32).to(self.device)

    def row0(self) -> torch.Tensor:
        """First packed latent row of every utterance in group order, then x_rows: the row table of ditto_randn_latents."""
        return torch.tensor([self.x_offset[i] for i in self.order] + [self.x_rows], dtype=torch.int64).to(self.device)

    def unpack(self, packed: torch.Tensor) -> List[torch.Tensor]:
        return [packed[self.x_offset[i]:self.x_offset[i] + self.lengths[i]].clone() for i in range(self.B)]

    def seq_t(self, t: torch.Tensor) -> torch.Tensor:
        """per-utterance t [B] -> per-sequence t in packed sequence order ([cond; uncond] per group when guided)."""
        t = t.to(device=self.device, dtype=torch.int64)
        parts = []
        for _, _, idx in self.groups:
            tg = t[torch.tensor(idx, device=self.device)]
            parts.append(torch.cat([tg, tg]) if self.guided else tg)
        return torch.cat(parts).contiguous()

    def unpack_eps(self, eps: torch.Tensor, w) -> List[torch.Tensor]:
        """packed sequence-layout output -> per-utterance eps_hat (guided: the CFG combine, as ditto_cfg_ddpm_update; ``w`` a
        scalar or one scale per utterance)."""
        out = [None] * self.B
        row = 0
        for T, _, idx in self.groups:
            n = len(idx)
            blk = eps[row:row + (2 if self.guided else 1) * n * T].view(-1, T, self.H)
            for j, i in enumerate(idx):
                wi = w[i] if isinstance(w, (list, tuple)) else w
                out[i] = (blk[n + j] + wi * (blk[j] - blk[n + j])) if self.guided else blk[j].clone()
            row += blk.shape[0] * T
        return out

    # -------------------------------------------------------------------------------------- device calls
    def forward(self, x_packed: torch.Tensor, t_seq: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty((self.seq_rows, self.H), dtype=torch.float32, device=self.device)
        ws = self.workspace()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().ditto_forward_ragged(self.model.engine(), _ptr(x_packed), self.c_groups, len(self.groups),
                                                        _ptr(t_seq), _ptr(out), _ptr(ws), ws.numel(), _stream()),
                       "ditto_forward_ragged")
        return out

    def p_sample(self, x_packed, t_seq, z_packed, w: float, eps: torch.Tensor, x_out: torch.Tensor, ws=None, hist=None,
                 known=None, mask=None, rng=None, seeds=None, w_dev=None, advance=None):
        """One sampler step (ditto_p_sample_ragged_per_utt); ``hist`` (packed like x): the multistep update; ``known`` /
        ``mask`` (packed like x / one byte per packed row): known frames; ``rng``: noise drawn in the per-group update kernels
        instead of ``z_packed``, and (unless ``advance`` is False) the "t -= 1" bookkeeping in a one-block kernel after them.
        ``seeds`` / ``w_dev`` [B] in group order (pack_seeds / pack_w): per-utterance noise keys (with rng) and scales."""
        ws = self.workspace() if ws is None else ws
        if advance is None:
            advance = rng is not None
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().ditto_p_sample_ragged_per_utt(self.model.engine(), _ptr(x_packed), self.c_groups, len(self.groups),
                                                                 _ptr(t_seq), _ptr(z_packed), _ptr(rng), _ptr(seeds),
                                                                 1 if self.guided else 0, float(w), _ptr(w_dev), _ptr(eps), _ptr(x_out),
                                                                 _ptr(hist), _ptr(known), _ptr(mask), _ptr(ws), ws.numel(),
                                                                 1 if advance else 0, _stream()),
                       "ditto_p_sample_ragged_per_utt")


class RaggedStepGraph(_CapturedStep):
    """One sampler iteration over a ragged batch as a CUDA graph (noise draw, forward, CFG + update, t decrement).  With
    ``multistep`` the update is DPM-Solver++(2M)'s and the graph owns its ``hist`` buffer (packed like x).  With ``known``
    it owns the known latents (packed like x) and the frame mask (one byte per packed row), filled by ``reset``.  A guided
    graph reads one guidance scale per utterance (group order) from ``w_dev`` (``set_scale``); a ``seeded`` one keys each
    utterance's noise by its entry of ``seeds`` (group order, filled by ``reset``)."""

    def __init__(self, batch: RaggedBatch, w, draw_noise: bool, multistep: bool = False, known: bool = False,
                 seeded: bool = False):
        self.batch = batch
        dev = batch.device
        self._buffers((batch.x_rows, batch.H), batch.n_seq, draw_noise, multistep, known, dev, batch.B, batch.guided, seeded)
        self.set_scale(w)
        self._ctx_ptrs = [c.data_ptr() for c in batch._ctx]
        self.eps = torch.empty((batch.seq_rows, batch.H), dtype=torch.float32, device=dev)
        self.ws = batch.workspace()
        self._capture(dev)

    def _p_sample(self, rng):
        self.batch.p_sample(self.x, self.t, self.z, 0.0, self.eps, self.x, ws=self.ws, hist=self.hist, known=self.known,
                            mask=self.mask, rng=rng, seeds=self.seeds, w_dev=self.w_dev)

    def valid_for(self, batch: "RaggedBatch") -> bool:
        """The captured kernels read the context buffers and the workspace by address."""
        return (self._ctx_ptrs == [c.data_ptr() for c in batch._ctx] and self.ws.data_ptr() == batch.workspace().data_ptr()
                and batch.x_rows == self.x.shape[0])

    def rebind(self, batch: "RaggedBatch"):
        self.batch = batch
