"""Host-side mirror of the reference's DiT modules (src/model/DiTTO.py, src/components/DiT.py).

Same class names, constructor arguments, parameter names (state_dict keys) and call signatures as the
reference, so a ``TrainDiTTO.py``-style inference script can switch by changing the import.  The modules
are PARAMETER CONTAINERS: their arithmetic runs in libditto_b200.so (hand-written sm_100a CUDA behind the
C-ABI of include/ditto_b200.h).  Inference only; no autograd; no CPU fallback (CPU tensors raise).
"""
from __future__ import annotations

import ctypes as C
import operator
import weakref
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import DittoError

__all__ = ["DiTTO", "DiT", "GlobalAdaLN", "RotaryEmbedding", "DittoError"]


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_t_range(t: torch.Tensor, steps: int, what: str):
    """The reference's ``t_embedding(t)`` / ``betas[t]`` raise on an out-of-range index; the kernels clamp (the captured step
    graph leaves t = -1 after its last step), so the eager API checks on the host (one small device->host read)."""
    if t.numel() == 0:
        return
    lo, hi = int(t.min()), int(t.max())
    if lo < 0 or hi >= steps:
        raise DittoError(f"{what}: timestep index out of range [0, {steps}): min {lo}, max {hi}")


def _need_cuda_f32(name: str, t: torch.Tensor) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise DittoError(f"{name} must be a CUDA tensor: ditto_tts_b200 has no CPU fallback")
    if t.dtype != torch.float32:
        raise DittoError(f"{name} must be float32 (the reference path is fp32 end to end), got {t.dtype}")
    return t.contiguous()


def _check_text_lengths(text_lengths, widths: List[int]) -> Optional[List[int]]:
    """None, or one integer text length per utterance with text_lengths[i] in [1, widths[i]], the text rows utterance i was
    given.  Lengths are data of the text context (ditto_text_context_masked): any value in range reuses the same graphs."""
    if text_lengths is None:
        return None
    try:
        vals = text_lengths.tolist() if hasattr(text_lengths, "tolist") else list(text_lengths)
    except TypeError:
        vals = None
    if isinstance(text_lengths, (str, bytes)) or not isinstance(vals, list):
        raise DittoError("text_lengths must be a sequence of one integer per utterance")
    if len(vals) != len(widths):
        raise DittoError(f"text_lengths must hold one length per utterance: {len(widths)} expected, got {len(vals)}")
    out = []
    for i, (v, hi) in enumerate(zip(vals, widths)):
        if isinstance(v, bool):
            raise DittoError(f"text_lengths[{i}] must be an integer, got a bool")
        try:
            v = operator.index(v)
        except TypeError:
            raise DittoError(f"text_lengths[{i}] must be an integer, got {type(v).__name__}") from None
        if not 1 <= v <= hi:
            raise DittoError(f"text_lengths[{i}] = {v} is outside [1, {hi}] (the text rows that utterance was given)")
        out.append(v)
    return out


class GlobalAdaLN(nn.Module):
    """Global AdaLN (reference: components/DiT.py:8-40).  Inside ``DiTTO.forward`` the modulation
    LN(x)*(1+ts+xs)+(tb+xb) is fused with block 0's LayerNorm; called on its own (same signature as the reference)
    it runs through ``ditto_adaln``."""

    def __init__(self, hidden_dim, time_dim, text_dim):
        super().__init__()
        self.time_mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_dim, 2 * hidden_dim))
        self.text_mlp = nn.Sequential(nn.SiLU(), nn.Linear(text_dim, 2 * hidden_dim))
        self.norm = nn.LayerNorm(hidden_dim, elementwise_affine=False)

    @torch.no_grad()
    def forward(self, x, time_emb, text_emb):
        """x [n,T,H], time_emb [n,time_dim] (output of ``time_embed``), text_emb [n,S,text_dim] -> [n,T,H]  (DiT.py:25-40)."""
        lib = _lib.load()
        x = _need_cuda_f32("x", x)
        time_emb = _need_cuda_f32("time_emb", time_emb)
        text_emb = _need_cuda_f32("text_emb", text_emb)
        wt, bt = self.time_mlp[1].weight, self.time_mlp[1].bias
        wx, bx = self.text_mlp[1].weight, self.text_mlp[1].bias
        if not wt.is_cuda:
            raise DittoError("GlobalAdaLN parameters are on the CPU: there is no CPU fallback")
        n, T, H = x.shape
        S, Xd, Td = text_emb.shape[1], text_emb.shape[2], time_emb.shape[1]
        if time_emb.shape[0] != n or text_emb.shape[0] != n or wt.shape != (2 * H, Td) or wx.shape != (2 * H, Xd):
            raise DittoError("GlobalAdaLN: shapes of x / time_emb / text_emb do not match the module")
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            nbytes = lib.ditto_adaln_workspace_bytes(n, H, Td, Xd)
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=x.device)
            w = [v.detach().float().contiguous() for v in (wt, bt, wx, bx)]
            _lib.check(lib.ditto_adaln(_ptr(x), _ptr(time_emb), _ptr(text_emb), _ptr(w[0]), _ptr(w[1]), _ptr(w[2]), _ptr(w[3]),
                                       _ptr(out), n, T, S, H, Td, Xd, _ptr(ws), ws.numel(), _stream()), "ditto_adaln")
        return out


class RotaryEmbedding(nn.Module):
    """RoPE angle table (reference: components/DiT.py:43-59).  ``forward`` returns the same [T, d] angle
    tensor as the reference (host-side table building); rotation itself happens in the QKV kernels."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim
        inv_freq = 1.0 / (10000 ** (torch.arange(0, dim, 2).float() / dim))
        self.register_buffer("inv_freq", inv_freq)

    def forward(self, seq_len, device):
        t = torch.arange(seq_len, device=device).type_as(self.inv_freq)
        freqs = torch.einsum("i,j->ij", t, self.inv_freq)
        return torch.cat((freqs, freqs), dim=-1)

    @torch.no_grad()
    def apply_rope(self, pos, t):
        """``t * cos(pos) + rotate_half(t) * sin(pos)`` (DiT.py:52-54,61-72): pos [T, head_dim] angles, t
        [batch, T, heads, head_dim] -> same shape.  (Inside DiTTO.forward the rotation is fused into the QKV GEMM epilogue.)"""
        t = _need_cuda_f32("t", t)
        pos = _need_cuda_f32("pos", pos)
        if t.dim() != 4 or pos.dim() != 2 or pos.shape[0] != t.shape[1] or pos.shape[1] != t.shape[3]:
            raise DittoError("apply_rope expects pos [T, head_dim] and t [batch, T, heads, head_dim]")
        out = torch.empty_like(t)
        b, T, h, d = t.shape
        with torch.cuda.device(t.device):
            _lib.check(_lib.load().ditto_rope(_ptr(t), _ptr(pos), _ptr(out), b, T, h, d, _stream()), "ditto_rope")
        return out


class DiT(nn.Module):
    """Parameters of one DiT block (reference: components/DiT.py:78-98), same names and init order."""

    def __init__(self, hidden_dim, num_heads, time_dim, text_dim):
        super().__init__()
        self.num_heads = num_heads
        self.head_dim = hidden_dim // num_heads
        self.norm1 = nn.LayerNorm(hidden_dim)
        self.attn = nn.MultiheadAttention(hidden_dim, num_heads)
        self.rotary = RotaryEmbedding(self.head_dim)
        self.norm2 = nn.LayerNorm(hidden_dim)
        self.cross_attn = nn.MultiheadAttention(hidden_dim, num_heads, dropout=0.1)
        self.norm3 = nn.LayerNorm(hidden_dim)
        self.mlp_fc1 = nn.Linear(hidden_dim, 4 * hidden_dim)
        self.act = nn.GELU()
        self.gate = nn.Linear(hidden_dim, 4 * hidden_dim)
        self.mlp_fc2 = nn.Linear(4 * hidden_dim, hidden_dim)

        self.hidden_dim, self.time_dim, self.text_dim = hidden_dim, time_dim, text_dim
        self._owner = None          # (weakref to the DiTTO that holds this block, layer index); None: stand-alone block
        self._own = None            # stand-alone block: a private one-block DiTTO-less engine holder

    @torch.no_grad()
    def forward(self, x, text_emb, time_emb=None, rotary_pos=None):
        """One DiT block, reference signature (DiT.py:100-157): x [n,T,H], text_emb [n,S,text_dim] -> [n,T,H].
        ``time_emb`` is accepted and ignored exactly as the reference block ignores it; ``rotary_pos`` must be the
        standard table ``RotaryEmbedding.forward(T)`` (None = that table): the kernels rotate with positions 0..T-1."""
        x = _need_cuda_f32("x", x)
        text_emb = _need_cuda_f32("text_emb", text_emb)
        if x.dim() != 3 or text_emb.dim() != 3 or x.shape[0] != text_emb.shape[0]:
            raise DittoError("expected x [n,T,H] and text_emb [n,S,text_dim] with the same n")
        n, T, H = x.shape
        if rotary_pos is not None:
            std = self.rotary(T, x.device)
            if tuple(rotary_pos.shape) != tuple(std.shape) or not torch.equal(rotary_pos.to(std), std):
                raise DittoError("DiT.forward: rotary_pos must equal RotaryEmbedding.forward(seq_len) (positions 0..T-1)")
        return self._run("ditto_dit_block", x, text_emb)

    def _run(self, symbol, x, text_emb):
        n, T, _ = x.shape
        host, layer = self._engine_host()
        ctx = host.text_context(text_emb, name="block_ctx", T_hint=T)
        out = torch.empty_like(x)
        with torch.cuda.device(x.device):
            ws = host.workspace(n, T, text_emb.shape[1])
            _lib.check(getattr(_lib.load(), symbol)(host.engine(), layer, _ptr(x), _ptr(ctx), n, T, text_emb.shape[1], _ptr(out), _ptr(ws),
                                                    ws.numel(), _stream()), symbol)
        return out

    @torch.no_grad()
    def section(self, name, x, text_emb):
        """One of the three sections of the block on its own, LayerNorm to residual add (``ditto_attn_self`` / ``ditto_attn_cross`` /
        ``ditto_gated_mlp``): name "self" (DiT.py:103-139), "cross" (:141-148) or "mlp" (:150-155); forward == the three in order.
        ``text_emb`` [n,S,text_dim] is needed by every section (it sizes the workspace), only "cross" reads it."""
        symbol = {"self": "ditto_attn_self", "cross": "ditto_attn_cross", "mlp": "ditto_gated_mlp"}.get(name)
        if symbol is None:
            raise DittoError("DiT.section: name must be 'self', 'cross' or 'mlp'")
        x = _need_cuda_f32("x", x)
        text_emb = _need_cuda_f32("text_emb", text_emb)
        if x.dim() != 3 or text_emb.dim() != 3 or x.shape[0] != text_emb.shape[0]:
            raise DittoError("expected x [n,T,H] and text_emb [n,S,text_dim] with the same n")
        return self._run(symbol, x, text_emb)

    def _engine_host(self):
        if self._owner is not None:
            owner = self._owner[0]()
            if owner is not None:
                return owner, self._owner[1]
        if self._own is None:
            self._own = _BlockEngine(self)
        return self._own, 0


class _Buffers:
    """Caller-owned device scratch for the C-ABI (workspace / text context), cached by size."""

    def __init__(self):
        self._bufs: Dict[str, torch.Tensor] = {}

    def get(self, name: str, nbytes: int, device) -> torch.Tensor:
        b = self._bufs.get(name)
        if b is None or b.numel() < nbytes or b.device != device:
            b = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
            self._bufs[name] = b
        return b


class _EngineHost:
    """What DiTTO and a stand-alone DiT block share: a native engine built from a state_dict-like set of tensors, refreshed
    when they change, plus the caller-owned scratch the C-ABI wants."""

    def _host_init(self):
        self._engine = None
        self._engine_key = None
        self._tensors = None       # cached [(key, tensor)] of the engine's weights (invalidated by _apply / load_state_dict)
        self._bufs = _Buffers()

    # -- to be provided: _engine_config() -> _lib.Config, _engine_tensors() -> [(key, tensor)], _device()
    def _weights_key(self):
        """(data_ptr, version) of every weight: cheap enough for every call (no state_dict rebuild).  In-place edits through
        ``.data`` do not bump ``_version`` -- call ``refresh_weights()`` after those."""
        if self._tensors is None:
            self._tensors = self._engine_tensors()
        return tuple((v.data_ptr(), v._version) for _, v in self._tensors)

    def refresh_weights(self):
        """Force the engine to re-read (and re-pack) every weight on its next use.  Needed after edits the version counter
        does not see: ``p.data.copy_(...)``, ``p.data.mul_(...)`` (EMA swaps), external writes through raw pointers.
        CUDA graphs captured earlier keep working: the engine's packed buffers are refreshed in place."""
        self._engine_key = None
        self._tensors = None

    def engine(self):
        """Create / refresh the native engine from the current parameters (must live on a CUDA device)."""
        lib = _lib.load()
        dev = self._device()
        if dev.type != "cuda":
            raise DittoError("parameters are on the CPU: move the module to a B200 (module.cuda()); there is no CPU fallback")
        key = self._weights_key()
        if self._engine is not None and key == self._engine_key:
            return self._engine
        with torch.cuda.device(dev):
            if self._engine is None:
                cfg = self._engine_config()
                h = C.c_void_p()
                _lib.check(lib.ditto_engine_create(C.byref(cfg), C.byref(h)), "ditto_engine_create")
                self._engine = h
            for k, v in self._tensors:
                w = v.detach().to(device=dev, dtype=torch.float32).contiguous()
                _lib.check(lib.ditto_engine_load_weight(self._engine, k.encode(), _ptr(w), w.numel(), _stream()),
                           f"ditto_engine_load_weight({k})")
            _lib.check(lib.ditto_engine_finalize(self._engine, _stream()), "ditto_engine_finalize")
        self._engine_key = key
        return self._engine

    def workspace(self, n_seq: int, T: int, S: int) -> torch.Tensor:
        eng = self.engine()
        nbytes = _lib.load().ditto_workspace_bytes(eng, n_seq, T, S)
        if nbytes < 0:
            raise DittoError("ditto_workspace_bytes: bad sizes")
        return self._bufs.get("ws", nbytes, self._device())

    def text_context(self, text_emb: torch.Tensor, name: str = "ctx", T_hint: int = 1, text_lengths=None) -> torch.Tensor:
        """Step-invariant text work (cross-attention K/V of every layer + text modulation) for a batch.  ``text_lengths``
        (one integer in [1, S] per sequence): sequence i uses text rows [0, text_lengths[i]) only (ditto_text_context_masked)."""
        eng = self.engine()
        lib = _lib.load()
        text_emb = _need_cuda_f32("text_emb", text_emb)
        if text_emb.dim() != 3:
            raise DittoError("text_emb must be [n, S, text_dim]")
        n, S, Xd = text_emb.shape
        if Xd != self.text_dim:
            raise DittoError(f"text_emb last dim {Xd} != text_dim {self.text_dim}")
        lens = _check_text_lengths(text_lengths, [S] * n)
        with torch.cuda.device(text_emb.device):
            ctx = self._bufs.get(name, lib.ditto_text_context_bytes(eng, n, S), text_emb.device)
            ws = self.workspace(n, T_hint, S)
            if lens is None:
                _lib.check(lib.ditto_text_context(eng, _ptr(text_emb), n, S, _ptr(ctx), _ptr(ws), ws.numel(), _stream()),
                           "ditto_text_context")
            else:
                _lib.check(lib.ditto_text_context_masked(eng, _ptr(text_emb), n, S, (C.c_int64 * n)(*lens), _ptr(ctx), _ptr(ws),
                                                         ws.numel(), _stream()), "ditto_text_context_masked")
        return ctx

    def _destroy_engine(self):
        try:
            if getattr(self, "_engine", None) is not None:
                _lib.load().ditto_engine_destroy(self._engine)
                self._engine = None
        except Exception:
            pass


class _BlockEngine(_EngineHost):
    """Engine holder of a stand-alone ``DiT`` block (DITTO_F_BLOCKS_ONLY, one layer, keys ``blocks.0.*``)."""

    def __init__(self, block: "DiT"):
        self._block = weakref.ref(block)
        self.text_dim = block.text_dim
        self._host_init()

    def _device(self):
        return self._block().norm1.weight.device

    def _engine_config(self):
        b = self._block()
        return _lib.Config(hidden_dim=b.hidden_dim, num_layers=1, num_heads=b.num_heads, time_dim=b.time_dim, text_dim=b.text_dim,
                           diffusion_steps=1, precision=_lib.PREC_BF16 if getattr(b, "precision", "bf16") == "bf16" else _lib.PREC_FP32,
                           max_seq_len=getattr(b, "max_seq_len", 4096),
                           flags=_lib.F_FUSED_ROPE | _lib.F_FOLD_CROSS | _lib.F_FUSED_ATTN | _lib.F_BLOCKS_ONLY)

    def _engine_tensors(self):
        return [("blocks.0." + k, v) for k, v in self._block().state_dict(keep_vars=True).items()]

    def __del__(self):
        self._destroy_engine()


class DiTTO(nn.Module, _EngineHost):
    """Drop-in for ``model.DiTTO.DiTTO`` (reference: src/model/DiTTO.py:7-126) on the inference path.

    Same constructor keywords; ``forward(x, text_emb, t)`` -> eps_hat with x [n,T,H] fp32, text_emb
    [n,S,text_dim] fp32, t [n] int64, all CUDA.  Differences, all outside the hot path:
      * the NAC (HF EnCodec/GPT-2 + a checkpoint file, DiTTO.py:22-34) is not constructed: pass
        ``nac=<module>`` to attach one; ``nac.*`` keys of reference checkpoints are ignored on load;
      * extra keywords ``precision`` ("bf16" tensor-core path | "fp32" CUDA-core parity path),
        ``max_seq_len`` (RoPE table rows), ``fused_rope`` (RoPE in the QKV GEMM epilogue) and ``fold_cross``
        (cross-attention q/out projections folded into the per-utterance text K/V; single-head models only),
        ``fused_attn`` (scores + softmax in one kernel) and ``defer_ln`` (block LayerNorms folded into the GEMMs
        on either side: no LayerNorm pass over HBM; parity-tested, off by default -- on B200 the heavier GEMM
        epilogues cost more than the 14 LayerNorm launches they replace, see profiles/README.md).
    """

    def __init__(self, hidden_dim=768, num_layers=12, num_heads=12, time_dim=256, text_dim=768,
                 diffusion_steps=1000, lambda_factor=0.1, nac_model_path=None, *, nac: Optional[nn.Module] = None,
                 precision: str = "bf16", max_seq_len: int = 4096, fused_rope: bool = True,
                 fold_cross: bool = True, fused_attn: bool = True, defer_ln: bool = False):
        super().__init__()
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.hidden_dim, self.num_layers, self.num_heads = hidden_dim, num_layers, num_heads
        self.time_dim, self.text_dim, self.diffusion_steps = time_dim, text_dim, diffusion_steps
        self.lambda_factor, self.nac_model_path = lambda_factor, nac_model_path
        self.precision, self.max_seq_len, self.fused_rope = precision, max_seq_len, fused_rope
        self.fold_cross = fold_cross
        self.fused_attn = fused_attn
        self.defer_ln = defer_ln and fused_rope
        if nac is not None:
            self.nac = nac
        # construction order == reference (DiTTO.py:36-64): seeded default init gives the same weights
        self.t_embedding = nn.Embedding(diffusion_steps, time_dim)
        self.time_embed = nn.Sequential(nn.Linear(time_dim, time_dim), nn.SiLU(), nn.Linear(time_dim, time_dim))
        self.ada_ln = GlobalAdaLN(hidden_dim, time_dim, text_dim)
        self.blocks = nn.ModuleList([DiT(hidden_dim, num_heads, time_dim, text_dim) for _ in range(num_layers)])
        self.proj_in = nn.Linear(hidden_dim, hidden_dim)
        self.proj_out = nn.Linear(hidden_dim, hidden_dim)
        self.rotary = RotaryEmbedding(hidden_dim // num_heads)
        self.register_buffer("alphas_cumprod", self.cosine_beta_schedule(diffusion_steps))
        for i, blk in enumerate(self.blocks):      # block.forward(x, text_emb, t, rotary_pos) runs block i of THIS engine
            blk._owner = (weakref.ref(self), i)
        self._host_init()
        self._schedule_loaded = False
        self.eval()

    # ------------------------------------------------------------------ reference API (host side)
    def cosine_beta_schedule(self, timesteps, s=0.008):
        """Identical arithmetic to DiTTO.py:96-104 (host torch ops; returns the clipped betas)."""
        steps = timesteps + 1
        x = torch.linspace(0, timesteps, steps)
        alphas_cumprod = torch.cos(((x / timesteps) + s) / (1 + s) * torch.pi * 0.5) ** 2
        alphas_cumprod = alphas_cumprod / alphas_cumprod[0]
        betas = 1 - (alphas_cumprod[1:] / alphas_cumprod[:-1])
        return torch.clip(betas, 0.0001, 0.9999)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Accepts reference checkpoints: ``nac.*`` entries are dropped unless a NAC is attached."""
        if not hasattr(self, "nac"):
            state_dict = {k: v for k, v in state_dict.items() if not k.startswith("nac.")}
        out = super().load_state_dict(state_dict, strict=strict, assign=assign)
        self.refresh_weights()
        return out

    # ------------------------------------------------------------------ engine plumbing (_EngineHost)
    def _device(self):
        return self.proj_in.weight.device

    def _engine_config(self):
        return _lib.Config(hidden_dim=self.hidden_dim, num_layers=self.num_layers, num_heads=self.num_heads,
                           time_dim=self.time_dim, text_dim=self.text_dim, diffusion_steps=self.diffusion_steps,
                           precision=_lib.PREC_BF16 if self.precision == "bf16" else _lib.PREC_FP32,
                           max_seq_len=self.max_seq_len,
                           flags=(_lib.F_FUSED_ROPE if self.fused_rope else 0) | (_lib.F_FOLD_CROSS if self.fold_cross else 0) |
                           (_lib.F_FUSED_ATTN if self.fused_attn else 0) | (_lib.F_DEFER_LN if self.defer_ln else 0))

    def _engine_tensors(self):
        return [(k, v) for k, v in self.state_dict(keep_vars=True).items() if not k.startswith("nac.")]

    def _apply(self, fn, *a, **k):   # .to() / .cuda() re-create buffers: drop the cached tensor list
        out = super()._apply(fn, *a, **k)
        self._tensors = None
        return out

    def load_schedule(self, betas: torch.Tensor, alphas: torch.Tensor, alphas_cumprod: torch.Tensor, owner=None):
        """Hand the sampler tables (SpeechGenerator.py:70-72) to the engine.  ``owner`` tags whose tables the engine
        holds (a sampler with its own schedule / update rule re-loads them when another user replaced them)."""
        eng = self.engine()
        dev = self.proj_in.weight.device
        tabs = [z.detach().to(device=dev, dtype=torch.float32).contiguous() for z in (betas, alphas, alphas_cumprod)]
        with torch.cuda.device(dev):
            _lib.check(_lib.load().ditto_engine_load_schedule(eng, _ptr(tabs[0]), _ptr(tabs[1]), _ptr(tabs[2]),
                                                             tabs[0].numel(), _stream()), "ditto_engine_load_schedule")
            torch.cuda.current_stream().synchronize()
        self._schedule_loaded = True
        self._schedule_owner = owner

    def load_update_table(self, coef: torch.Tensor):
        """Replace the per-timestep update coefficients [diffusion_steps, 3] (sampler variants, schedules.py)."""
        self._load_table("update", coef, 3)

    def load_multistep_table(self, coef: torch.Tensor):
        """Hand a [diffusion_steps, 6] multistep update table (schedules.dpmpp_2m_coef) to the engine."""
        self._load_table("multistep", coef, 6)

    def load_known_table(self, coef: torch.Tensor):
        """Hand a [diffusion_steps, 2] known-frame table (schedules.known_coef: the re-noising of a speech prompt or of the
        frames around an infilled span) to the engine."""
        self._load_table("known", coef, 2)

    def _load_table(self, kind: str, coef: torch.Tensor, cols: int):
        """ditto_engine_load_<kind>_table with a checked [diffusion_steps, cols] fp32 copy of ``coef`` on the engine's device."""
        eng = self.engine()
        dev = self.proj_in.weight.device
        if tuple(coef.shape) != (self.diffusion_steps, cols):
            raise DittoError(f"{kind} table must be [{self.diffusion_steps}, {cols}]")
        tab = coef.detach().to(device=dev, dtype=torch.float32).contiguous()
        name = f"ditto_engine_load_{kind}_table"
        with torch.cuda.device(dev):
            _lib.check(getattr(_lib.load(), name)(eng, _ptr(tab), self.diffusion_steps, _stream()), name)
            torch.cuda.current_stream().synchronize()

    def _ensure_schedule(self):
        """The module's own (reference) schedule: what q_sample reads (DiTTO.py:63-64,106-126)."""
        if not self._schedule_loaded or getattr(self, "_schedule_owner", None) is not None:
            betas = self.cosine_beta_schedule(self.diffusion_steps)
            alphas = 1.0 - betas
            self.load_schedule(betas, alphas, torch.cumprod(alphas, dim=0))

    def forward_with_context(self, x: torch.Tensor, ctx: torch.Tensor, t: torch.Tensor, n_seq: int, S: int,
                             out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """eps_hat for n_seq sequences whose text context is already built; x [n_x,T,H] with n_seq % n_x == 0."""
        eng = self.engine()
        lib = _lib.load()
        x = _need_cuda_f32("x", x)
        n_x, T, H = x.shape
        if H != self.hidden_dim:
            raise DittoError(f"x last dim {H} != hidden_dim {self.hidden_dim}")
        if not t.is_cuda or t.dtype != torch.int64 or t.numel() != n_seq:
            raise DittoError("t must be a CUDA int64 tensor with one entry per sequence")
        t = t.contiguous()
        if out is None:
            out = torch.empty((n_seq, T, H), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            ws = self.workspace(n_seq, T, S)
            _lib.check(lib.ditto_forward(eng, _ptr(x), n_x, _ptr(ctx), _ptr(t), n_seq, T, S, _ptr(out), _ptr(ws),
                                         ws.numel(), _stream()), "ditto_forward")
        return out

    @torch.no_grad()
    def forward(self, x, text_emb, t, *, text_lengths=None):
        """eps_hat = DiTTO.forward(x, text_emb, t)  (reference: DiTTO.py:66-94).  ``text_lengths`` (one integer in [1, S] per
        sequence): texts of different lengths padded to one S; sequence i then equals its run with ``text_emb[i, :len]``."""
        x = _need_cuda_f32("x", x)
        text_emb = _need_cuda_f32("text_emb", text_emb)
        if x.dim() != 3 or text_emb.dim() != 3 or x.shape[0] != text_emb.shape[0]:
            raise DittoError("expected x [n,T,H] and text_emb [n,S,text_dim] with the same n")
        t = t.to(device=x.device, dtype=torch.int64)
        _check_t_range(t, self.diffusion_steps, "DiTTO.forward")
        ctx = self.text_context(text_emb, T_hint=x.shape[1], text_lengths=text_lengths)
        return self.forward_with_context(x, ctx, t, x.shape[0], text_emb.shape[1])

    @torch.no_grad()
    def forward_ragged(self, xs, texts, t, *, text_lengths=None):
        """``DiTTO.forward`` on a mixed-length batch, every utterance at its own length (no padding, no masks -- the
        reference has none): xs[i] [T_i,H], texts[i] [S_i,text_dim], t [B] -> list of eps_hat [T_i,H].
        Equals ``[forward(x[None], text[None], t[i:i+1])[0] for ...]`` of the reference (DiTTO.py:66-94).
        ``text_lengths[i]`` in [1, S_i]: utterance i uses ``texts[i][:len]`` (padded texts that share a group)."""
        from .ragged import RaggedBatch
        rb = RaggedBatch(self, texts, [int(x.shape[0]) for x in xs], guided=False, text_lengths=text_lengths)
        out = rb.forward(rb.pack(xs), rb.seq_t(t))
        return rb.unpack(out)

    @torch.no_grad()
    def q_sample(self, x_start, t, noise=None):
        """Forward diffusion (reference: DiTTO.py:106-126, incl. its betas-as-alphas_cumprod buffer)."""
        x_start = _need_cuda_f32("x_start", x_start)
        if noise is None:
            noise = torch.randn_like(x_start)
        noise = _need_cuda_f32("noise", noise)
        self._ensure_schedule()
        t = t.to(device=x_start.device, dtype=torch.int64).contiguous()
        _check_t_range(t, self.diffusion_steps, "DiTTO.q_sample")
        out = torch.empty_like(x_start)
        B = x_start.shape[0]
        with torch.cuda.device(x_start.device):
            _lib.check(_lib.load().ditto_q_sample(self.engine(), _ptr(x_start), _ptr(noise), _ptr(t), _ptr(out), B,
                                                  x_start.numel() // B, _stream()), "ditto_q_sample")
        return out

    def __del__(self):
        self._destroy_engine()
