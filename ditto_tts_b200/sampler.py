"""DDPM ancestral sampler around the native DiTTO engine.

Mirrors the sampling part of the reference's ``SpeechGenerator`` (src/model/SpeechGenerator.py):
schedule tables :70-72, ``__p_sample`` :131-147, ``__sample_latents`` :150-164 -- same arithmetic, same
argument meaning -- plus the classifier-free-guidance extension BASELINE.json asks for
(eps = eps_u + w (eps_c - eps_u), unconditional branch = zero text embedding unless supplied).
One sampler iteration is a single C-ABI call (ditto_p_sample_known, which without known frames is ditto_p_sample): the
2B-sequence forward and the fused CFG-combine + update kernel; the text K/V and modulation vectors are built once per
utterance batch.
``method="dpmpp_2m"`` (DPM-Solver++(2M), schedules.dpmpp_2m_coef) also carries the previous step's x0 prediction in a
device buffer ``hist`` that the update kernel reads and rewrites.
``sample_latents(..., known=p, known_mask=m)`` continues a speech prompt or fills a span: frames with m True are given
(replacement conditioning, schedules.known_coef; the update kernel re-noises them).
``sample_latents(..., seeds=[s_0, ...], guidance_scale=[w_0, ...])`` gives every utterance its own noise stream (x_T and every
step's noise depend on its seed alone, not on its batch-mates: include/ditto_b200.h, ditto_p_sample_per_utt) and its own
guidance scale; one captured step graph serves every scale.
``text_lengths=[l_0, ...]`` lets texts of different token counts share one padded ``text_emb`` [B, S, text_dim]: utterance b
(and its unconditional branch) uses text rows [0, l_b) only and samples as it would with ``text_emb[b, :l_b]``.  The lengths
live in the text context, so one captured step graph serves every set of lengths.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
import operator
from collections import OrderedDict
from typing import List, Optional, Union

import torch

from . import _lib, schedules
from ._lib import DittoError
from .model import DiTTO, _check_t_range, _check_text_lengths, _need_cuda_f32, _ptr, _stream

__all__ = ["DiTTOSampler", "StepGraph", "randn_latents"]


def _check_seeds(seeds, B: int, noise=None, generator=None) -> Optional[List[int]]:
    """None, or B integer seeds in [0, 2^64) (one per utterance); refused together with ``noise`` / ``generator``, which
    are the other two sources of the job's noise."""
    if seeds is None:
        return None
    if noise is not None or generator is not None:
        raise DittoError("seeds excludes noise= and generator=: each is a different source of the job's noise")
    try:
        vals = seeds.tolist() if hasattr(seeds, "tolist") else list(seeds)
    except TypeError:
        vals = None
    if isinstance(seeds, (str, bytes)) or not isinstance(vals, list):
        raise DittoError("seeds must be a sequence of one integer per utterance")
    out = []
    for i, v in enumerate(vals):
        if isinstance(v, bool):
            raise DittoError(f"seeds[{i}] must be an integer, got a bool")
        try:
            v = operator.index(v)
        except TypeError:
            raise DittoError(f"seeds[{i}] must be an integer, got {type(v).__name__}") from None
        if not 0 <= v < 1 << 64:
            raise DittoError(f"seeds[{i}] = {v} is outside [0, 2^64)")
        out.append(v)
    if len(out) != B:
        raise DittoError(f"seeds must hold one seed per utterance: {B} expected, got {len(out)}")
    return out


def _check_scale(w, B: int) -> Union[None, float, List[float]]:
    """The guidance scale of a job: None (unguided), a scalar for every utterance, or a sequence of B finite scales.
    A scalar is whatever ``float(w)`` took before per-utterance scales existed: a real number (numpy scalars too) or a
    one-element tensor / array, whatever B is.  It is passed on as before, without a finiteness check, so a scalar job
    behaves exactly as it did; only per-utterance lists are checked to be finite."""
    if w is None:
        return None
    if isinstance(w, numbers.Real):
        return float(w)
    size = w.numel() if isinstance(w, torch.Tensor) else getattr(w, "size", None)
    if size == 1 and (isinstance(w, torch.Tensor) or hasattr(w, "__array__")):
        return float(w.item())
    try:
        vals = w.tolist() if hasattr(w, "tolist") else list(w)
    except TypeError:
        raise DittoError("guidance_scale must be a number or a sequence of one number per utterance") from None
    if len(vals) != B:
        raise DittoError(f"guidance_scale must be a scalar or hold one scale per utterance: {B} expected, got {len(vals)}")
    out = [float(v) for v in vals]
    if not all(math.isfinite(v) for v in out):
        raise DittoError("guidance_scale: every per-utterance scale must be finite")
    return out


def _seed_tensor(seeds: List[int], dev) -> torch.Tensor:
    """uint64 seeds as the int64 bit patterns the device reads as uint64."""
    return torch.tensor([v - (1 << 64) if v >= 1 << 63 else v for v in seeds], dtype=torch.int64).to(dev)


def randn_latents(seeds: torch.Tensor, row0: torch.Tensor, rows: int, H: int) -> torch.Tensor:
    """x_T of a seeded job in one launch (ditto_randn_latents): utterance b owns rows row0[b] .. row0[b + 1] - 1 of the
    [rows, H] result and gets the normals of its own seed's reserved draw.  seeds int64 [B] (uint64 bit patterns), row0
    int64 [B + 1], both on the device."""
    out = torch.empty((rows, H), dtype=torch.float32, device=seeds.device)
    with torch.cuda.device(seeds.device):
        _lib.check(_lib.load().ditto_randn_latents(_ptr(seeds), _ptr(row0), seeds.numel(), H, _ptr(out), _stream()),
                   "ditto_randn_latents")
    return out


class _CapturedStep:
    """What StepGraph and RaggedStepGraph share: the buffers a captured sampler step reads and writes (owned here, so that
    the captured pointers stay valid), the capture, the per-job reset and the replay loop.  A subclass allocates eps and the
    workspace and makes the step's one C call in ``_p_sample(rng)``."""

    def _buffers(self, shape, n_seq: int, draw_noise: bool, multistep: bool, known: bool, device, n_utt: int = 0,
                 guided: bool = False, seeded: bool = False):
        self.draw_noise = draw_noise
        self.x = torch.zeros(shape, dtype=torch.float32, device=device)
        # caller-supplied noise lands here; drawn noise never touches HBM
        self.z = None if draw_noise else torch.zeros_like(self.x)
        self.rng = torch.zeros((4,), dtype=torch.int64, device=device)   # {seed, draw counter, ticket, -} of ditto_p_sample_rng
        self.hist = torch.zeros_like(self.x) if multistep else None       # the x0 prediction one multistep step carries
        self.known = torch.zeros_like(self.x) if known else None          # known frames and their mask, filled by reset
        self.mask = torch.zeros(tuple(shape[:-1]), dtype=torch.uint8, device=device) if known else None
        self.t = torch.zeros((n_seq,), dtype=torch.int64, device=device)
        # per-utterance guidance scales (a scalar scale is broadcast into it, so one capture serves every scale) and seeds
        self.w_dev = torch.zeros((n_utt,), dtype=torch.float32, device=device) if guided else None
        self.seeds = torch.zeros((n_utt,), dtype=torch.int64, device=device) if seeded else None

    def set_scale(self, w):
        """The guidance scale the next replays use: a scalar for every utterance or a [n_utt] tensor (graph order)."""
        if self.w_dev is not None:
            if isinstance(w, torch.Tensor):
                self.w_dev.copy_(w)
            else:
                self.w_dev.fill_(float(w))

    def _capture(self, device):
        # eager warm-up (engine set-up, lazy initialisation) on a side stream, then capture
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            self._step()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        self.graph = torch.cuda.CUDAGraph()
        n0 = _lib.launch_count()
        with torch.cuda.graph(self.graph):
            self._step()
        self.launches_per_step = _lib.launch_count() - n0

    def _step(self):
        # drawn noise: drawn every step incl. t = 0, like the reference's randn_like (SpeechGenerator.py:145), and the update
        # kernel does the "t -= 1" and draw-counter bookkeeping
        self._p_sample(self.rng if self.draw_noise else None)
        if not self.draw_noise:
            self.t.sub_(1)

    def reset(self, x_init: torch.Tensor, t_start: int, seed: Optional[int] = None, known: Optional[torch.Tensor] = None,
              known_mask: Optional[torch.Tensor] = None, seeds: Optional[torch.Tensor] = None):
        self.x.copy_(x_init)
        self.t.fill_(t_start)
        if self.hist is not None:
            self.hist.zero_()
        if self.known is not None:
            self.known.copy_(known)
            self.mask.copy_(known_mask)
        if self.seeds is not None:   # per-utterance seeds (graph order) key the noise; the draw counter starts at 0
            self.seeds.copy_(seeds)
            self.rng.zero_()
        elif self.draw_noise:   # fresh seed per sampling job (from torch's CPU generator: torch.manual_seed makes runs repeatable)
            if seed is None:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            self.rng.copy_(torch.tensor([seed, 0, 0, 0], dtype=torch.int64), non_blocking=False)

    def replay(self):
        self.graph.replay()

    def run(self, x_init: torch.Tensor, taus: List[int], consecutive: bool, noise=None, known=None, known_mask=None, seeds=None):
        """One sampling job: reset, then one replay per visited timestep (``noise`` indexed by timestep, as ``x``)."""
        self.reset(x_init, taus[0], known=known, known_mask=known_mask, seeds=seeds)
        for t_val in taus:
            if noise is not None:
                self.z.copy_(noise[t_val], non_blocking=True)
            if not consecutive:
                self.t.fill_(t_val)      # the graph's own "t -= 1" only covers the reference's consecutive timesteps
            self.replay()


class StepGraph(_CapturedStep):
    """One sampler iteration captured as a CUDA graph and replayed once per step.

    The graph holds the 2B-sequence forward and the fused CFG + DDPM update (in place on ``x``); when the noise is not
    supplied by the caller that same kernel draws it (Philox, ``ditto_p_sample_rng``) and, as its last act, decrements
    the device-resident step index ``t`` and bumps the draw counter -- so the host issues ONE launch per denoising step
    instead of ~70 and the graph contains kernels of libditto_b200 only.  A multistep sampler's graph also owns ``hist``,
    the x0 prediction one step carries to the next (zero-filled by ``reset``).  A graph for known frames (speech prompt,
    infilling) owns the known latents and the frame mask, filled by ``reset``; it launches as many kernels per step.  A guided
    graph reads its guidance scales from ``w_dev`` (one per utterance, ``set_scale``); a ``seeded`` graph keys every
    utterance's noise by its entry of ``seeds`` (filled by ``reset``)."""

    def __init__(self, sampler: "DiTTOSampler", B: int, T: int, S: int, guided: bool, w, ctx: torch.Tensor,
                 draw_noise: bool, device, known: bool = False, seeded: bool = False):
        m = sampler.model
        n = 2 * B if guided else B
        self.B, self.T, self.S, self.guided = B, T, S, guided
        self._buffers((B, T, m.hidden_dim), n, draw_noise, sampler.multistep, known, device, B, guided, seeded)
        self.set_scale(w)
        self.eps = torch.empty((n, T, m.hidden_dim), dtype=torch.float32, device=device)
        self.ctx = ctx
        self.ws = m.workspace(n, T, S)
        self._sampler = sampler
        self._capture(device)
        self._keys = (self.ctx.data_ptr(), self.ws.data_ptr())

    def _p_sample(self, rng):
        self._sampler._p_sample_raw(self.x, self.ctx, self.t, self.z, self.guided, 0.0, self.S, self.eps, self.x, ws=self.ws,
                                    hist=self.hist, known=self.known, mask=self.mask, rng=rng, seeds=self.seeds, w_dev=self.w_dev)

    def valid_for(self, ctx: torch.Tensor, ws: torch.Tensor) -> bool:
        return self._keys == (ctx.data_ptr(), ws.data_ptr())


class DiTTOSampler:
    """``method`` / ``num_steps`` / ``eta`` / ``schedule_scale`` select the sampler variants of SURVEY.md 8f row 4
    (schedules.py); the defaults are the reference's sampler: DDPM over every timestep of the cosine schedule.
    ``method="dpmpp_2m"`` is the second-order multistep DPM-Solver++(2M) (eta = 0) or its SDE variant (eta = 1), e.g.
    ``DiTTOSampler(model, 5.0, method="dpmpp_2m", num_steps=16)``; it has state across steps, so ``p_sample`` refuses it.
    Every method also samples around known frames (``sample_latents(..., known=, known_mask=)``)."""

    def __init__(self, model: DiTTO, guidance_scale: Optional[float] = None, *, method: str = "ddpm",
                 num_steps: Optional[int] = None, eta: float = 0.0, schedule_scale: Optional[float] = None):
        if method not in ("ddpm", "ddim", "dpmpp_2m"):
            raise ValueError("method must be 'ddpm', 'ddim' or 'dpmpp_2m'")
        self.model = model
        self.guidance_scale = guidance_scale
        self.method, self.eta, self.schedule_scale = method, float(eta), schedule_scale
        steps = model.diffusion_steps
        # SpeechGenerator.py:70-72 (host torch ops => bit-identical tables)
        self.betas = model.cosine_beta_schedule(steps) if schedule_scale is None else \
            schedules.shifted_cosine_betas(steps, schedule_scale)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_steps = steps if num_steps is None else int(num_steps)
        # model timesteps visited, descending (the reference: reversed(range(DIFFUSION_STEPS)), SpeechGenerator.py:161)
        self.timesteps = schedules.spaced_timesteps(steps, self.num_steps)
        self.update_table = None        # [steps, 3] DDPM-form table (ditto_engine_load_update_table)
        self.multistep_table = None     # [steps, 6] multistep table (ditto_engine_load_multistep_table)
        self.multistep = method == "dpmpp_2m"
        acp64 = torch.cumprod(1.0 - self.betas.to(torch.float64), dim=0)
        taus = self.timesteps.tolist()
        if self.multistep:
            self.multistep_table = schedules.coef_table(steps, taus, schedules.dpmpp_2m_coef(acp64, taus, eta))
        elif method == "ddim" or self.num_steps != steps:
            coef = schedules.ddim_coef(acp64, taus, eta) if method == "ddim" else schedules.ddpm_coef(acp64, taus)
            self.update_table = schedules.coef_table(steps, taus, coef)
        # known frames (speech prompt, infilling): re-noised to the level of each step's output under THIS schedule
        self._acp64 = acp64
        self.known_table = schedules.coef_table(steps, taus, schedules.known_coef(acp64, taus))   # [steps, 2]
        self._variant = self.update_table is not None or self.multistep or schedule_scale is not None
        self._tau_dev = None
        # captured step graphs pin x / eps / a private memory pool (hundreds of MB at B = 16, T = 750) and TTS serving sees a
        # new predicted length on almost every request: keep the few most recently used shapes only
        self.max_cached_graphs = 4
        self._graphs = OrderedDict()
        self._ragged_graphs = OrderedDict()
        self._activate()

    def _activate(self, known: bool = False):
        """Make the engine hold THIS sampler's schedule / update table (another sampler or q_sample may have replaced them)
        and, for a job with known frames, its known-frame table (every sampler has one, so it has its own owner tag)."""
        m = self.model
        owner = self if self._variant else None
        if not (m._schedule_loaded and getattr(m, "_schedule_owner", None) is owner and
                getattr(m, "_schedule_engine", None) is m._engine):
            m.load_schedule(self.betas, self.alphas, self.alphas_cumprod, owner=owner)
            if self.update_table is not None:
                m.load_update_table(self.update_table)
            if self.multistep_table is not None:
                m.load_multistep_table(self.multistep_table)
            m._schedule_engine = m._engine
        if known and (getattr(m, "_known_owner", None) is not self or getattr(m, "_known_engine", None) is not m._engine):
            m.load_known_table(self.known_table)
            m._known_owner, m._known_engine = self, m._engine

    def _known_start(self, x: torch.Tensor, known: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        """x_T with its known frames replaced by q(x_T | p) = sqrt(abar_tau0) p + sqrt(1 - abar_tau0) x (float64, same x)."""
        a = float(self._acp64[int(self.timesteps[0])])
        xk = (math.sqrt(a) * known.double() + math.sqrt(1.0 - a) * x.double()).to(x.dtype)
        return torch.where(mask.bool().unsqueeze(-1), xk, x)

    def _taus(self, device):
        if self._tau_dev is None or self._tau_dev.device != device:
            self._tau_dev = self.timesteps.to(device)
        return self._tau_dev

    # ------------------------------------------------------------------------------------------
    def _context(self, text_emb: torch.Tensor, guided: bool, null_text_emb: Optional[torch.Tensor], T: int, text_lengths=None):
        text_emb = _need_cuda_f32("text_emb", text_emb)
        if text_emb.dim() != 3:
            raise DittoError("text_emb must be [B, S, text_dim]")
        lens = _check_text_lengths(text_lengths, [text_emb.shape[1]] * text_emb.shape[0])
        if guided:
            null = torch.zeros_like(text_emb) if null_text_emb is None else _need_cuda_f32("null_text_emb", null_text_emb)
            if null.shape != text_emb.shape:
                raise DittoError("null_text_emb must have the shape of text_emb")
            text_emb = torch.cat([text_emb, null], dim=0)  # [cond(B); uncond(B)]
            if lens is not None:
                lens = lens + lens                         # the unconditional branch uses the same lengths
        return self.model.text_context(text_emb, name="sampler_ctx", T_hint=T, text_lengths=lens)

    def _p_sample_raw(self, x, ctx, t_n, z, guided, w, S, eps, x_out, ws=None, hist=None, known=None, mask=None, rng=None,
                      seeds=None, w_dev=None, advance=None):
        """One step: ``hist`` the multistep update, ``known`` / ``mask`` known frames, ``rng`` the noise drawn in the update
        kernel (which then also does the "t -= 1" bookkeeping unless ``advance`` is False) instead of ``z``; ``seeds`` [B]
        keys utterance b's noise (with rng), ``w_dev`` [B] its guidance scale (instead of ``w``)."""
        if advance is None:
            advance = rng is not None
        m = self.model
        B, T, H = x.shape
        n = 2 * B if guided else B
        with torch.cuda.device(x.device):
            if ws is None:
                ws = m.workspace(n, T, S)
            _lib.check(_lib.load().ditto_p_sample_per_utt(m.engine(), _ptr(x), _ptr(ctx), _ptr(t_n), _ptr(z), _ptr(rng), _ptr(seeds),
                                                          1 if guided else 0, float(w), _ptr(w_dev), B, T, S, _ptr(eps), _ptr(x_out),
                                                          _ptr(hist), _ptr(known), _ptr(mask), _ptr(ws), ws.numel(), 1 if advance else 0,
                                                          _stream()), "ditto_p_sample_per_utt")

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def predict_noise(self, x, t, text_emb, guidance_scale=None, null_text_emb=None, *, text_lengths=None):
        """eps_hat (guided when a scale is given): the call at SpeechGenerator.py:135 + CFG combine."""
        w = self.guidance_scale if guidance_scale is None else guidance_scale
        guided = w is not None
        x = _need_cuda_f32("x", x)
        B, T, H = x.shape
        ctx = self._context(text_emb, guided, null_text_emb, T, text_lengths)
        t = t.to(device=x.device, dtype=torch.int64)
        t_n = torch.cat([t, t]) if guided else t
        eps = self.model.forward_with_context(x, ctx, t_n.contiguous(), t_n.numel(), text_emb.shape[1])
        if not guided:
            return eps
        return eps[B:] + w * (eps[:B] - eps[B:])

    @torch.no_grad()
    def p_sample(self, x, t, text_emb, noise=None, guidance_scale=None, null_text_emb=None, *, text_lengths=None):
        """One reverse step (reference: __p_sample, SpeechGenerator.py:131-147).  ``noise`` replaces the
        reference's in-place ``torch.randn_like(x)``; when omitted it is drawn the same way.  Not for ``dpmpp_2m``: its
        update needs the previous step's x0 prediction, which only sample_latents(_ragged) carries from step to step."""
        if self.multistep:
            raise DittoError("p_sample: method 'dpmpp_2m' is a multistep solver and has state across steps; "
                             "use sample_latents / sample_latents_ragged")
        w = self.guidance_scale if guidance_scale is None else guidance_scale
        guided = w is not None
        x = _need_cuda_f32("x", x)
        B, T, H = x.shape
        self._activate()
        ctx = self._context(text_emb, guided, null_text_emb, T, text_lengths)
        t = t.to(device=x.device, dtype=torch.int64)
        _check_t_range(t, self.model.diffusion_steps, "p_sample")
        t_n = (torch.cat([t, t]) if guided else t).contiguous()
        z = torch.randn_like(x) if noise is None else _need_cuda_f32("noise", noise)
        eps = torch.empty((t_n.numel(), T, H), dtype=torch.float32, device=x.device)
        out = torch.empty_like(x)
        self._p_sample_raw(x, ctx, t_n, z, guided, w if guided else 0.0, text_emb.shape[1], eps, out)
        return out

    def step_graph(self, B: int, T: int, S: int, guided: bool, w, ctx: torch.Tensor, draw_noise: bool, device,
                   known: bool = False, seeded: bool = False):
        """Cached CUDA graph of one sampler iteration for this shape (re-captured if the buffers moved), set to the guidance
        scale ``w`` (a scalar, or a [B] tensor of per-utterance scales).  The scale is not part of the key: the graph reads
        it from its own buffer."""
        key = (B, T, S, guided, draw_noise, str(device), bool(known), bool(seeded))
        g = self._graphs.get(key)
        n = 2 * B if guided else B
        if g is None or not g.valid_for(ctx, self.model.workspace(n, T, S)):
            self._graphs.pop(key, None)
            while len(self._graphs) >= self.max_cached_graphs:
                self._graphs.popitem(last=False)          # least recently used; its buffers and graph pool are released
            g = StepGraph(self, B, T, S, guided, w, ctx, draw_noise, device, known=known, seeded=seeded)
            self._graphs[key] = g
        else:
            self._graphs.move_to_end(key)
            g.set_scale(w)
        return g

    @torch.no_grad()
    def sample_latents(self, text_emb, audio_emb=None, *, x_init=None, noise=None, guidance_scale=None,
                       null_text_emb=None, cond_by_audio=False, record: Optional[List[torch.Tensor]] = None,
                       generator: Optional[torch.Generator] = None, use_graph: bool = True,
                       known: Optional[torch.Tensor] = None, known_mask: Optional[torch.Tensor] = None, seeds=None,
                       text_lengths=None):
        """All reverse steps (reference: __sample_latents, SpeechGenerator.py:150-164).

        text_emb [B,S,text_dim]; ``audio_emb`` [B,T,H] gives the latent shape (and the start point when
        ``cond_by_audio``), exactly as in the reference; ``x_init`` overrides the initial N(0,I) draw;
        ``noise`` [steps,B,T,H] (indexed by t) replaces the per-step randn_like for parity runs;
        ``record`` collects the guided eps_hat of every step (parity tests).

        ``known`` [B,T,H] fp32 latents and ``known_mask`` [B,T] bool (True = known) give frames to keep: a speech prompt
        (``known_mask[:, :P] = True``, ``known[:, :P]`` = the prompt's codec latents) to continue, or the context of a span
        to fill.  Replacement conditioning (Song et al. 2021, score SDE): each step writes the known frames as p re-noised
        to the level of its output, with the noise the step draws, so the result holds them exactly.  Both CFG branches see
        them.

        ``seeds`` (B integers in [0, 2^64)) gives utterance b a noise stream of its own: x_T (unless ``x_init`` /
        ``cond_by_audio`` supplies it) and every step's noise are functions of seeds[b] alone (include/ditto_b200.h), so an
        utterance samples the same whatever else is in the batch.  Not together with ``noise`` or ``generator``.
        ``guidance_scale`` may hold one scale per utterance.

        ``text_lengths`` (B integers in [1, S]): utterance b uses ``text_emb[b, :text_lengths[b]]`` (and the same rows of
        ``null_text_emb``); what the other rows hold never reaches its result."""
        m = self.model
        w = self.guidance_scale if guidance_scale is None else guidance_scale
        guided = w is not None
        text_emb = _need_cuda_f32("text_emb", text_emb)
        dev = text_emb.device
        x = None
        if x_init is not None:
            x = _need_cuda_f32("x_init", x_init).clone()
        elif audio_emb is not None:
            audio_emb = _need_cuda_f32("audio_emb", audio_emb)
            if cond_by_audio:
                x = audio_emb.clone()
            elif seeds is None:
                x = torch.randn(audio_emb.shape, device=dev, generator=generator)
        else:
            raise DittoError("sample_latents needs audio_emb (shape donor) or x_init")
        B, T, H = x.shape if x is not None else audio_emb.shape
        seeds = _check_seeds(seeds, B, noise, generator)
        w = _check_scale(w, B)
        seeds_dev = None if seeds is None else _seed_tensor(seeds, dev)
        if x is None:   # x_T from the seeds
            x = randn_latents(seeds_dev, torch.arange(0, (B + 1) * T, T, dtype=torch.int64, device=dev), B * T, H).view(B, T, H)
        # per-utterance scales on the device; a scalar stays a kernel argument outside the graphs
        w_dev = torch.tensor(w, dtype=torch.float32, device=dev) if isinstance(w, list) else None
        S = text_emb.shape[1]
        has_known = known is not None or known_mask is not None
        if has_known:
            known, known_mask = _known_inputs(known, known_mask, (B, T, H), dev)
        self._activate(known=has_known)
        taus = self.timesteps.tolist()
        consecutive = self.num_steps == m.diffusion_steps
        ctx = self._context(text_emb, guided, null_text_emb, T, text_lengths)
        n = 2 * B if guided else B
        if has_known:
            x = self._known_start(x, known, known_mask)
        if use_graph and record is None and generator is None:
            # one CUDA-graph replay per denoising step (noise drawn inside the graph unless supplied)
            g = self.step_graph(B, T, S, guided, (w if w_dev is None else w_dev) if guided else 0.0, ctx, noise is None, dev,
                                known=has_known, seeded=seeds is not None)
            g.run(x, taus, consecutive, noise=noise, known=known, known_mask=known_mask, seeds=seeds_dev)
            return g.x.clone()
        # t for every step, all sequences share it (SpeechGenerator.py:162)
        t_all = self._taus(dev).unsqueeze(1).repeat(1, n).contiguous()
        eps = torch.empty((n, T, H), dtype=torch.float32, device=dev)
        x_next = torch.empty_like(x)
        z_buf = None if noise is not None or seeds is not None else torch.empty_like(x)
        # seeded: the update kernel draws step i's noise as draw i of every utterance's seed (rng[1] = i, no bookkeeping)
        rng = torch.zeros((4,), dtype=torch.int64, device=dev) if seeds is not None else None
        hist = torch.empty_like(x) if self.multistep else None   # first step is first order: never read before written
        w_rec = w_dev.view(B, 1, 1) if w_dev is not None else w
        for i, t_val in enumerate(taus):
            z = None
            if noise is not None:
                z = noise[t_val]
                if not z.is_cuda:
                    raise DittoError("noise must live on the GPU")
                z = z.contiguous()
            elif rng is not None:
                rng[1] = i
            else:
                z = z_buf.normal_(generator=generator)  # drawn every step incl. t = 0, as the reference does
            self._p_sample_raw(x, ctx, t_all[i], z, guided, w if guided and w_dev is None else 0.0, S, eps, x_next, hist=hist,
                               known=known, mask=known_mask, rng=rng, seeds=seeds_dev, w_dev=w_dev if guided else None,
                               advance=False)
            if record is not None:
                record.append((eps[B:] + w_rec * (eps[:B] - eps[B:])).clone() if guided else eps.clone())
            x, x_next = x_next, x
        return x

    # ------------------------------------------------------------------------------------------ ragged batches
    @torch.no_grad()
    def sample_latents_ragged(self, texts, lengths, *, x_init=None, noise=None, guidance_scale=None, null_texts=None,
                              record: Optional[List[List[torch.Tensor]]] = None, use_graph: bool = True,
                              known=None, known_mask=None, seeds=None, text_lengths=None):
        """``__sample_latents`` (SpeechGenerator.py:150-164) for a mixed-length batch: utterance i has ``lengths[i]`` latent
        frames (what the speech-length predictor returns x 75 fps, SpeechGenerator.py:157-158) and text ``texts[i]``
        [S_i, text_dim].  Every utterance is sampled at its own length, unpadded (see ragged.py).  ``x_init`` /
        ``noise`` are per-utterance lists ([T_i,H] / [steps,T_i,H]) for parity runs.  ``known`` / ``known_mask`` are
        per-utterance lists ([T_i,H] fp32 / [T_i] bool) of frames to keep, as in ``sample_latents``.  ``seeds`` and a
        per-utterance ``guidance_scale`` (utterance order) as in ``sample_latents``: an utterance's result does not depend on
        which utterances share its batch, beyond the forward's batch-dependent rounding.  ``text_lengths[i]`` in [1, S_i]:
        utterance i uses ``texts[i][:len]`` only; padding texts to a few widths lets them share groups (and graphs, which the
        lengths do not key).  Returns a list of [T_i,H]."""
        from .ragged import RaggedBatch, RaggedStepGraph
        m = self.model
        w = self.guidance_scale if guidance_scale is None else guidance_scale
        guided = w is not None
        seeds = _check_seeds(seeds, len(texts), noise)
        w = _check_scale(w, len(texts))
        # graphs (and the text-context buffers their kernels read) are cached per batch signature: a new batch with the same
        # (frames, tokens, count) groups re-fills the cached context buffers instead of capturing again
        sig = RaggedBatch.signature(texts, lengths, guided)
        cached = self._ragged_graphs.get(sig) if (use_graph and record is None) else None
        rb = RaggedBatch(m, texts, lengths, guided=guided, null_texts=null_texts,
                         ctx_storage=cached[0] if cached is not None else None, text_lengths=text_lengths)
        dev, H, steps = rb.device, m.hidden_dim, m.diffusion_steps
        seeds_dev = None if seeds is None else rb.pack_seeds(seeds)
        w_dev = rb.pack_w(w) if isinstance(w, list) else None
        has_known = known is not None or known_mask is not None
        kp = km = None
        if has_known:
            if known is None or known_mask is None or len(known) != rb.B or len(known_mask) != rb.B:
                raise DittoError("known and known_mask go together: one [T_i, H] latent and one [T_i] mask per utterance")
            pairs = [_known_inputs(known[i], known_mask[i], (rb.lengths[i], H), dev, f"[{i}]") for i in range(rb.B)]
            kp, km = rb.pack([p for p, _ in pairs]), rb.pack_mask([q for _, q in pairs])
        self._activate(known=has_known)
        taus = self.timesteps.tolist()
        consecutive = self.num_steps == steps
        if x_init is not None:
            x = rb.pack(x_init)
        elif seeds_dev is not None:
            x = randn_latents(seeds_dev, rb.row0(), rb.x_rows, H)
        else:
            x = torch.randn((rb.x_rows, H), dtype=torch.float32, device=dev)
        if has_known:
            x = self._known_start(x, kp, km)
        zs = None
        if noise is not None:   # [steps, sum T, H] packed once
            zs = torch.empty((steps, rb.x_rows, H), dtype=torch.float32, device=dev)
            for i, z in enumerate(noise):
                z = _need_cuda_f32(f"noise[{i}]", z)
                zs[:, rb.x_offset[i]:rb.x_offset[i] + rb.lengths[i]] = z
        if use_graph and record is None:
            # the scale is not part of the key: the graph reads it from its own buffer
            wv, draw, key = ((w if w_dev is None else w_dev) if guided else 0.0), zs is None, (zs is None, has_known, seeds is not None)
            g = cached[1].get(key) if cached is not None else None
            if g is None or not g.valid_for(rb):
                g = RaggedStepGraph(rb, wv, draw, multistep=self.multistep, known=has_known, seeded=seeds is not None)
                if cached is None:
                    while len(self._ragged_graphs) >= self.max_cached_graphs:
                        self._ragged_graphs.popitem(last=False)
                    cached = (rb._ctx, {})
                    self._ragged_graphs[sig] = cached
                cached[1][key] = g
            else:
                g.rebind(rb)
                g.set_scale(wv)
            self._ragged_graphs.move_to_end(sig)
            g.run(x, taus, consecutive, noise=zs, known=kp, known_mask=km, seeds=seeds_dev)
            return rb.unpack(g.x)
        eps = torch.empty((rb.seq_rows, H), dtype=torch.float32, device=dev)
        x_next = torch.empty_like(x)
        z_buf = torch.empty_like(x) if zs is None and seeds is None else None
        rng = torch.zeros((4,), dtype=torch.int64, device=dev) if seeds is not None else None   # as in sample_latents
        hist = torch.empty_like(x) if self.multistep else None
        for i, t_val in enumerate(taus):
            t_seq = torch.full((rb.n_seq,), t_val, dtype=torch.int64, device=dev)
            z = None
            if rng is not None:
                rng[1] = i
            else:
                z = zs[t_val] if zs is not None else z_buf.normal_()
            rb.p_sample(x, t_seq, z, w if guided and w_dev is None else 0.0, eps, x_next, hist=hist, known=kp, mask=km, rng=rng,
                        seeds=seeds_dev, w_dev=w_dev if guided else None, advance=False)
            if record is not None:
                record.append(rb.unpack_eps(eps, w))
            x, x_next = x_next, x
        return rb.unpack(x)


def _known_inputs(known, known_mask, shape, dev, what: str = ""):
    """Checked (known fp32 [*shape] contiguous, mask uint8 [*shape[:-1]]) on the device of the job; both or neither."""
    if known is None or known_mask is None:
        raise DittoError(f"known{what} and known_mask{what} go together: the latents of the known frames and which frames they are")
    known = _need_cuda_f32(f"known{what}", known)
    if tuple(known.shape) != tuple(shape):
        raise DittoError(f"known{what} must be {list(shape)}, got {list(known.shape)}")
    if not isinstance(known_mask, torch.Tensor) or known_mask.dtype != torch.bool:
        raise DittoError(f"known_mask{what} must be a bool tensor, True = known frame")
    if tuple(known_mask.shape) != tuple(shape[:-1]):
        raise DittoError(f"known_mask{what} must be {list(shape[:-1])}, got {list(known_mask.shape)}")
    if known.device != dev or known_mask.device != dev:
        raise DittoError(f"known{what} and known_mask{what} must live on {dev}")
    return known, known_mask.to(torch.uint8).contiguous()
