"""Ragged batches at the C5 length mix (BASELINE.json config 5, ``parallel.c5_lengths``) at the repo-default width, guided.

The ragged path runs what uniform batches never do: per-group self-attention, LN2, cross-attention and norm3 on up to
eight side streams (C5 has 19 groups, so groups share streams), per-group slices of the attention scratch, per-group kernel
choices inside one batch, and per-row tables (RoPE positions, t per sequence, x_skip per packed row).  It is pinned
  * per sequence: every row of every utterance equals the same utterance run alone through the uniform path, which
    tests/test_gpu_section_increments.py pins against fp64 section by section;
  * per schedule: the forward on eight side streams is bitwise the forward of a serial engine and of a three-stream one
    (same kernels on the same data, no atomics), and a CUDA-graph sampler step is bitwise its eager run;
  * independently of the CUDA code: one utterance per group against the fp64 oracle at the bf16 bar.
Beside the 19 C5 groups the batch holds edge groups (EDGES, SCRATCH), so that every cross-attention path and max_seq_len
run in the same batch."""
import ctypes as C

import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib
from ditto_tts_b200.parallel import c5_lengths
from ditto_tts_b200.ragged import RaggedBatch
from oracle import ditto_oracle as O  # checker only

pytestmark = pytest.mark.gpu
CFG = O.OracleConfig(768, 2, 1, 256, 768, 50)
W, BAR = 3.0, 2e-2
# (T, S) of the groups beside the C5 ones, two utterances each
EDGES = [
    (1, 1),        # constant text in every sequence; two-CTA self-attention
    (4096, 40),    # max_seq_len: RoPE positions up to 4095, 32 key tiles
]
# groups that use their slice of the attention scratch (group_view), six utterances each: folded cross-attention through
# the scores GEMM + softmax + P.V and a norm3 launch (S = 300, 320); unfolded q / out projections, the two-tile scores +
# softmax kernel with row_lsum and gemm_resid_ln (S = 480, 512).  Each path has a twin on the neighbouring side stream, so
# that two groups run the same scratch kernels at the same time: with one group per path they need not overlap in time, and
# slices that overlapped in memory went unnoticed.
SCRATCH = [(129, 480), (129, 512), (257, 300), (257, 320)]
# kernel classes the batch must reach: self-attention + norm2, cross_fused (S <= 64), <CROSS> (64 < S <= 256), the folded
# P.V of S = 300 / 320, the out-projection + norm3 of S = 480 / 512
KERNELS = ("tc_gemm.flash768_ln", "tc_gemm.cross_fused_ln", "tc_gemm.cross_flash_ln", "tc_gemm.cross_pv", "tc_gemm.cross_out")
ROW_BAR = 1e-5
SIDE = 8    # side streams of the default engine (engine.cu: ditto_engine::kSide)
E_BADARG, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -5


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def models(dev):
    """Three models of the same weights: the default engine (eight side streams), a serial one and a three-stream one.
    side_streams is sampled when an engine is created."""
    sd = O.make_state_dict(CFG, 91)

    def build(side_streams=None):
        m = D.DiTTO(hidden_dim=CFG.hidden_dim, num_layers=CFG.num_layers, num_heads=CFG.num_heads, time_dim=CFG.time_dim,
                    text_dim=CFG.text_dim, diffusion_steps=CFG.diffusion_steps, precision="bf16")
        m.load_state_dict(sd, strict=True)
        m = m.to(dev)
        if side_streams is not None:
            _lib.debug_option("side_streams", side_streams)
        try:
            m.engine()
        finally:
            _lib.debug_option("reset", 0)
        return m

    return sd, {"default": build(), "serial": build(0), "three": build(3)}


def make_job(pairs, seed, device="cpu"):
    """Utterances of the given (T, S): latents, texts, zero null texts, t per utterance."""
    g = torch.Generator(device=device).manual_seed(seed)
    H = CFG.hidden_dim
    xs = [torch.randn(T, H, generator=g, device=device) for T, _ in pairs]
    texts = [torch.randn(S, H, generator=g, device=device) for _, S in pairs]
    t = torch.randint(0, CFG.diffusion_steps, (len(pairs),), generator=g, device=device)
    return xs, texts, t


def c5_pairs(n_utts=256):
    return list(zip(*c5_lengths(n_utts)))


def guided_ragged(m, xs, texts, t, dev):
    """Guided ragged forward: (batch, packed [seq_rows, H] output) with every group laid out [cond; uncond]."""
    texts = [c.to(dev) for c in texts]
    rb = RaggedBatch(m, texts, [x.shape[0] for x in xs], guided=True, null_texts=[torch.zeros_like(c) for c in texts])
    return rb, rb.forward(rb.pack([x.to(dev) for x in xs]), rb.seq_t(t))


def split(rb, out):
    """packed guided output -> per utterance [2, T, H] (cond, uncond): the layout of a uniform guided forward."""
    per, row = [None] * rb.B, 0
    for T, _, idx in rb.groups:
        n = len(idx)
        blk = out[row:row + 2 * n * T].view(2 * n, T, rb.H)
        for j, i in enumerate(idx):
            per[i] = torch.stack([blk[j], blk[n + j]])
        row += 2 * n * T
    return per


def guided_alone(m, x, text, t, dev):
    """The same utterance alone through the uniform path: cond and uncond sequences sharing x (n_x = 1, n_seq = 2)."""
    both = torch.stack([text, torch.zeros_like(text)]).to(dev)
    ctx = m.text_context(both, T_hint=x.shape[0])
    return m.forward_with_context(x[None].to(dev), ctx, t.view(1).repeat(2).to(dev), 2, both.shape[1])


def worst_row(got, want):
    """Largest rel-L2 of one row."""
    got, want = got.double().cpu().flatten(0, -2), want.double().cpu().flatten(0, -2)
    return float(((got - want).norm(dim=-1) / want.norm(dim=-1).clamp_min(1e-300)).max())


def check_against_alone(m, rb, out, xs, texts, t, dev, which):
    """Rows of utterances ``which`` against their uniform runs.  Not bitwise: the row-wise GEMMs (QKV, GLU, fc2, projections)
    run over all packed rows, and the GEMM launcher picks the SM-pair or the one-CTA kernel by M, so they accumulate in
    another order than at the M of one utterance."""
    per = split(rb, out)
    errs = {i: worst_row(per[i], guided_alone(m, xs[i], texts[i], t[i], dev)) for i in which}
    print(f"[ragged-c5] {len(errs)} utterances against their uniform runs: largest row error {max(errs.values()):.2e}")
    bad = [(i, rb.lengths[i], texts[i].shape[0], e) for i, e in errs.items() if not e <= ROW_BAR]
    assert not bad, bad


def one_per_group(rb):
    return [idx[0] for _, _, idx in rb.groups]


@pytest.fixture(scope="module")
def batch(dev, models):
    """Two utterances of every C5 (T, S) and EDGES group, six of every SCRATCH group, run once on each engine and once more
    on the default one."""
    _, ms = models
    pairs = [p for p in sorted(set(c5_pairs())) + EDGES for _ in range(2)] + [p for p in SCRATCH for _ in range(6)]
    xs, texts, t = make_job(pairs, 92)
    _lib.profile_start()
    try:
        rb, out = guided_ragged(ms["default"], xs, texts, t, dev)
    finally:
        prof = _lib.profile_stop()
    outs = {name: guided_ragged(ms[name], xs, texts, t, dev)[1] for name in ("serial", "three")}
    outs["default_again"] = guided_ragged(ms["default"], xs, texts, t, dev)[1]
    return xs, texts, t, rb, out, outs, prof


def differing_groups(rb, a, b):
    """(T, S, largest |difference|) of every group whose rows differ between two packed outputs."""
    diff, row = [], 0
    for T, S, idx in rb.groups:
        rows = 2 * len(idx) * T
        if not torch.equal(a[row:row + rows], b[row:row + rows]):
            diff.append((T, S, float((a[row:row + rows] - b[row:row + rows]).abs().max())))
        row += rows
    return diff


def test_every_sequence_equals_its_uniform_run(dev, models, batch):
    _, ms = models
    xs, texts, t, rb, out, _, prof = batch
    assert [g[:2] for g in rb.groups] == sorted(set(c5_pairs()) | set(EDGES) | set(SCRATCH))
    missing = [k for k in KERNELS if k not in prof]
    assert not missing, (missing, sorted(prof))
    check_against_alone(ms["default"], rb, out, xs, texts, t, dev, range(rb.B))


def test_side_streams_are_bitwise_a_serial_schedule(batch):
    """Eight side streams (25 groups: up to four per stream), three (other groups share a stream) and none: the same bits.
    The groups that use the attention scratch run on four different streams of the default engine, so slices that
    overlapped would race there."""
    *_, rb, out, outs, _ = batch
    keys = [g[:2] for g in rb.groups]
    assert len({keys.index(k) % SIDE for k in SCRATCH}) == len(SCRATCH)
    bad = {name: differing_groups(rb, o, out) for name, o in outs.items()}
    assert not any(bad.values()), bad


def test_graph_step_is_bitwise_the_eager_step(dev, models):
    """A one-step guided ragged job with supplied noise, through a captured step graph (fork / join become parallel
    branches) and eagerly: the same bits.  Thirteen groups, so that groups share side streams inside the graph too."""
    _, ms = models
    pairs = sorted(set(c5_pairs()))[:8] + [(1, 1)] + SCRATCH
    xs, texts, _ = make_job(pairs, 93, device=dev)
    g = torch.Generator(device=dev).manual_seed(94)
    noise = [torch.randn(CFG.diffusion_steps, T, CFG.hidden_dim, generator=g, device=dev) for T, _ in pairs]
    s = D.DiTTOSampler(ms["default"], guidance_scale=W, num_steps=1)
    lengths = [T for T, _ in pairs]
    eager = s.sample_latents_ragged(texts, lengths, x_init=xs, noise=noise, use_graph=False)
    graph = s.sample_latents_ragged(texts, lengths, x_init=xs, noise=noise, use_graph=True)
    bad = [pairs[i] for i in range(len(pairs)) if not torch.equal(graph[i], eager[i])]
    assert not bad, bad
    assert all(bool(torch.isfinite(z).all()) for z in graph)


def test_full_c5_batch(dev, models):
    """All 256 C5 utterances (412 k packed sequence rows) as one guided forward: eight side streams bitwise the serial
    engine, and one utterance per group equal to its uniform run."""
    _, ms = models
    pairs = c5_pairs()
    xs, texts, t = make_job(pairs, 96, device=dev)
    rb, out = guided_ragged(ms["default"], xs, texts, t, dev)
    assert len(rb.groups) == 19 and rb.seq_rows == 2 * sum(T for T, _ in pairs)
    serial = guided_ragged(ms["serial"], xs, texts, t, dev)[1]
    bad = differing_groups(rb, serial, out)
    assert not bad, bad
    del serial
    check_against_alone(ms["default"], rb, out, xs, texts, t, dev, one_per_group(rb))


def test_one_utterance_per_group_against_fp64_oracle(models, batch):
    """The pin that does not depend on the CUDA code: conditional and unconditional rows of one utterance per group against
    the fp64 oracle at the bf16 bar."""
    sd, _ = models
    sd64 = {k: v.double() for k, v in sd.items()}
    xs, texts, t, rb, out, _, _ = batch
    per = split(rb, out)
    bad = []
    for i in one_per_group(rb):
        for k, text in enumerate((texts[i], torch.zeros_like(texts[i]))):
            ref = O.ditto_forward(sd64, CFG, xs[i][None].double(), text[None].double(), t[i:i + 1])[0]
            e = O.rel_l2(per[i][k].cpu(), ref)
            if not e <= BAR:
                bad.append((rb.lengths[i], texts[i].shape[0], "cond" if k == 0 else "uncond", e))
    assert not bad, bad


def test_group_list_edges(dev, models):
    """ditto_forward_ragged refuses a workspace one byte short, a group longer than max_seq_len and more than 4096 groups,
    without launching a kernel; with exactly ditto_workspace_bytes_ragged bytes it runs and gives the bits of a larger
    workspace."""
    _, ms = models
    m, lib = ms["default"], _lib.load()
    pairs = [(150, 13), (300, 26), (129, 512)]
    xs, texts, t = make_job(pairs, 95, device=dev)
    rb = RaggedBatch(m, texts, [T for T, _ in pairs], guided=True)
    x, ts = rb.pack(xs), rb.seq_t(t)
    out = torch.empty(rb.seq_rows, rb.H, device=dev)
    ws = torch.empty(rb.ws_bytes, dtype=torch.uint8, device=dev)
    P = lambda z: C.c_void_p(z.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def forward(groups, n, nbytes):
        return lib.ditto_forward_ragged(m.engine(), P(x), groups, n, P(ts), P(out), P(ws), nbytes, stream)

    too_long = (_lib.SeqGroup * 1)(_lib.SeqGroup(n_seq=2, n_x=1, T=m.max_seq_len + 1, S=13, ctx=rb.c_groups[0].ctx))
    too_many = (_lib.SeqGroup * 4097)(*([rb.c_groups[0]] * 4097))
    torch.cuda.synchronize()
    before = _lib.launch_count()
    assert forward(rb.c_groups, len(rb.groups), rb.ws_bytes - 1) == E_WORKSPACE
    assert forward(too_long, 1, rb.ws_bytes) == E_UNSUPPORTED
    assert lib.ditto_workspace_bytes_ragged(m.engine(), too_long, 1) == -1
    assert forward(too_many, 4097, rb.ws_bytes) == E_BADARG
    assert _lib.launch_count() == before
    assert forward(rb.c_groups, len(rb.groups), rb.ws_bytes) == 0
    assert _lib.launch_count() > before
    assert torch.equal(out, rb.forward(x, ts))
