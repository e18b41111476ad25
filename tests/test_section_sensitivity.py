"""CPU guard of the bars of tests/test_gpu_section_increments.py (runs under -m "not gpu").

For the guard cases of oracle/section_ref.py (every attention path of the case table, each with its sharpened twin) it
asserts that the bars can still tell a correct kernel from a wrong one:
  (a) the bf16-emulated error floor of every section is at most half its bar (the per-row floor at most half the row bar);
  (b) every planted defect moves the checked error by at least 2.5x its bar, in the default case or in its sharpened twin.
A change that loosens a bar, the sharpening or the inputs until a defect could pass fails here."""
import pytest
import torch

from oracle import section_ref as R

# defects that only exist where the kernels have the structure they break
APPLIES = {
    "keys_from_256_ignored": lambda c: c.T > 256,                       # a second key tile exists
    "score_bias_dropped": lambda c: c.heads * ((c.S + 7) // 8 * 8) * 2 <= c.hidden,   # folded cross-attention only
    "last_token_ignored": lambda c: 1 < c.S <= 256,      # one token of 512 moves the increment by < 2 bars only
}


@pytest.fixture(scope="module")
def evaluated():
    """case name -> (case, reference increments, emulated increments, {(section, defect): increment})."""
    torch.set_num_threads(max(1, min(8, torch.get_num_threads())))
    out = {}
    for name in R.GUARD_CASES:
        for c in R.twins(name):
            _, sd, x, text = R.case_inputs(c)
            want = R.increments(c, sd, x, text)
            emul = {s: R.restated(c, sd, x, text, s, bf16=True) for s in c.sections}
            bad = {(s, d): R.restated(c, sd, x, text, s, defect=(s, d))
                   for s in c.sections if s in R.DEFECTS for d in R.DEFECTS[s] if APPLIES.get(d, lambda _: True)(c)}
            out[c.name] = (c, sd, x, text, want, emul, bad)
    return out


@pytest.mark.parametrize("name", R.GUARD_CASES)
def test_restatement_is_the_oracle(evaluated, name):
    """Without rounding and defects the restatement the floors and defects come from is the oracle itself."""
    for c in R.twins(name):
        c, sd, x, text, want, _, _ = evaluated[c.name]
        for s in c.sections:
            assert R.errors(R.restated(c, sd, x, text, s), want[s])[0] <= 1e-12, (c.name, s)


@pytest.mark.parametrize("name", R.GUARD_CASES)
def test_bf16_floor_is_at_most_half_the_bar(evaluated, name):
    for c in R.twins(name):
        c, _, _, _, want, emul, _ = evaluated[c.name]
        for s in c.sections:
            e, row = R.errors(emul[s], want[s])
            assert e <= R.FLOOR_MARGIN * R.bar(c, "bf16", s), (c.name, s, e)
            rb = R.row_bar(c, "bf16", s)
            assert rb is None or row <= R.FLOOR_MARGIN * rb, (c.name, s, row)


def margin(c, section, got, want):
    """How many bars the checked error of an increment is away from passing (the larger of the global and the row check)."""
    e, row = R.errors(got, want)
    rb = R.row_bar(c, "bf16", section)
    return max(e / R.bar(c, "bf16", section), 0.0 if rb is None else row / rb)


@pytest.mark.parametrize("name", R.GUARD_CASES)
def test_every_planted_defect_clears_the_bar_by_a_margin(evaluated, name):
    cases = [evaluated[c.name] for c in R.twins(name)]
    keys = sorted({k for *_, bad in cases for k in bad})
    assert keys, name
    for key in keys:
        m = max(margin(c, key[0], bad[key], want[key[0]]) for c, _, _, _, want, _, bad in cases if key in bad)
        if key in R.INVISIBLE:
            assert m < 1.0, (name, key, m)          # recorded: below what bf16 rounding lets a test see
        else:
            assert m >= R.DEFECT_MARGIN, (name, key, m)
