"""CPU checks of per-utterance text lengths: the host validation of ``text_lengths=``, the C-ABI entry of
ditto_text_context_masked (header, ctypes table, argument errors reported without a device) and the keyword on every
public entry point the lengths reach."""
import ctypes as C
import inspect
import os
import re

import numpy as np
import pytest
import torch

import ditto_tts_b200 as D
from ditto_tts_b200 import _lib, build
from ditto_tts_b200.model import _check_text_lengths
from ditto_tts_b200.ragged import RaggedBatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_valid_lengths_are_plain_ints():
    assert _check_text_lengths(None, [4, 4]) is None
    for v in ([4, 1], (4, 1), torch.tensor([4, 1]), np.array([4, 1], dtype=np.int32), [np.int64(4), 1]):
        out = _check_text_lengths(v, [4, 2])
        assert out == [4, 1] and all(type(z) is int for z in out)


@pytest.mark.parametrize("bad,match", [([4], "one length per utterance"), ([4, 1, 1], "one length per utterance"),
                                       ([True, 1], "bool"), ([0, 1], "outside"), ([4, 3], "outside"), ([-1, 1], "outside"),
                                       ([2.0, 1], "integer"), ("ab", "sequence"), (3, "sequence")])
def test_bad_lengths_raise(bad, match):
    with pytest.raises(D.DittoError, match=match):
        _check_text_lengths(bad, [4, 2])


def test_header_and_ctypes_entry():
    src = open(os.path.join(ROOT, "include", "ditto_b200.h")).read()
    decl = re.search(r"int32_t ditto_text_context_masked\(([^)]*)\)", src)
    assert decl and "const int64_t* text_len" in decl.group(1)
    res, args = _lib.SIGNATURES["ditto_text_context_masked"]
    assert res is C.c_int32 and len(args) == 9 and args[4] is C.POINTER(C.c_int64)


def test_c_call_reports_bad_arguments():
    build.build()
    lib = _lib.load()
    lens = (C.c_int64 * 2)(1, 2)
    assert lib.ditto_text_context_masked(None, None, 2, 2, lens, None, None, 0, None) == -1
    assert lib.ditto_text_context_masked(None, None, 2, 2, None, None, None, 0, None) == -1
    assert b"text_len" in lib.ditto_last_error()


def test_every_entry_point_takes_text_lengths():
    for fn in (D.DiTTO.text_context, D.DiTTO.forward, D.DiTTO.forward_ragged, D.DiTTOSampler.predict_noise,
               D.DiTTOSampler.p_sample, D.DiTTOSampler.sample_latents, D.DiTTOSampler.sample_latents_ragged, RaggedBatch.__init__):
        p = inspect.signature(fn).parameters.get("text_lengths")
        assert p is not None and p.default is None, fn.__qualname__
