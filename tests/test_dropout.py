"""Fused dropout after the ReLU (include/egc_b200.h, egc_dropout): what can be checked without a GPU - the host model of
the mask, the constants, the interface and the argument guards that fire before anything reaches the device."""
import inspect
import os
import re

import numpy as np
import pytest
import torch

import egc_b200
from egc_b200 import _lib
from egc_b200.functional import check_dropout, dropout_constants as lib_constants
from tests.dropout_model import dropout_constants, keep_mask, philox4x32_10

NEW_SYMBOLS = ["egc_aggregate_fwd_dropout", "egc_aggregate_fwd_bf16_dropout"]


def test_philox_known_answer():
    # Random123 known-answer vector of Philox4x32-10, zero counter and zero key
    assert [int(w) for w in philox4x32_10(0, 0, 0, 0, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


@pytest.mark.parametrize("seed,ctr,expect", [
    # computed with PyTorch's host Philox engine (ATen/core/PhiloxRNGEngine.h: key = seed, counter = (offset lo, offset hi,
    # 0, 0)), an implementation independent of the model under test
    (0x0123456789ABCDEF, (5, 77), [0xA913728E, 0x71C49528, 0x1799ECBA, 0x3A5EE636]),
    (0x7FFFFFFFFFFFFFFF, (31, 169342), [0xAD7FFCDC, 0x877543AD, 0x502EFBE9, 0xB5C1EB06]),
])
def test_philox_nonzero_counter_and_key(seed, ctr, expect):
    words = philox4x32_10(ctr[0], ctr[1], 0, 0, seed & 0xFFFFFFFF, seed >> 32)
    assert [int(w) for w in words] == expect


def test_keep_mask_layout():
    seed, p = 0x0123456789ABCDEF, 0.5
    m = keep_mask(seed, 77, 1, 24, p)
    t, _ = dropout_constants(p)
    words = philox4x32_10(5, 77, 0, 0, seed & 0xFFFFFFFF, seed >> 32)     # columns 20..23 of global row 77
    assert list(m[0, 20:24]) == [int(w) < t for w in words]
    # a block of rows starting at row 70 holds rows 70.. of the mask: the mask is keyed by the global row
    assert np.array_equal(keep_mask(seed, 0, 100, 13, p)[70:], keep_mask(seed, 70, 30, 13, p))


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9, 1e-3, 0.999, 2.0 ** -60])
def test_constants(p):
    t, k = dropout_constants(p)
    p32 = float(np.float32(p))
    assert t == min(int(np.floor((1.0 - p32) * 2.0 ** 32)), 2 ** 32 - 1)
    assert k == float(np.float32(1.0 / (1.0 - p32)))
    assert lib_constants(p) == (t, k)


@pytest.mark.parametrize("p", [-0.1, 1.0, 1.5, float("nan")])
def test_check_dropout_rejects(p):
    with pytest.raises(ValueError):
        check_dropout(p)


def test_check_dropout_accepts():
    assert check_dropout(0) == 0.0 and check_dropout(0.5) == 0.5


def test_symbols_declared_and_signed():
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "egc_b200.h")).read()
    for name in NEW_SYMBOLS:
        assert re.search(rf"\b{name}\(", header), name
        assert name in _lib.SIGNATURES, name
    assert "typedef struct egc_dropout" in header
    assert "#define EGC_ABI_VERSION 5" in header
    assert [f for f, _ in _lib.Dropout._fields_] == ["seed", "p", "row_offset"]


def test_public_arguments():
    assert inspect.signature(egc_b200.EGConv.forward).parameters["dropout"].default == 0.0
    assert inspect.signature(egc_b200.functional.egconv).parameters["dropout_seed"].default is None
    assert inspect.signature(egc_b200.dist.partitioned_egconv).parameters["dropout"].default == 0.0
    stack = egc_b200.EGC(32, 3, 0.5, 4, 4, ["symnorm"], in_features=16, out_rounded=40, out_true=40)
    assert stack.fused_dropout is False
    on = egc_b200.EGC(32, 3, 0.5, 4, 4, ["symnorm"], in_features=16, out_rounded=40, out_true=40, fused_dropout=True)
    assert on.fused_dropout is True
    assert list(on.state_dict()) == list(stack.state_dict())
    with pytest.raises(TypeError):                    # keyword-only, and never handed to EGConv
        egc_b200.EGC(32, 3, 0.5, 4, 4, ["symnorm"], 16, 40, 40, True)


def test_layer_runs_on_cuda_only():
    conv = egc_b200.EGConv(16, 32, aggrs=["symnorm"], num_heads=4, num_bases=4)
    with pytest.raises(RuntimeError):
        conv(torch.zeros(4, 16), torch.zeros(2, 0, dtype=torch.long), relu=True, dropout=0.5)
