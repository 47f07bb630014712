"""The residual model of residual_ref.py (h263cu_decode_step_device_residual's definition) on every case of the motion
model, without a GPU: (a) against the pictures the oracle actually decoded, where its prediction is visible -- every
8x8 block of an INTER macroblock that carries no coefficients is the prediction itself, so its residual must be 0 --
and (b) against the prediction restated independently with np_restatement.gather_block."""
import numpy as np
import pytest

import np_restatement as R
import residual_ref as RR


def average_sum_of_mvs(s):
    """types.rs:759-768, restated"""
    whole, frac = (s >> 4) * 2, s & 15
    return whole if frac <= 2 else whole + 2 if frac >= 14 else whole + 1


def restated_prediction(ref, inter, mv, w, h):
    cw, ch = (w + 1) // 2, (h + 1) // 2
    mb_w = (w + 15) // 16
    pred = [np.zeros((h, w), np.uint8), np.zeros((ch, cw), np.uint8), np.zeros((ch, cw), np.uint8)]

    def put(p, x, y, block):
        hh, ww = p[y : y + 8, x : x + 8].shape
        p[y : y + 8, x : x + 8] = block[:hh, :ww]

    for i in np.flatnonzero(inter.reshape(-1)):
        X, Y = int(i) % mb_w, int(i) // mb_w
        v = [(int(mv[i, k, 0]), int(mv[i, k, 1])) for k in range(4)]
        for k in range(4):
            x, y = 16 * X + 8 * (k & 1), 16 * Y + 8 * (k >> 1)
            if x < w and y < h:
                put(pred[0], x, y, R.gather_block(ref[0], (x, y), v[k]))
        c = (average_sum_of_mvs(sum(a for a, _ in v)), average_sum_of_mvs(sum(b for _, b in v)))
        for p in (1, 2):
            put(pred[p], 8 * X, 8 * Y, R.gather_block(ref[p], (8 * X, 8 * Y), c))
    return pred


_MODELS = {}


def model(case):
    if case["id"] not in _MODELS:
        pk, opt = RR.packets_of(case)
        _MODELS[case["id"]] = (pk, opt, RR.reference_stream(pk, opt))
    return _MODELS[case["id"]]


@pytest.mark.parametrize("case", RR.CASES, ids=[c["id"] for c in RR.CASES])
def test_residual_is_zero_where_the_oracle_added_nothing(case):
    """(a) the model's prediction is the oracle's own wherever the oracle added no coefficients; intra macroblocks and
    I pictures carry the samples themselves"""
    _, _, refs = model(case)
    checked = 0
    for r in refs:
        if isinstance(r, int):
            continue
        mb_w = r["inter"].shape[1]
        for i, inter in enumerate(r["inter"].reshape(-1)):
            X, Y = i % mb_w, i // mb_w
            for b in range(6):  # Y0..Y3, Cb, Cr
                k = max(b - 3, 0)
                x, y = (16 * X + 8 * (b & 1), 16 * Y + 8 * (b >> 1)) if b < 4 else (8 * X, 8 * Y)
                blk = r[("y", "cb", "cr")[k]][y : y + 8, x : x + 8]
                cur = r["cur"][k][y : y + 8, x : x + 8]
                if not inter:
                    assert np.array_equal(blk, cur), (case["id"], i, b)  # pred 0: the samples themselves
                elif not r["coded"][i] or r["nev"][i, b] == 0:
                    assert blk.size == 0 or not blk.any(), (case["id"], i, b)
                    checked += blk.size
        for k in range(3):
            assert np.array_equal(r["pred"][k].astype(np.int16) + r[("y", "cb", "cr")[k]], r["cur"][k])
        assert r["y"].min() >= -255 and r["y"].max() <= 255
    assert checked > 0 or all(isinstance(r, int) or not r["inter"].any() for r in refs)


@pytest.mark.parametrize("case", RR.CASES, ids=[c["id"] for c in RR.CASES])
def test_prediction_against_the_numpy_restatement(case):
    """(b) every picture's prediction, rebuilt from the oracle's reference planes with np_restatement.gather_block"""
    refs = model(case)[2]
    ref = None
    for r in refs:
        if isinstance(r, int):
            continue
        if r["inter"].any():
            pred = restated_prediction(ref, r["inter"], r["mv"], r["width"], r["height"])
            for k in range(3):
                assert np.array_equal(pred[k], r["pred"][k]), (case["id"], k)
        else:
            assert not any(p.any() for p in r["pred"])
        if not r["disposable"]:
            ref = r["cur"]


def test_some_case_reads_outside_the_picture():
    """the clamp to the picture is exercised: some block's source window leaves the picture"""
    assert any(not isinstance(r, int) and r["leaves"] for c in RR.CASES for r in model(c)[2])
