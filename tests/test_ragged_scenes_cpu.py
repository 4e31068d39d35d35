"""Host side of scenes of different sizes: the prefix tables and the weight-gradient slice plan the library writes
(siren_b200_ragged_tables, the host copy of what siren_b200_prepare_ragged writes) against a plain restatement, and
the refusals that need no device."""
import numpy as np
import pytest

from siren_mri_b200 import _lib


def plan(counts, kinds, sms):
    """K (128-row tiles per weight-gradient slice): the longest scene cut into s = 1..64 slices, the first s at which
    min(items / (waves * sms), the total tiles per SM over the longest item) reaches 0.95, else the best."""
    tiles = [-(-n // 128) for n in counts]
    tmax, total = max(tiles), sum(tiles)
    best, best_eff, prev = tmax, 0.0, None
    for s in range(1, min(64, tmax) + 1):
        K = -(-tmax // s)
        if K == prev:
            continue
        prev = K
        items = kinds * sum(-(-t // K) for t in tiles)
        waves = -(-items // sms)
        eff = min(items / (waves * sms), kinds * total / (sms * K))
        if eff > best_eff + 1e-9:
            best_eff, best = eff, K
        if eff >= 0.95:
            break
    return best


def tables(counts, kinds, sms):
    K = plan(counts, kinds, sms)
    unit, prow, xrow, slc = [0], [0], [0], [0]
    for n in counts:
        tiles = -(-n // 128)
        unit.append(unit[-1] + -(-tiles // 4))          # units: two 256-row tiles of a CTA pair
        prow.append(prow[-1] + 128 * tiles)
        xrow.append(xrow[-1] + n)
        slc.append(slc[-1] + -(-tiles // K))
    return unit + prow + xrow + slc + [K]


def desc_for(T, nh=3, d=2, o=1, prec="bf16", per_task=1):
    desc = _lib.SirenDesc()
    desc.d_in, desc.hidden, desc.n_hidden, desc.d_out = d, 256, nh, o
    desc.w0, desc.tasks, desc.per_task, desc.n_coords = 30.0, T, per_task, 1
    desc.precision, desc.deriv_order = _lib.PRECISIONS[prec], 0
    return desc


def lib_tables(counts, nh, sms):
    import ctypes
    out = (ctypes.c_int * (4 * (len(counts) + 1) + 1))()
    rc = _lib.load().siren_b200_ragged_tables(desc_for(len(counts), nh), _lib.long_array(counts), sms, out)
    return rc, list(out)


CASES = {
    "edges": [1, 127, 128, 129, 255, 256, 257, 511, 512, 513, 4097, 65536],
    "eq64x4096": [4096] * 64,
    "mix16": [4096, 16384, 65536, 262144] * 4,
    "one": [262144],
    "many_tiny": [1] * 1024,
    "random": list(np.random.default_rng(1).integers(1, 200000, size=37)),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("nh,sms", [(1, 148), (3, 148), (4, 132), (2, 8)])
def test_tables_match_restatement(case, nh, sms):
    counts = [int(c) for c in CASES[case]]
    rc, got = lib_tables(counts, nh, sms)
    assert rc == 0, _lib.load().siren_b200_last_error()
    assert got == tables(counts, nh, sms)
    T = len(counts)
    slc = got[3 * (T + 1):4 * (T + 1)]
    K = got[-1]
    for t, n in enumerate(counts):
        tiles = -(-n // 128)
        s = slc[t + 1] - slc[t]
        assert 1 <= s <= tiles and -(-tiles // s) <= K      # a slice per K tiles, at least one per scene


def test_equal_counts_split_like_equal_n():
    """64 scenes of 4096 coordinates (32 tiles), three hidden layers, 148 SMs: three slices per scene, the split the
    equal-N plan picks (576 items in four waves)."""
    _, got = lib_tables([4096] * 64, 3, 148)
    slc = got[3 * 65:4 * 65]
    assert all(b - a == 3 for a, b in zip(slc, slc[1:]))


def test_small_scenes_pay_for_their_tiles_only():
    """One large scene and 63 thumbnails: a thumbnail has one slice, the large scene as many as its tiles call for."""
    counts = [512 * 512] + [64 * 64] * 63
    _, got = lib_tables(counts, 3, 148)
    slc = got[3 * 65:4 * 65]
    per = [b - a for a, b in zip(slc, slc[1:])]
    assert all(p == 1 for p in per[1:]) and per[0] > 1


def test_one_large_scene_among_many_tiny_ones_is_cut():
    """1024 one-tile scenes fill the waves by themselves; the large scene is still cut so that no item outlasts them."""
    counts = [262144] + [100] * 1023
    _, got = lib_tables(counts, 3, 148)
    slc = got[3 * 1025:4 * 1025]
    assert slc[1] - slc[0] >= 32 and got[-1] <= 64


@pytest.mark.parametrize("counts,kw,rc", [
    ([10, 0], {}, 2), ([-1], {}, 2), ([10, 20], dict(per_task=0), 2), ([10], dict(prec="fp32"), 1),
    ([10], dict(d=5), 1), ([10], dict(o=3), 1), ([10], dict(nh=5), 1), ([10] * 1025, {}, 1),
])
def test_refusals(counts, kw, rc):
    import ctypes
    lib = _lib.load()
    out = (ctypes.c_int * (4 * (len(counts) + 1) + 1))()
    n_c = _lib.long_array(counts)
    d = desc_for(len(counts), **kw)
    assert lib.siren_b200_ragged_tables(d, n_c, 148, out) == rc
    assert lib.siren_b200_workspace_bytes_ragged(d, n_c) == 0


def test_workspace_follows_the_sum_of_counts():
    lib = _lib.load()
    small = lib.siren_b200_workspace_bytes_ragged(desc_for(64), _lib.long_array([4096] * 63 + [262144]))
    padded = desc_for(64)
    padded.n_coords = 262144
    assert 0 < small < lib.siren_b200_workspace_bytes_ex(padded, 0) / 10


def test_trainer_rejects_bad_counts():
    """Checked before anything touches the device."""
    from siren_mri_b200 import modules
    from siren_mri_b200.trainer import SirenTrainer
    m = lambda: modules.SingleBVPNet(in_features=2, out_features=1)  # noqa: E731
    with pytest.raises(ValueError, match="counts"):
        SirenTrainer([m(), m()], [64])
    with pytest.raises(ValueError, match="positive"):
        SirenTrainer([m(), m()], [64, 0])
