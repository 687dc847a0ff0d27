"""CPU: the record decoder and rounding emulation of tests/tc_chain_oracle.py, on tiles encoded in Python by the layout
tc_layout.cuh documents.  The GPU checks of each chain step (test_gpu_tc_layers.py) rest on these."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import oracle as O
import tc_chain_oracle as T


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from keras_nerf_b200 import _lib
    return _lib


@pytest.mark.parametrize("rows", [1, 64, 128, 129, 384, 37 * 192, 1031 * 192, 4096 * 192])
@pytest.mark.parametrize("rec8", [False, True])
def test_layout_reproduces_workspace_bytes(lib, rows, rec8):
    """the restated record sizes and scratch offsets add up to what the library allocates: a changed layout fails
    here instead of being decoded as garbage"""
    oc = O.NerfConfig()
    cfg = lib.Config(oc.n_coarse, oc.n_fine, oc.pos_emb_xyz, oc.pos_emb_dir, oc.n_layers, oc.dense_units,
                     oc.skip_layer, 0, 0)
    prec = lib.BF16 | (lib.REC_FP8 if rec8 else 0)
    assert lib.load().knerf_workspace_bytes(C.byref(cfg), rows, prec, 1) == T.workspace_bytes(rows, rec8)
    assert T.REC_BYTES == 576 * 1024 and T.DZ_BYTES == 548 * 1024
    assert T.REC8_BYTES == 304 * 1024 and T.DZ8_BYTES == 258 * 1024


def _by_formula_bf16(x):
    """chunk-major bytes element by element: (r, c) at (c / 8) * 2048 + r * 16 + (c % 8) * 2"""
    n, Cc = x.shape[0] // 128, x.shape[1]
    raw = x.view(torch.int16).numpy().astype(np.uint16)
    out = np.zeros((n, Cc * 256), np.uint8)
    for t in range(n):
        for r in range(128):
            for c in range(Cc):
                b = (c // 8) * 2048 + r * 16 + (c % 8) * 2
                v = int(raw[t * 128 + r, c])
                out[t, b], out[t, b + 1] = v & 0xFF, v >> 8
    return torch.from_numpy(out)


def test_bf16_decoder_round_trip():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2 * 128, 32, generator=g).to(torch.bfloat16)
    raw = _by_formula_bf16(x)
    assert torch.equal(T.encode_bf16(x), raw)
    assert torch.equal(T.decode_bf16(raw, 32).view(torch.int16), x.view(torch.int16))


@pytest.mark.parametrize("dtype", [torch.float8_e4m3fn, torch.float8_e5m2])
def test_fp8_decoder_round_trip(dtype):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2 * 128, 48, generator=g).to(dtype)
    raw = np.zeros((2, 48 * 128), np.uint8)
    xb = x.view(torch.uint8).numpy()
    for t in range(2):
        for r in range(128):
            for c in range(48):
                raw[t, (c // 16) * 2048 + r * 16 + c % 16] = xb[t * 128 + r, c]
    raw = torch.from_numpy(raw)
    assert torch.equal(T.encode_fp8(x), raw)
    assert torch.equal(T.decode_fp8(raw, 48, dtype).view(torch.uint8), x.view(torch.uint8))


def test_tile_bytes_addresses_records():
    """tile t's forward record at kXBytes + t kRecBytes, its dgrad record behind all n forward records"""
    n = 3
    for rec8 in (False, True):
        rb, db = (T.REC8_BYTES, T.DZ8_BYTES) if rec8 else (T.REC_BYTES, T.DZ_BYTES)
        ws = torch.zeros(T.X_BYTES + n * (rb + db), dtype=torch.uint8)
        for t in range(n):
            ws[T.X_BYTES + t * rb + 100] = 1 + t
            ws[T.X_BYTES + n * rb + t * db + 200] = 11 + t
        assert T.tile_bytes(ws, n, rec8, False, 100, 1).flatten().tolist() == [1, 2, 3]
        assert T.tile_bytes(ws, n, rec8, True, 200, 1).flatten().tolist() == [11, 12, 13]


def test_mask_bit_map_on_hand_built_words():
    """word (h, r, g) at h * 2048 + r * 16 + g * 4; bit 8 t + q is column h * 128 + g * 32 + 4 q + t"""
    raw = np.zeros((1, 4096), np.uint8)
    # h = 1, r = 5, g = 2, bit 8 * 3 + 6 (t = 3, q = 6): column 128 + 64 + 24 + 3 = 219
    w = np.zeros(1, np.uint32)
    w[0] = 1 << (8 * 3 + 6)
    raw[0, 2048 + 5 * 16 + 2 * 4: 2048 + 5 * 16 + 2 * 4 + 4] = w.view(np.uint8)
    # h = 0, r = 127, g = 0, bit 0 (t = 0, q = 0): column 0; and bit 31 (t = 3, q = 7): column 31
    w[0] = 1 | (1 << 31)
    raw[0, 127 * 16: 127 * 16 + 4] = w.view(np.uint8)
    m = T.decode_mask(torch.from_numpy(raw))
    assert m.shape == (128, 256)
    assert sorted(map(tuple, m.nonzero().tolist())) == [(5, 219), (127, 0), (127, 31)]
    g = torch.Generator().manual_seed(2)
    rnd = torch.rand(3 * 128, 256, generator=g) < 0.5
    assert torch.equal(T.decode_mask(T.encode_mask(rnd)), rnd)
    assert torch.equal(T.encode_mask(T.decode_mask(torch.from_numpy(raw))), torch.from_numpy(raw))


@pytest.mark.parametrize("x,want", [(448.0, 448.0), (464.0, 448.0), (465.0, 448.0), (500.0, 448.0), (1e9, 448.0),
                                    (-500.0, -448.0), (2.0 ** -9, 2.0 ** -9), (2.0 ** -10, 0.0),
                                    (2.0 ** -10 * 1.001, 2.0 ** -9), (3 * 2.0 ** -10, 2.0 ** -8),
                                    (7 * 2.0 ** -9, 7 * 2.0 ** -9), (2.0 ** -6 * 1.0625, 2.0 ** -6)])
def test_e4m3_satfinite(x, want):
    """cvt.rn.satfinite.e4m3: round to nearest even, subnormals down to 2^-9 (2^-10 is the tie to 0), finite
    saturation at 448 (464 is the tie between 448 and the NaN code and rounds to 448; above it torch gives NaN)"""
    assert float(T.e4m3(torch.tensor([x])).float()) == want


@pytest.mark.parametrize("x,want", [(57344.0, 57344.0), (61440.0, 57344.0), (70000.0, 57344.0), (-1e9, -57344.0),
                                    (2.0 ** -16, 2.0 ** -16), (2.0 ** -17, 0.0), (1.125, 1.0), (1.375, 1.5)])
def test_e5m2_satfinite(x, want):
    assert float(T.e5m2(torch.tensor([x])).float()) == want


def _bits(x):
    return int(np.array([x], np.float32).view(np.uint32)[0])


@pytest.mark.parametrize("amax,k", [(1.0, 5), (0.75, 6), (0.5, 6), (0.9999, 6), (1.5, 5), (2.0, 4), (63.0, 0),
                                    (64.0, -1), (2.0 ** -20, 25), (3e38, -94), (0.0, 106), (1e-45, 106)])
def test_dz8_scale_table(amax, k):
    """scale = 2^k with max|d_pre| * scale in [32, 64) (kDz8Top = 6); e clamped to [-100, 100]: zero and denormal
    maxima give 2^106, the largest floats 2^-94.  The inverse is 2^-k."""
    s = T.dz8_scale(_bits(amax))
    assert s == 2.0 ** k and T.dz8_scale(_bits(amax), inverse=True) == 2.0 ** -k
    if 2.0 ** -100 <= amax <= 2.0 ** 100:
        assert 32.0 <= amax * s < 64.0


@pytest.mark.parametrize("kw,cmap,x5", [({}, [0, 1, 2, 3, 4, 5, 6, 7], True),
                                        (dict(n_layers=6), [0, 1, 2, 3, 4, 5, -1, -1], True),
                                        (dict(n_layers=4), [0, 1, 2, 3, -1, -1, -1, -1], False),
                                        (dict(n_layers=6, skip_layer=3), [0, 1, 2, 3, -1, 4, 5, -1], True),
                                        (dict(n_layers=7, skip_layer=4), [0, 1, 2, 3, 4, 5, 6, -1], True),
                                        (dict(dense_units=128), [0, 1, 2, 3, 4, 5, 6, 7], True),
                                        (dict(pos_emb_xyz=6, pos_emb_dir=2), [0, 1, 2, 3, 4, 5, 6, 7], True)])
def test_chain_map(kw, cmap, x5):
    """api.cu tc_chain_map: model layers keep their order, the concat layer sits at chain layer 5, the rest are
    identity layers"""
    ch = T.Chain(O.NerfConfig(**kw))
    assert ch.cmap == cmap and ch.x5 == x5
    assert ch.n_params == O.param_count(O.NerfConfig(**kw))


def test_chain_weights_embed_the_model():
    cfg = O.NerfConfig(dense_units=64, pos_emb_xyz=6, pos_emb_dir=2, n_layers=6)
    ch = T.Chain(cfg)
    p = torch.randn(ch.n_params, generator=torch.Generator().manual_seed(3))
    W0, b0 = ch.fwd_weight(p, 0)
    assert W0.shape == (64, 256) and torch.equal(W0[:39, :64], ch.kernel(p, 0).double())
    assert float(W0[39:].abs().max()) == 0 and float(W0[:, 64:].abs().max()) == 0
    W5, _ = ch.fwd_weight(p, 5)
    assert W5.shape == (320, 256)
    assert torch.equal(W5[:64, :64], ch.kernel(p, 5)[:64].double())
    assert torch.equal(W5[256:256 + 39, :64], ch.kernel(p, 5)[64:].double())
    W6, b6 = ch.fwd_weight(p, 6)
    assert torch.equal(W6, torch.eye(256, dtype=torch.float64)) and float(b6.abs().max()) == 0
    assert torch.equal(ch.bwd_weight(p, 7), torch.eye(256, dtype=torch.float64))
    assert torch.equal(ch.bwd_weight(p, 3)[:64, :64], ch.kernel(p, 3).double())


def test_work_items_cover_every_tile_once():
    """the restated item list of the weight-gradient kernel: every (task, tile) exactly once, longest first"""
    for n, rec8 in ((1, False), (1547, False), (6144, True), (6144, False)):
        items = T.work_items(n, rec8)
        seen = np.zeros((10, n), np.int64)
        for _, k, lo, hi in items:
            seen[k, lo:hi] += 1
        assert (seen == 1).all()
        assert all(a[0] >= b[0] for a, b in zip(items, items[1:]))
        assert len(items) <= 1024


def test_item_rule_follows_the_source():
    """the task costs and item-size constants restated in tc_chain_oracle.py are those of mlp_tc_bwd.cu / common.cuh:
    the weight-gradient bound and the tiles W2 picks depend on them"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "keras_nerf_b200", "csrc", "mlp_tc_bwd.cu")).read()
    common = open(os.path.join(root, "keras_nerf_b200", "csrc", "common.cuh")).read()

    def const(text, name):
        return int(re.search(r"constexpr int %s = (\d+);" % name, text).group(1))
    assert const(common, "kNumSMs") == T.NUM_SMS
    assert (const(src, "kHeadsCost"), const(src, "kXpartCost8"), const(src, "kHeadsCost8")) == \
        (T.HEADS_COST, T.XPART_COST8, T.HEADS_COST8)
    assert (const(src, "kWGuide"), const(src, "kWMinShare"), const(src, "kWMinTiles")) == \
        (T.GUIDE, T.MIN_SHARE, T.MIN_TILES)
    table = src[src.index("static WTaskTable build_task_table(int dx"):src.index("static WTaskTable build_task_table8")]
    big = table[table.index("auto big"):table.index("auto xpart")]
    xpart = table[table.index("auto xpart"):table.index("xpart(0,")]
    assert re.findall(r"t\.cost = (\d+);", big) == [str(T.BIG_COST)]
    assert re.findall(r"t\.cost = (\d+);", xpart) == [str(T.XPART_COST)]
    assert re.search(r"min_cost = std::max\(total / kNumSMs / kWMinShare, 128\.0 \* kWMinTiles\)", src)
    assert re.search(r"want = std::max\(min_cost, left / \(kWGuide \* kNumSMs\)\)", src)
    assert "if (n_tiles - lo - n < (n + 1) / 2) n = n_tiles - lo;" in src
