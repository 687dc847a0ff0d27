"""GPU (-m gpu): every GEMM step of the bf16 training kernels against float64 on the operands the kernels saved.

The training forward and knerf_mlp_backward save the exact operand of each step as per-tile records (tc_layout.cuh).
tests/tc_chain_oracle.py decodes them, so each layer of tc_mlp_fwd_kernel, tc_mlp_dgrad_kernel, tc_wgrad_kernel and
tc_finish_kernel is checked to an fp32-summation bound -- tight enough that a dropped or doubled tile fails it: with a
10x margin at 1,547 tiles, and narrowly at 6,144 (test_w2_bound_resolves_one_tile) -- where
test_gpu_tc.py compares the whole chain with the fp32 mode at bf16 tolerances.  A failure names the kernel, the layer
and the worst element."""
import ctypes as C

import pytest
import torch

import oracle as O
import tc_chain_oracle as T

pytestmark = pytest.mark.gpu

# Bounds.  PE: 1 bf16 ulp plus 2^-14: fast_sincos is accurate to ~2^-20.7 on the reduced range (MUFU 2^-21.4 plus the
# rounding of the reduced argument), and each of up to five angle doublings about doubles the error (mlp_tc.cu;
# measured 3.05e-5 = 2^-15.0 at most, on scene rays and for |p| up to 100 alike).
PE_ABS = 2.0 ** -14
INEXACT_MAX = 1e-3      # F2 / D2: elements whose bf16 value differs from the bf16 rounding of the exact step


def grad_c(run, rec):
    """W1 for the tensors of the heads task and the fp32 scratch: |g - ref| <= c sum |terms| + M 2^-126 per element, with
    c = 2^-24 x the MMA count of the longest work item (8 MMAs per tile with bf16 records, 4 with fp8), at least 2^-16.
    (The hidden layers get a bound per work item: hidden_grads.)  M 2^-126: fp32 subnormals are flushed to zero."""
    longest = max(hi - lo for _, _, lo, hi in T.work_items(run.n, rec == "fp8"))
    return max(2.0 ** -16, 2.0 ** -24 * longest * (8 if rec == "bf16" else 4))


CHUNK_TILES = 1024      # the float64 references run over tile ranges of this size (bounded memory)


def _rays(R, S, seed=0, wide=False):
    """test_gpu_tc.py's rays; `wide`: origins in [-60, 60]^3 and depths in [0, 40], so |p| reaches 100 per coordinate
    (the range of fast_sincos' two-term reduction; LLFF scenes without NDC reach ~37)"""
    g = torch.Generator().manual_seed(seed)
    o = torch.zeros(R, 3)
    o[:, 2] = 4.0
    d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g) * 0.2 + torch.tensor([0, 0, -1.0]), dim=-1)
    t = torch.sort(torch.rand(R, S, generator=g) * 4 + 2, dim=-1).values.contiguous()
    if wide:
        o = torch.rand(R, 3, generator=g) * 120 - 60
        d = torch.nn.functional.normalize(torch.randn(R, 3, generator=g), dim=-1)
        t = torch.sort(torch.rand(R, S, generator=g) * 40, dim=-1).values.contiguous()
    tgt = torch.rand(R, 3, generator=g)
    dev = torch.device("cuda")
    return o.to(dev), d.to(dev), t.to(dev), tgt.to(dev)


def _fwd(m, net, o, d, t, training, flags=0):
    from keras_nerf_b200 import _lib
    R, S = t.shape
    out = torch.full((R, S, 4), float("nan"), device=t.device)
    _lib.call("knerf_mlp_forward", C.byref(m.cfg), _lib.ptr(net.params), m._packed_ptr("fine" if net is m.fine else "coarse"),
              _lib.ptr(o), _lib.ptr(d), _lib.ptr(t), R, S, (m._prec_train if training else m._prec) | flags, int(training), _lib.ptr(out), m._ws.data_ptr(),
              m._ws.numel(), _lib.stream())
    return out


SHAPES = [(1, 64), (1, 128), (1, 129), (2, 192), (4, 128), (37, 192), (1031, 192), (4096, 192)]
# (model, weights, R, S, rays): the default model at every shape, then other embeddings and weight sets
CASES = ([("default", "init", R, S, "scene") for R, S in SHAPES]
         + [("default", "scaled", 37, 192, "scene"), ("default", "scaled", 1031, 192, "scene"),
            ("default", "init", 1031, 192, "wide"),
            ("layers6_skip4", "init", 300, 192, "scene"), ("layers6_skip4", "scaled", 300, 192, "scene"),
            ("units128", "init", 1031, 192, "scene"), ("pos_emb_6_2", "init", 1031, 192, "scene")])
MODELS = {"default": {}, "layers6_skip4": dict(n_layers=6, skip_layer=4), "units128": dict(dense_units=128),
          "pos_emb_6_2": dict(pos_emb_xyz=6, pos_emb_dir=2)}


def _report(case, name, value, bound):
    print(f"\n[tc-layers] {case} {name} {value:.4g} (bound {bound:.4g})", end="")


class Run:
    """One model in both record formats on the same weights and rays: the training forward, the compositing backward
    (its d_pre drives both backward calls) and knerf_mlp_backward into a gradient buffer with guard bands.  Keeps a
    copy of each workspace, the packed weights and the gradients."""

    def __init__(self, case):
        import keras_nerf_b200 as K
        from keras_nerf_b200 import _lib
        from keras_nerf_b200.model.nerf import mlp as mlp_mod
        model, weights, R, S, rays = case
        self.name = "-".join(map(str, case))
        self.case, self.hidden_cache = case, {}
        self.cfg = O.NerfConfig(**MODELS[model])
        self.ch = T.Chain(self.cfg)
        self.R, self.S, self.M = R, S, R * S
        self.n = T.n_tiles(self.M)
        ms = {}
        for rec in ("bf16", "fp8"):
            mlp_mod.set_seed(42)
            m = K.NeRF(precision="bf16", records=rec, **MODELS[model])
            m.compile(optimizer="adam", loss="mse", batch_size=1, image_height=1, image_width=R, ray_chunks=R,
                      white_background=True)
            assert m.precision == "bf16"
            ms[rec] = m
        self.o, self.d, self.t, tgt = _rays(R, S, seed=R + S, wide=rays == "wide")
        p = ms["bf16"].fine.params.clone()
        g = torch.Generator(device="cuda").manual_seed(5)
        for L in range(len(self.ch.shapes)):     # non-zero biases everywhere
            b = self.ch.bias(p, L)
            b.copy_(0.05 * torch.randn(b.shape, generator=g, device="cuda"))
        if weights == "scaled":
            self._scale_hidden(p)
        self.params = p
        for m in ms.values():
            m.fine.params.copy_(p)
            m._repack()
        self.packed = ms["bf16"]._packed["fine"].clone()
        self.ws, self.out, self.grads, self.guards = {}, {}, {}, {}
        for rec, m in ms.items():
            out = _fwd(m, m.fine, self.o, self.d, self.t, True)
            if rec == "bf16":
                dpre, sq = torch.empty(R, S, 4, device="cuda"), torch.empty(R, device="cuda")
                _lib.call("knerf_composite_backward", _lib.ptr(out), _lib.ptr(self.t), R, S, 1, 1, 1e-10, None,
                          _lib.ptr(tgt), 2.0 / (3 * R), 1, _lib.ptr(dpre), _lib.ptr(sq), _lib.stream())
                self.dpre = dpre.view(self.M, 4)
            G, n = 4096, p.numel()
            guarded = torch.zeros(n + 2 * G, device="cuda")
            _lib.call("knerf_mlp_backward", C.byref(m.cfg), _lib.ptr(m.fine.params), m._packed_ptr("fine"),
                      _lib.ptr(dpre), R, S, m._prec_train, guarded[G:G + n].data_ptr(), m._ws.data_ptr(), m._ws.numel(),
                      _lib.stream())
            torch.cuda.synchronize()
            rb, db = (T.REC8_BYTES, T.DZ8_BYTES) if rec == "fp8" else (T.REC_BYTES, T.DZ_BYTES)
            self.ws[rec] = m._ws[:T.X_BYTES + self.n * (rb + db)].clone()
            self.out[rec] = out.view(self.M, 4)
            self.grads[rec] = guarded[G:G + n].clone()
            self.guards[rec] = float(torch.cat([guarded[:G], guarded[G + n:]]).abs().max())
        del ms
        torch.cuda.empty_cache()
        if weights == "scaled":
            hmax = max(float(self.h(c).max()) for c in range(8))
            _report(self.name, "scaled weights: largest activation", hmax, T.E4M3_MAX)
            assert 16.0 <= hmax < T.E4M3_MAX

    def _scale_hidden(self, p):
        """scale each hidden layer (kernel and bias) so that the float64 forward's largest activation of chain layer c
        is 2^(c - 1): h7 reaches 2^6 while the smallest non-zero activations lie far below 2^-9 (e4m3 subnormals)"""
        pts, dirs = T.sample_points(self.o, self.d, self.t, self.n)
        xs = T.pe_reference(pts, 10, 64, 63)
        h = None
        for c in range(8):
            A = xs if c == 0 else (torch.cat([h, xs], 1) if c == 5 else h)
            W, b = self.ch.fwd_weight(p, c)
            z = torch.relu(A @ W + b)
            L = self.ch.cmap[c]
            if L >= 0:
                f = 2.0 ** (c - 1) / float(z.max())
                self.ch.kernel(p, L).mul_(f)
                self.ch.bias(p, L).mul_(f)
                z = z * f
            h = z

    # ---- decoded records ----
    def tiles(self, rec, dz, off, nbytes):
        return T.tile_bytes(self.ws[rec], self.n, rec == "fp8", dz, off, nbytes)

    def h(self, c):                     # bf16 records: h_c [n * 128, 256]
        return T.decode_bf16(self.tiles("bf16", False, T.REC_H0 + c * T.HS, T.HS), 256)

    def xs(self):
        return T.decode_bf16(self.tiles("bf16", False, T.REC_XS, 16384), 64)

    def ds(self):
        return T.decode_bf16(self.tiles("bf16", False, T.REC_DS, 8192), 32)

    def mask(self, rec, c):
        off = (T.REC8_MASK if rec == "fp8" else T.REC_MASK) + c * T.MASK_LAYER
        return T.decode_mask(self.tiles(rec, False, off, T.MASK_LAYER))

    def dz(self, c):                    # bf16 records: dZ_c
        return T.decode_bf16(self.tiles("bf16", True, T.DZ_Z0 + c * T.HS, T.HS), 256)

    def h8(self, c):
        return T.decode_fp8(self.tiles("fp8", False, T.REC8_H0 + c * T.H8, T.H8), 256, torch.float8_e4m3fn)

    def xs8(self):
        return T.decode_fp8(self.tiles("fp8", False, T.REC8_XS, 8192), 64, torch.float8_e4m3fn)

    def ds8(self):
        return T.decode_fp8(self.tiles("fp8", False, T.REC8_DS, 4096), 32, torch.float8_e4m3fn)

    def dz8(self, c):
        return T.decode_fp8(self.tiles("fp8", True, T.DZ8_Z0 + c * T.H8, T.H8), 256, torch.float8_e5m2)

    def dpre_op(self, rec):
        """the packed (d rgb_pre, d sigma_pre) operand, as the weight-gradient GEMMs read it (fp8: divided by the scale)"""
        if rec == "bf16":
            return T.decode_bf16(self.tiles("bf16", True, T.DZ_P, 4096), 16).double()
        return T.decode_fp8(self.tiles("fp8", True, T.DZ8_P, 2048), 16, torch.float8_e5m2).double() * self.inv_scale()

    def xbuf(self, rec):
        return self.ws[rec][:T.X_BYTES].view(torch.float32)

    def amax_bits(self):
        return int(self.xbuf("fp8").view(torch.int32)[T.X_AMAX])

    def inv_scale(self):
        return T.dz8_scale(self.amax_bits(), inverse=True)

    def operand(self, c, rec):
        """A operand of forward step c (also the weight-gradient GEMM's A of chain layer c), float64"""
        if rec == "bf16":
            xs, hp = self.xs().double(), (self.h(c - 1).double() if c > 0 else None)
        else:
            xs, hp = self.xs8().double(), (self.h8(c - 1).double() if c > 0 else None)
        return xs if c == 0 else (torch.cat([hp, xs], 1) if c == 5 else hp)

    def head_packed(self):
        return self.packed[T.HEAD_OFF:T.HEAD_OFF + T.HEAD_ROWS * 16].view(torch.float32).view(T.HEAD_ROWS, 4)

    def fold_packed(self):
        return self.packed[T.FOLD_OFF:T.FOLD_OFF + 257 * 128 * 4].view(torch.float32).view(257, 128)


@pytest.fixture(scope="module", params=CASES, ids=lambda c: "-".join(map(str, c)))
def run(request):
    r = Run(request.param)
    yield r
    del r
    torch.cuda.empty_cache()


def _amax(x):
    """max |x| (0 for an empty tensor)"""
    return float(x.float().abs().max()) if x.numel() else 0.0


def _ratio(err, bound):
    """err / bound, where a zero bound admits only a zero error"""
    return torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, float("inf"), 0.0))


# ---- forward ---------------------------------------------------------------------------------------------------
def test_f1_encoding_records(run):
    """F1: PE(xyz) and PE(dir) records against the float64 encoding of the fp32 sample point"""
    pts, dirs = T.sample_points(run.o, run.d, run.t, run.n)
    res = {}
    for name, rec, ref in (("PE(xyz)", run.xs(), T.pe_reference(pts, 10, 64, 63)),
                           ("PE(dir)", run.ds(), T.pe_reference(dirs, 4, 32, 31))):
        rec = rec.double()
        err = (rec - ref).abs()
        bound = T.ulp_bf16(torch.maximum(ref.abs(), rec.abs())) + PE_ABS
        res[name] = float((err / bound).max())
        excess = (err - T.ulp_bf16(torch.maximum(ref.abs(), rec.abs()))).clamp_min(0)
        _report(run.name, f"F1 {name} worst / bound", res[name], 1.0)
        _report(run.name, f"F1 {name} largest error beyond 1 ulp", float(excess.max()), PE_ABS)
    _report(run.name, "F1 max |p|", float(pts.abs().max()), 100.0)
    xs, ds = run.xs().float(), run.ds().float()
    assert bool((xs[:, 63] == 1).all()) and bool((ds[:, 31] == 1).all())
    assert float(ds[:, 27:31].abs().max()) == 0.0
    for name, v in res.items():
        assert v <= 1.0, name


def test_f2_hidden_layers(run):
    """F2: h_c = bf16(relu(A_c bf16(W_c) + bf16(b_c))) for every chain layer, every tile (padding rows included)"""
    fails = []
    for c in range(8):
        A, rec = run.operand(c, "bf16"), run.h(c)
        W, b = run.ch.fwd_weight(run.params, c)
        Wb, bb = T.bf16(W), T.bf16(b)
        worst, inexact = _chunked_step_check(rec, A, lambda a: torch.relu(a @ Wb + bb),
                                             lambda a: a.abs() @ Wb.abs() + bb.abs())
        _report(run.name, f"F2 h{c} worst / bound", worst[0], 1.0)
        _report(run.name, f"F2 h{c} inexact fraction", inexact, INEXACT_MAX)
        if worst[0] > 1.0 or inexact > INEXACT_MAX:
            fails.append((f"h{c}", worst[0], inexact, worst[1]))
    assert not fails, fails


def _chunked_step_check(rec, A, exact_of, absum_of, mask=None):
    """T.step_check over tile ranges: (worst ratio, where), inexact fraction"""
    worst, where, n_inexact = 0.0, "", 0.0
    for r0 in range(0, A.shape[0], CHUNK_TILES * T.TILE):
        rows = slice(r0, r0 + CHUNK_TILES * T.TILE)
        a = A[rows]
        exact, absum = exact_of(a), absum_of(a)
        if mask is not None:
            exact, absum = exact * mask[rows], absum * mask[rows]
        w, inexact = T.step_check(rec[rows], exact, absum)
        n_inexact += inexact * a.shape[0]
        if w > worst:
            i = int((rec[rows].double() - exact).abs().argmax())
            worst, where = w, f"tile {(r0 + i // 256) // T.TILE} row {(r0 + i // 256) % T.TILE} col {i % 256}"
    return (worst, where), n_inexact / A.shape[0]


def test_f3_relu_bits(run):
    """F3: the ReLU' bits are h_c > 0 bit for bit, padding rows included; the fp8-records run writes the same bits"""
    for c in range(8):
        m = run.mask("bf16", c)
        assert torch.equal(m, run.h(c).float() > 0), c
        assert torch.equal(m, run.mask("fp8", c)), c


def test_f4_heads(run):
    """F4: the fp32 folded heads against float64 products of the parameters, and the output against sigmoid / relu of
    the float64 last step on the decoded h7 and PE(dir) with the packed heads' bf16 + residual split"""
    fold, head, afold, ahead = T.fold_reference(run.ch, run.params)
    # fold_kernel: W' by U fmas in order, then the heads W' W_c over H = U / 2 products and a 7-level shuffle tree, each
    # step one fp32 rounding of a sum whose |terms| add up to at most the |.| product: K 2^-24, K = U + 1 and U + 1 + 8
    U = run.ch.U
    for name, got, ref, aref, K in (("W'", run.fold_packed(), fold, afold, U + 1),
                                    ("heads", run.head_packed(), head, ahead, U + 9)):
        err = (got.double() - ref).abs()
        r = float(_ratio(err, K * 2.0 ** -24 * aref).max())
        _report(run.name, f"F4 {name} worst / bound (K 2^-24 |.| products)", r, 1.0)
        _report(run.name, f"F4 {name} max err / max |ref|", float(err.max() / ref.abs().max()), 1.0)
        assert r <= 1.0, (name, r)
    hp = run.head_packed()
    w = T.fold_split(hp)
    A = torch.cat([run.h(7).double(), run.ds().double()], 1)
    z = A @ w[:288] + w[288]
    az = A.abs() @ w[:288].abs() + w[288].abs()
    ref = torch.cat([torch.sigmoid(z[:, :3]), torch.relu(z[:, 3:])], 1)[:run.M]
    err = (run.out["bf16"].double() - ref).abs()
    bound = 2.0 ** -20 * az[:run.M] + 2.0 ** -22
    r = float((err / bound).max())
    _report(run.name, "F4 rgbsigma max err", float(err.max()), float(bound.max()))
    _report(run.name, "F4 rgbsigma worst / bound", r, 1.0)
    assert r <= 1.0


def test_fp8_activation_records(run):
    """fp8 records: every e4m3 record within 1 e4m3 ulp of e4m3(bf16 record) (the fp8 run rounds the fp32 value once,
    the reference twice)"""
    pairs = [("PE(xyz)", run.xs8(), run.xs()), ("PE(dir)", run.ds8(), run.ds())]
    pairs += [(f"h{c}", run.h8(c), run.h(c)) for c in range(8)]
    for name, r8, r16 in pairs:
        ref = T.e4m3(r16.float()).double()
        got = r8.double()
        err = (got - ref).abs()
        assert float((err / T.ulp_fp8(torch.maximum(got.abs(), ref.abs()), 3, -6)).max()) <= 1.0, name
        _report(run.name, f"fp8 {name} fraction != e4m3(bf16)", float((err > 0).double().mean()), 1.0)


# ---- dgrad -----------------------------------------------------------------------------------------------------
def test_d1_dpre_operand(run):
    """D1: bf16(d_pre) / e5m2(d_pre scale) in the packed operand, zero padding columns and rows; amax = max|d_pre|"""
    M = run.M
    op = T.decode_bf16(run.tiles("bf16", True, T.DZ_P, 4096), 16)
    assert torch.equal(op[:M, :4].view(torch.int16), run.dpre.to(torch.bfloat16).view(torch.int16))
    assert float(op[:, 4:].float().abs().max()) == 0 and _amax(op[M:]) == 0
    amax = float(run.dpre.abs().max())
    assert run.amax_bits() == int(torch.tensor([amax]).view(torch.int32))
    scale = T.dz8_scale(run.amax_bits())
    op8 = T.decode_fp8(run.tiles("fp8", True, T.DZ8_P, 2048), 16, torch.float8_e5m2)
    assert torch.equal(op8[:M, :4].view(torch.uint8), T.e5m2(run.dpre * scale).view(torch.uint8))
    assert float(op8[:, 4:].float().abs().max()) == 0 and _amax(op8[M:]) == 0
    _report(run.name, "D1 max|d_pre| * scale", amax * scale, 64.0)


def test_d2_dz_records(run):
    """D2: dZ7 = bf16(mask7 (dpre_op bf16([W''' | w_s])^T)), dZ_c = bf16(mask_c (dZ_{c+1} bf16(W_{c+1}[:U, :U])^T));
    fp8: e5m2(scale dZ) within 1 e5m2 ulp of the bf16 run's"""
    M = run.M
    fails = []
    dpre = run.dpre_op("bf16")[:, :4]
    B = T.bf16(run.head_packed()[:256].double())                       # [n][k]: one bf16 rounding, no residual
    A, Bw = dpre, B
    scale = T.dz8_scale(run.amax_bits())
    for c in range(7, -1, -1):
        if c < 7:
            A, Bw = run.dz(c + 1).double(), T.bf16(run.ch.bwd_weight(run.params, c + 1))
        mask = run.mask("bf16", c)
        rec = run.dz(c)
        worst, inexact = _chunked_step_check(rec, A, lambda a: a @ Bw.T, lambda a: a.abs() @ Bw.abs().T, mask)
        _report(run.name, f"D2 dZ{c} worst / bound", worst[0], 1.0)
        _report(run.name, f"D2 dZ{c} inexact fraction", inexact, INEXACT_MAX)
        if worst[0] > 1.0 or inexact > INEXACT_MAX:
            fails.append((f"dZ{c}", worst[0], inexact, worst[1]))
        assert _amax(rec[M:]) == 0, c
        ref8 = T.e5m2(rec.float() * scale).double()
        got8 = run.dz8(c).double()
        err8 = (got8 - ref8).abs()
        r8 = float((err8 / T.ulp_fp8(torch.maximum(got8.abs(), ref8.abs()), 2, -14)).max())
        _report(run.name, f"D2 fp8 dZ{c} fraction != e5m2(scale bf16 dZ)", float((err8 > 0).double().mean()), 1.0)
        if r8 > 1.0:
            fails.append((f"fp8 dZ{c}", r8))
    assert not fails, fails


# ---- weight gradients ------------------------------------------------------------------------------------------
def hidden_kernel_grad(ch, c, full):
    """the model kernel's rows of A_c^T dZ_c [K, 256]: encoding rows (layer 0), hidden rows, and the concat layer's
    encoding rows behind them"""
    U = ch.U
    if c == 0:
        return full[:ch.dx, :U]
    if c == 5 and ch.x5:
        return torch.cat([full[:U, :U], full[256:256 + ch.dx, :U]])
    return full[:U, :U]


def hidden_grads(run, rec):
    """{chain layer c: (kernel ref, kernel bound, bias ref, bias bound)} of every hidden layer the model has.
    The reference is summed item by item over the weight-gradient kernel's own work items (mlp_tc_bwd.cu build_items),
    and so is the bound: an item of L tiles adds m L MMAs (m = 8 with bf16 records, 4 with fp8) into one fp32 TMEM
    accumulator, the bias sums 16 L samples per thread plus 3 shuffles, and the n items of a task meet in fp32 atomics:
      |g - ref| <= 2^-24 (sum_items m L_i S_i + n S) + M 2^-126,   S_i = sum over the item's tiles of |A|^T |dZ|."""
    if rec in run.hidden_cache:
        return run.hidden_cache[rec]
    ch, U = run.ch, run.ch.U
    inv = 1.0 if rec == "bf16" else run.inv_scale()
    m = 8 if rec == "bf16" else 4
    items = T.work_items(run.n, rec == "fp8")
    tiny = run.M * 2.0 ** -126
    out = {}
    for c in range(8):
        if ch.cmap[c] < 0:
            continue
        A = run.operand(c, rec)
        dZ = (run.dz(c) if rec == "bf16" else run.dz8(c)).double() * inv
        K = A.shape[1]
        kref = torch.zeros(K, 256, dtype=torch.float64, device=A.device)
        kbound = torch.zeros_like(kref)
        bref = torch.zeros(256, dtype=torch.float64, device=A.device)
        bbound = torch.zeros_like(bref)
        groups = [(T.hidden_task(c), slice(0, 256 if c > 0 else K))]
        if c == 5:
            groups.append((T.hidden_task(c, encoding_rows=True), slice(256, K)))
        for task, cols in groups:
            mine = [(lo, hi) for _, k, lo, hi in items if k == task]
            S, Sb = torch.zeros_like(kref[cols]), torch.zeros_like(bref)
            for lo, hi in mine:
                rows = slice(lo * T.TILE, hi * T.TILE)
                a, dz = A[rows, cols], dZ[rows]
                si = a.abs().T @ dz.abs()
                kref[cols] += a.T @ dz
                kbound[cols] += m * (hi - lo) * 2.0 ** -24 * si
                S += si
                if cols.start == 0:            # the bias gradient comes from the task of the hidden rows
                    sbi = dz.abs().sum(0)
                    bref += dz.sum(0)
                    bbound += (16 * (hi - lo) + 3) * 2.0 ** -24 * sbi
                    Sb += sbi
            kbound[cols] += len(mine) * 2.0 ** -24 * S
            bbound += len(mine) * 2.0 ** -24 * Sb
        out[c] = (hidden_kernel_grad(ch, c, kref), hidden_kernel_grad(ch, c, kbound) + tiny, bref[:U], bbound[:U] + tiny)
    run.hidden_cache[rec] = out
    return out


def grad_reference(run, rec, absolute=False):
    """float64 gradients of the head tensors from the decoded operands (fp8: divided by the record scale), plus
    the fp32 scratch Y = h7^T d(rgb_pre), Yd = PE(dir)^T d(rgb_pre), s3 = sum d(rgb_pre).  absolute: the same sums over
    the absolute values of their terms (the scale of an fp32 summation error)."""
    ch, U, H, dd = run.ch, run.ch.U, run.ch.U // 2, run.ch.dd
    f = torch.abs if absolute else (lambda x: x)
    ref = {}
    h7 = f((run.h(7) if rec == "bf16" else run.h8(7)).double()[:, :U])
    ds = f((run.ds() if rec == "bf16" else run.ds8()).double()[:, :dd])
    dR = f(run.dpre_op(rec)[:, :4])
    dp = f(run.dpre.double())
    s3 = dR[:, :3].sum(0) if rec == "bf16" else dp[:, :3].sum(0)     # mlp_tc_bwd.cu dgrad prologue
    ref["sigma kernel"] = h7.T @ dR[:, 3:4]
    ref["sigma bias"] = dp[:, 3:4].sum(0)
    # features / rgb_features / rgb: autograd of the unfolded head layers (mlp.py:42-48), independent of the fold algebra
    # tc_finish_kernel uses.  The sum of d(rgb_pre) the kernels multiply into bias terms is s3; a sample with h7 = 0,
    # PE(dir) = 0 and upstream gradient s3 - sum dR carries the difference (zero with bf16 records).
    hd = ch.heads
    P = {k: f(ch.kernel(run.params, hd[k]).double()).requires_grad_() for k in ("features", "rgb_features", "rgb")}
    B = {k: f(ch.bias(run.params, hd[k]).double()).requires_grad_() for k in ("features", "rgb_features", "rgb")}
    X = torch.cat([h7, torch.zeros(1, U, dtype=torch.float64, device=h7.device)])
    D = torch.cat([ds, torch.zeros(1, dd, dtype=torch.float64, device=h7.device)])
    up = torch.cat([dR[:, :3], f(s3 - dR[:, :3].sum(0))[None]])
    F = X @ P["features"] + B["features"]
    G = torch.cat([F, D], 1) @ P["rgb_features"] + B["rgb_features"]
    rgb = G @ P["rgb"] + B["rgb"]
    (rgb * up).sum().backward()
    for k in P:
        ref[f"{k} kernel"] = P[k].grad
        ref[f"{k} bias"] = B[k].grad
    ref["rgb bias"] = dp[:, :3].sum(0)                                 # from the fp32 d_pre (dgrad prologue)
    scratch = {"Y": torch.zeros(256, 4, dtype=torch.float64, device=h7.device),
               "Yd": torch.zeros(32, 4, dtype=torch.float64, device=h7.device)}
    scratch["Y"][:U, :3] = h7.T @ dR[:, :3]
    scratch["Yd"][:dd, :3] = ds.T @ dR[:, :3]
    scratch["S"] = s3
    return ref, scratch


def _grad_tensors(run, rec):
    g = run.grads[rec]
    out = {}
    for L, (name, fi, fo) in enumerate(run.ch.shapes):
        out[f"{name} kernel"] = run.ch.kernel(g, L)
        out[f"{name} bias"] = run.ch.bias(g, L)
    return out


def _w1_ratios(run, rec, got):
    """{tensor: worst |g - ref| / bound} over every gradient tensor and the fp32 scratch"""
    ratios = {}
    for c, (kref, kbound, bref, bbound) in hidden_grads(run, rec).items():
        L = run.ch.cmap[c]
        ratios[f"layer_{L} kernel"] = float(_ratio((got[f"layer_{L} kernel"].double() - kref).abs(), kbound).max())
        ratios[f"layer_{L} bias"] = float(_ratio((got[f"layer_{L} bias"].double() - bref).abs(), bbound).max())
    ref, scratch = grad_reference(run, rec)
    aref, ascratch = grad_reference(run, rec, absolute=True)
    xb = run.xbuf(rec)
    got_s = {"Y": xb[T.X_Y:T.X_Y + 1024].view(256, 4), "Yd": xb[T.X_YD:T.X_YD + 128].view(32, 4),
             "S": xb[T.X_S:T.X_S + 3]}
    c = grad_c(run, rec)
    for name in list(ref) + list(scratch):
        r, a, g = (ref[name], aref[name], got[name]) if name in ref else (scratch[name], ascratch[name], got_s[name])
        r, a = r.reshape(g.shape), a.reshape(g.shape)
        ratios[name] = float(_ratio((g.double() - r).abs(), c * a + run.M * 2.0 ** -126).max())
    return ratios, got_s


@pytest.mark.parametrize("rec", ["bf16", "fp8"])
def test_w1_weight_gradients(run, rec):
    """W1: every gradient tensor and the fp32 scratch against float64 on the decoded operands; nothing written outside
    the gradient buffer or the scratch rows the model uses"""
    got = _grad_tensors(run, rec)
    ratios, got_s = _w1_ratios(run, rec, got)
    assert set(ratios) == set(got) | {"Y", "Yd", "S"}
    name = max(ratios, key=ratios.get)
    _report(run.name, f"W1 {rec} worst |g - ref| / bound ({name})", ratios[name], 1.0)
    assert run.guards[rec] == 0.0
    assert _amax(got_s["Y"][run.ch.U:]) == 0 and _amax(got_s["Yd"][run.ch.dd:]) == 0
    fails = [(k, v) for k, v in ratios.items() if v > 1.0]
    assert not fails, fails


# W2 at 1,547 and 6,144 tiles.  At 1,547 tiles one tile moves each hidden-layer kernel gradient by more than 10x the W1
# bound (measured 32x with bf16 records, 63x with fp8).  At 6,144 tiles the items are longer and the bound with them: one
# tile's change is only about 1.1x the bound with bf16 records (2.4x with fp8), while the kernel's own error uses up to
# 0.64 of it.  What is asserted there is the detection itself: W1 fails on the kernel's gradients with any of the chosen
# tiles dropped or doubled (measured ratio 1.09 with bf16 records, 2.36 with fp8).
W2_MARGIN = {CASES[len(SHAPES) - 2]: 10.0, CASES[len(SHAPES) - 1]: 1.0}


@pytest.mark.parametrize("rec", ["bf16", "fp8"])
def test_w2_bound_resolves_one_tile(run, rec):
    """W2: for the first tile, the last tile and the tiles on either side of a weight-gradient work-item boundary, every
    hidden-layer kernel gradient computed with that tile dropped or doubled fails W1"""
    if run.case not in W2_MARGIN:
        pytest.skip("W2 runs at 1,547 and 6,144 tiles")
    n = run.n
    items = T.work_items(n, rec == "fp8")
    lows = sorted(lo for _, k, lo, _ in items if k == 1 and lo > 0)
    tiles = sorted({0, n - 1, lows[0] - 1, lows[0], lows[-1]})
    got = _grad_tensors(run, rec)
    margin, detect = float("inf"), float("inf")
    inv = 1.0 if rec == "bf16" else run.inv_scale()
    for c, (kref, kbound, _, _) in hidden_grads(run, rec).items():
        g = got[f"layer_{run.ch.cmap[c]} kernel"].double()
        A = run.operand(c, rec)
        dZ = (run.dz(c) if rec == "bf16" else run.dz8(c)).double() * inv
        for t in tiles:
            rows = slice(t * T.TILE, (t + 1) * T.TILE)
            one = hidden_kernel_grad(run.ch, c, A[rows].T @ dZ[rows])
            margin = min(margin, float(_ratio(one.abs(), kbound).max()))
            for s in (-1.0, 1.0):
                detect = min(detect, float(_ratio((g + s * one - kref).abs(), kbound).max()))
    _report(run.name, f"W2 {rec} smallest one-tile change / W1 bound (tiles {tiles})", margin, W2_MARGIN[run.case])
    _report(run.name, f"W2 {rec} smallest W1 ratio with a tile dropped or doubled", detect, 1.0)
    assert margin > W2_MARGIN[run.case]
    assert detect > 1.0
