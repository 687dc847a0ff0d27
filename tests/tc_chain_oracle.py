"""Decoder of the per-tile records the bf16 training kernels save (csrc/tc_layout.cuh) and a float64 reference of
every GEMM step of the chain (mlp_tc.cu, mlp_tc_bwd.cu) on the operands those records hold.

Given the exact operand of a step, its result is fixed up to the fp32 accumulation order, so each step of each kernel
can be checked to within an fp32-summation bound instead of the bf16-versus-fp32 bound of the whole chain.  Nothing
here calls the library's kernels: the layout is restated from tc_layout.cuh (and checked against
knerf_workspace_bytes), the rounding is torch's, the arithmetic float64 torch matmuls.
"""
import torch

import oracle as O

# ---- tc_layout.cuh, restated -------------------------------------------------------------------------------
TILE = 128                                   # kTileM: samples per tile; tile t holds samples 128 t .. 128 t + 127
HS = TILE * 256 * 2                          # kHSBytes: one [128 x 256] bf16 operand, chunk-major
CHUNK = TILE * 16                            # kChunkA: bytes between 8-element (bf16) / 16-element (fp8) chunks
REC_XS, REC_DS, REC_H0 = 0, 16384, 32768     # kRecXS, kRecDS, kRecH0
REC_MASK = REC_H0 + 8 * HS                   # kRecMask
MASK_LAYER = 4096                            # kMaskLayerBytes
REC_BYTES = REC_MASK + 8 * MASK_LAYER        # kRecBytes
DZ_Z0 = 0                                    # kDzZ0
DZ_P = 8 * HS + 32768                        # kDzP = kDzG + 32768
DZ_BYTES = DZ_P + 4096                       # kDzBytes
H8 = TILE * 256                              # kH8Bytes
REC8_XS, REC8_DS, REC8_H0 = 0, 8192, 16384   # kRec8XS, kRec8DS, kRec8H0
REC8_MASK = REC8_H0 + 8 * H8                 # kRec8Mask
REC8_BYTES = REC8_MASK + 8 * MASK_LAYER      # kRec8Bytes
DZ8_Z0, DZ8_P = 0, 8 * H8                    # kDz8Z0, kDz8P
DZ8_BYTES = DZ8_P + 2048                     # kDz8Bytes
DZ8_TOP = 6                                  # kDz8Top
# fp32 scratch at the head of the workspace (float offsets)
X_Y = 4                                      # kXOffY   [256][4]
X_YD = X_Y + 256 * 4                         # kXOffYd  [32][4]
X_S = X_YD + 32 * 4                          # kXOffS   [4]
X_T = X_S + 4                                # kXOffT
X_U = X_T + 256 * 4                          # kXOffU
X_AMAX = X_U + 256 * 4                       # kXOffAmax
X_BYTES = ((X_AMAX + 4) * 4 + 255) // 256 * 256   # kXBytes
# packed weights (byte offsets)
FOLD_OFF = 0                                 # kFoldOff: fp32 W' [256][128], then b' [128]
HEAD_OFF = FOLD_OFF + (256 * 128 + 128) * 4  # kHeadOff: fp32 [289][4]
HEAD_ROWS = 289                              # kHeadRows

E4M3_MAX, E5M2_MAX = 448.0, 57344.0


def n_tiles(M):
    return (M + TILE - 1) // TILE


def workspace_bytes(rows, rec8):
    """knerf_workspace_bytes(cfg, rows, KNERF_BF16 [| KNERF_REC_FP8], training=1): tc_workspace_bytes (mlp_tc.cu) plus
    the chunk-level scratch that api.cu adds"""
    per_tile = (REC8_BYTES + DZ8_BYTES) if rec8 else (REC_BYTES + DZ_BYTES)
    return X_BYTES + n_tiles(rows) * per_tile + 256 + rows * 64 + 8192


def tile_bytes(ws, n, rec8, dz, off, nbytes):
    """[n, nbytes] uint8 view of bytes off .. off + nbytes of every tile's forward (dz = False) or dgrad record.  The
    forward records start after the fp32 scratch, tile t at + t * kRecBytes; the dgrad records follow all n of them
    (mlp_tc_bwd.cu tc_backward: dz = rec + n_tiles * kRecBytes), tile t at + t * kDzBytes."""
    rb = REC8_BYTES if rec8 else REC_BYTES
    base = X_BYTES + (n * rb if dz else 0)
    stride = (DZ8_BYTES if rec8 else DZ_BYTES) if dz else rb
    return ws.as_strided((n, nbytes), (stride, 1), ws.storage_offset() + base + off)


# ---- element maps --------------------------------------------------------------------------------------------
def decode_bf16(tiles, C):
    """[n, C * 256] uint8, chunk-major bf16 (element (r, c) at (c // 8) * 2048 + r * 16 + (c % 8) * 2) -> [n * 128, C]"""
    n = tiles.shape[0]
    x = tiles.contiguous().view(torch.int16).view(n, C // 8, TILE, 8).permute(0, 2, 1, 3).reshape(n * TILE, C)
    return x.view(torch.bfloat16)


def encode_bf16(x):
    """inverse of decode_bf16: [n * 128, C] bf16 -> [n, C * 256] uint8"""
    C = x.shape[1]
    n = x.shape[0] // TILE
    y = x.view(torch.int16).view(n, TILE, C // 8, 8).permute(0, 2, 1, 3).contiguous()
    return y.view(torch.uint8).view(n, C * 2 * TILE)


def decode_fp8(tiles, C, dtype):
    """[n, C * 128] uint8, chunk-major fp8 (element (r, c) at (c // 16) * 2048 + r * 16 + c % 16) -> [n * 128, C]"""
    n = tiles.shape[0]
    x = tiles.contiguous().view(n, C // 16, TILE, 16).permute(0, 2, 1, 3).reshape(n * TILE, C)
    return x.view(dtype)


def encode_fp8(x):
    C = x.shape[1]
    n = x.shape[0] // TILE
    return x.view(torch.uint8).view(n, TILE, C // 16, 16).permute(0, 2, 1, 3).contiguous().view(n, C * TILE)


def _mask_shifts(device):
    q = torch.arange(8, device=device)[:, None]
    t = torch.arange(4, device=device)[None, :]
    return (8 * t + q).to(torch.int32)               # [q][t]: bit 8 t + q holds column 4 q + t of the group


def decode_mask(tiles):
    """[n, 4096] uint8 ReLU' bits of one layer -> bool [n * 128, 256].  Word (h, r, g) at h * 2048 + r * 16 + g * 4;
    its bit 8 t + q is column h * 128 + g * 32 + 4 q + t."""
    n = tiles.shape[0]
    w = tiles.contiguous().view(torch.int32).view(n, 2, TILE, 4)                      # (h, r, g)
    bits = (w[..., None, None] >> _mask_shifts(w.device)) & 1                       # (h, r, g, q, t)
    return bits.permute(0, 2, 1, 3, 4, 5).reshape(n * TILE, 256).bool()


def encode_mask(m):
    """inverse of decode_mask: bool [n * 128, 256] -> [n, 4096] uint8"""
    n = m.shape[0] // TILE
    b = m.view(n, TILE, 2, 4, 8, 4).permute(0, 2, 1, 3, 4, 5).to(torch.int64)        # (h, r, g, q, t)
    w = (b << _mask_shifts(m.device).to(torch.int64)).sum(dim=(-1, -2))             # (h, r, g), < 2^32
    w = torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)
    return w.contiguous().view(torch.uint8).view(n, MASK_LAYER)


# ---- rounding --------------------------------------------------------------------------------------------------
def bf16(x):
    """round to bf16 (nearest even), returned in x's dtype"""
    return x.to(torch.bfloat16).to(x.dtype)


def e4m3(x):
    """cvt.rn.satfinite.e4m3: torch's cast rounds to nearest even but does not saturate (500 -> NaN), so clamp first"""
    return x.float().clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn)


def e5m2(x):
    """cvt.rn.satfinite.e5m2 (torch's cast gives inf from 61440 up)"""
    return x.float().clamp(-E5M2_MAX, E5M2_MAX).to(torch.float8_e5m2)


def ulp_bf16(x):
    """spacing of bf16 numbers at |x| (x float64; the smallest normal's spacing below it)"""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.exp2(e - 7)


def ulp_fp8(x, mant, emin):
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** emin)))
    return torch.exp2(e - mant)


def dz8_scale(amax_bits, inverse=False):
    """tc_layout.cuh dz8_scale: 2^(kDz8Top - e) for max|d_pre| = m 2^e, m in [0.5, 1); e clamped to [-100, 100]"""
    e = ((amax_bits >> 23) & 0xFF) - 126
    if amax_bits == 0 or e < -100:
        e = -100
    e = min(e, 100)
    return 2.0 ** (e - DZ8_TOP if inverse else DZ8_TOP - e)


# ---- the model embedded in the chain (api.cu build_model / tc_chain_map) ------------------------------------------
class Chain:
    """Chain layer c of the fixed eight-layer program runs model layer cmap[c] (-1: an identity layer).  Offsets are
    those of the flat Keras-order parameter buffer."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.U, self.dx, self.dd, n = cfg.dense_units, cfg.dx, cfg.dd, cfg.n_layers
        self.shapes = O.layer_shapes(cfg)
        self.w_off, self.b_off, off = [], [], 0
        for _, fi, fo in self.shapes:
            self.w_off.append(off)
            self.b_off.append(off + fi * fo)
            off += fi * fo + fo
        self.n_params = off
        # layer i + 1 takes the [h, x] concat when i % skip == 0, i > 0 (mlp.py:36-38)
        takes = [i for i in range(1, n) if (i - 1) % cfg.skip_layer == 0 and i > 1]
        assert len(takes) <= 1 and not ((n - 1) % cfg.skip_layer == 0 and n > 1), "not a chain model"
        self.cmap = [c if c < n else -1 for c in range(8)]
        if takes:
            s = takes[0]
            assert s <= 5 and n - 1 - s <= 2, "not a chain model"
            self.cmap = [c if c < s else -1 for c in range(8)]
            for i in range(s, n):
                self.cmap[5 + i - s] = i
        self.x5 = self.cmap[5] >= 0 and self.shapes[self.cmap[5]][1] > self.U
        self.heads = {name: n + i for i, name in enumerate(("sigma", "features", "rgb_features", "rgb"))}

    def kernel(self, params, L):
        _, fi, fo = self.shapes[L]
        return params[self.w_off[L]:self.w_off[L] + fi * fo].view(fi, fo)

    def bias(self, params, L):
        fo = self.shapes[L][2]
        return params[self.b_off[L]:self.b_off[L] + fo]

    def fwd_weight(self, params, c):
        """B operand of forward step c < 8 as a float64 [K, 256] matrix over the step's A operand: h_{c-1} (256 columns,
        c > 0), then PE(xyz) (64 columns, c = 0 and c = 5) -- mlp_tc.cu fwd_weight -- and the bias [256]"""
        U, dev = self.U, params.device
        kh = 0 if c == 0 else 256
        kx = 64 if c in (0, 5) else 0
        W = torch.zeros(kh + kx, 256, dtype=torch.float64, device=dev)
        b = torch.zeros(256, dtype=torch.float64, device=dev)
        L = self.cmap[c]
        if L < 0:
            W[:kh, :kh] = torch.eye(kh, dtype=torch.float64, device=dev)
            return W, b
        K = self.kernel(params, L).double()
        if c == 0:
            W[:self.dx, :U] = K
        else:
            W[:U, :U] = K[:U]
            if c == 5 and self.x5:
                W[256:256 + self.dx, :U] = K[U:]
        b[:U] = self.bias(params, L).double()
        return W, b

    def bwd_weight(self, params, c):
        """dgrad B operand into h_{c-1} for chain layer c >= 1: W_c[:U, :U] (or I) padded to [256, 256]"""
        dev = params.device
        L = self.cmap[c]
        if L < 0:
            return torch.eye(256, dtype=torch.float64, device=dev)
        W = torch.zeros(256, 256, dtype=torch.float64, device=dev)
        W[:self.U, :self.U] = self.kernel(params, L)[:self.U].double()
        return W


def fold_reference(ch, params):
    """float64 W' = W_f W_g[:U] [256, 128] + b' = b_f W_g[:U] + b_g, and the folded heads [289, 4] (mlp_tc.cu
    fold_kernel), each with the same products over |.| (for an fp32 summation bound)"""
    U, H, dd = ch.U, ch.U // 2, ch.dd
    p = params.double()
    hd = ch.heads
    Wf, bf = ch.kernel(p, hd["features"]), ch.bias(p, hd["features"])
    Wg, bg = ch.kernel(p, hd["rgb_features"]), ch.bias(p, hd["rgb_features"])
    Wc, bc = ch.kernel(p, hd["rgb"]), ch.bias(p, hd["rgb"])
    ws, bs = ch.kernel(p, hd["sigma"]), ch.bias(p, hd["sigma"])
    out = []
    for a in (False, True):
        f = (lambda x: x.abs()) if a else (lambda x: x)
        fold = torch.zeros(257, 128, dtype=torch.float64, device=params.device)
        fold[:U, :H] = f(Wf) @ f(Wg[:U])
        fold[256, :H] = f(bf) @ f(Wg[:U]) + f(bg)
        head = torch.zeros(HEAD_ROWS, 4, dtype=torch.float64, device=params.device)
        head[:U, :3] = fold[:U, :H] @ f(Wc)
        head[:U, 3] = f(ws[:, 0])
        head[256:256 + dd, :3] = f(Wg[U:]) @ f(Wc)
        head[288, :3] = fold[256, :H] @ f(Wc) + f(bc)
        head[288, 3] = f(bs[0])
        out += [fold, head]
    return out   # fold, head, |fold|, |head|


def fold_split(head):
    """the last forward step's weights: bf16(v) + bf16(v - bf16(v)) of the packed fp32 heads (mlp_tc.cu fold_split)"""
    hi = bf16(head)
    return hi.double() + bf16(head - hi).double()


# ---- forward references ----------------------------------------------------------------------------------------
def sample_points(o, d, t, n):
    """fp32 p = o + d t per sample, rounded product then sum (mlp_tc.cu load_sample); rows past R * S are 0, as are
    their directions"""
    R, S = t.shape
    p = (o[:, None, :] + d[:, None, :] * t[..., None]).reshape(R * S, 3)
    dirs = d[:, None, :].expand(R, S, 3).reshape(R * S, 3)
    pad = n * TILE - R * S
    z = torch.zeros(pad, 3, dtype=p.dtype, device=p.device)
    return torch.cat([p, z]), torch.cat([dirs, z])


def pe_reference(x, L, width, one_col):
    """float64 [x, sin(2^0 x), cos(2^0 x), ...] (utils.py:176-186) in `width` columns: zeros after the encoding, 1 at
    column one_col (the constant-1 column that carries the folded bias)"""
    x = x.double()
    parts = [x]
    for f in range(L):
        parts += [torch.sin(2.0 ** f * x), torch.cos(2.0 ** f * x)]
    e = torch.cat(parts, dim=1)
    out = torch.zeros(x.shape[0], width, dtype=torch.float64, device=x.device)
    out[:, :e.shape[1]] = e
    out[:, one_col] = 1.0
    return out


def step_check(rec, exact, absum):
    """An fp32-accumulated, bf16-rounded step: |rec - exact| <= 1 bf16 ulp + 2^-16 sum|terms| (K <= 320 fp32 additions
    of a sum whose terms cancel).  Returns (worst ratio to that bound, fraction of elements that differ from the bf16
    rounding of the exact value)."""
    rec = rec.double()
    err = (rec - exact).abs()
    bound = ulp_bf16(torch.maximum(exact.abs(), rec.abs())) + 2.0 ** -16 * absum
    inexact = (rec != bf16(exact.float()).double()).double().mean()
    return float((err / bound).max()), float(inexact)


# ---- weight-gradient check -------------------------------------------------------------------------------------
def grad_error(g, ref):
    """max |g - ref| / max |ref| of one tensor"""
    return float((g.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


# ---- mlp_tc_bwd.cu build_task_table / build_items, restated: where the weight-gradient work items start --------------
# These values must follow the source; test_tc_records_cpu.py::test_item_rule_follows_the_source reads them back from it.
NUM_SMS = 148                        # kNumSMs (common.cuh)
HEADS_COST, XPART_COST8, HEADS_COST8 = 178, 80, 94   # kHeadsCost, kXpartCost8, kHeadsCost8
BIG_COST, XPART_COST = 128, 76       # t.cost of build_task_table's `big` and `xpart` tasks
GUIDE, MIN_SHARE, MIN_TILES = 2, 16, 4   # kWGuide, kWMinShare, kWMinTiles
# per task: layer 0 (x part), layers 1..7 (h part), layer 5 (x part), heads
TASK_COSTS = {False: [XPART_COST] + [BIG_COST] * 7 + [XPART_COST, HEADS_COST],
              True: [XPART_COST8] + [BIG_COST] * 7 + [XPART_COST8, HEADS_COST8]}


def hidden_task(c, encoding_rows=False):
    """the weight-gradient task that computes chain layer c's kernel rows (and, for its hidden rows, its bias)"""
    return 8 if (c == 5 and encoding_rows) else c


def work_items(n, rec8):
    """(cost, task, lo, hi) of every item in list order"""
    costs = TASK_COSTS[rec8]
    total = sum(c * n for c in costs)
    min_cost = max(total / NUM_SMS / MIN_SHARE, 128.0 * MIN_TILES)
    items, left = [], total
    for k, c in enumerate(costs):
        lo = 0
        while lo < n:
            want = max(min_cost, left / (GUIDE * NUM_SMS))
            m = max(1, int(want / c + 0.5))
            if n - lo - m < (m + 1) // 2:
                m = n - lo
            items.append((c * m, k, lo, lo + m))
            left -= c * m
            lo += m
    return sorted(items, key=lambda it: -it[0])   # (stable)
