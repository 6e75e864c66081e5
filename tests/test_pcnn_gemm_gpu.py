"""GPU: the PixelCNN prior's tcgen05 GEMM (``dvq_pcnn_gemm``, csrc/pcnn_sm100.cu) against an exact float64 reference at
the grasp benchmark's shapes (GatedPixelCNN(512, 512, 15) sampled at batch 4096), plus its argument checks and the two
packing kernels ``dvq_pcnn_embed`` / ``dvq_pcnn_rows_to_image``.

The operands are small multiples of powers of two: A = k/8 and W = k/16 with |k| <= 4, bias and residual k/128 with
|k| <= 64, cond k/64 with |k| <= 8.  Every product is then a multiple of 2^-7 of magnitude <= 1/8, so even 12 segments
x 1024 columns keep every partial sum under 2^11 with 7 fractional bits: FP32 accumulation in any order is exact, and so
is the float64 reference.  FP32 outputs (logits, the residual image) must equal it bit for bit, FP16 outputs (RES / RELU
images, GATE's pre-activations) its round-to-nearest-even (``cvt.rn.f16x2.f32`` on an exact FP32 value).  Only GATE's
gated output goes through ``tanh.approx.f32`` and has an error bar."""
import ctypes as C

import pytest
import torch

from dvq import _cabi
from dvq.pixelcnn_tc import PC_GATE, PC_LOGITS, PC_RELU, PC_RES, _Gemm, _w_image, gate_perm

pytestmark = pytest.mark.gpu

BAD_SHAPE, BAD_ALIGN, BAD_ARG = -1, -2, -7
PAD = 37                 # padding rows per batch: B = Bp - PAD
GATE_BAR = 2.0 ** -9     # tanh.approx.f32: ~2^-11 per factor, plus the FP16 rounding of the output


def to_image16(m):
    """[rows, K] -> FP16 operand image [rows/128][K/8][128][8]."""
    rows, k = m.shape
    return m.reshape(rows // 128, 128, k // 8, 8).permute(0, 2, 1, 3).contiguous().to(torch.float16)


def from_image16(img, k):
    return img.reshape(-1, k // 8, 128, 8).permute(0, 2, 1, 3).reshape(-1, k)


def to_image32(m):
    """[rows, K] -> FP32 residual image [rows/128][K/4][128][4]."""
    rows, k = m.shape
    return m.reshape(rows // 128, 128, k // 4, 4).permute(0, 2, 1, 3).contiguous().to(torch.float32)


def from_image32(img, k):
    return img.reshape(-1, k // 4, 128, 4).permute(0, 2, 1, 3).reshape(-1, k)


def _q(gen, shape, n, den, dev):
    """Integers in [-n, n] over den: exact in FP16 and in every sum the tests form."""
    return torch.randint(-n, n + 1, shape, generator=gen, device=dev).float() / den


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.float16 else torch.int32)


# ---- the cases --------------------------------------------------------------------------------------------------
# A case: epilogue mode, T = 128-row tiles per grid column (Bp = 128 T), output grid columns `cols` (m_tiles = cols T),
# ncols_src, n_tiles, activation images {name: (grid columns, K width)} and segments (image, ks, col_shift, tile_shift).

def _case(mode, T, cols, ncols_src, n_tiles, images, segs, res_in=0, pre=False, cond=False):
    return dict(mode=mode, T=T, cols=cols, ncols_src=ncols_src, n_tiles=n_tiles, images=images, segs=segs, res_in=res_in,
                pre=pre, cond=cond)


def _vertical(T, rows, taps):
    """The vertical stack of a grid row: one segment per (kernel row image, column tap), shifted by whole columns."""
    return [(r, 512, cs, cs * T) for r in rows for cs in taps]


def _horizontal(n, T=32):
    return _case(PC_GATE, T, n, n, 4, {"pre": (3, 1024), "xh": (3, 512)},
                 [("pre", 1024, 0, 0), ("xh", 512, -1, -T), ("xh", 512, 0, 0)], cond=True)


def _skipped(mode, T=64, n_tiles=2, ks=256):
    # grid column 2 has no valid segment (2 + 1 and 2 + 2 are outside the 3 source columns): its tiles must be exactly bias
    # (+ residual), whatever the CTA's accumulator stage held; at T = 64, 384 tiles, so most CTAs reach column 2 as their
    # third tile
    return _case(mode, T, 3, 3, n_tiles, {"a": (3, ks)}, [("a", ks, 1, T), ("a", ks, 2, 2 * T)], res_in=int(mode == PC_RES))


_MAXSEG_T = 40
CASES = {
    # output head at column j = 2 of the grid: ReLU 512 -> 2048 (8 n-tiles), logits 2048 -> 512 (K ring wraps 8x per tile)
    "head_relu_T32": _case(PC_RELU, 32, 1, 1, 8, {"xh": (3, 512)}, [("xh", 512, 0, 64)]),
    "head_relu_T64": _case(PC_RELU, 64, 1, 1, 8, {"xh": (3, 512)}, [("xh", 512, 0, 128)]),
    "head_logits_T32": _case(PC_LOGITS, 32, 1, 1, 2, {"hid": (1, 2048)}, [("hid", 2048, 0, 0)]),
    "head_logits_T64": _case(PC_LOGITS, 64, 1, 1, 2, {"hid": (1, 2048)}, [("hid", 2048, 0, 0)]),
    # vertical stack, d = 512: layer > 0 (kernel rows r-1, r; taps -1, 0, +1) and layer 0 (rows r-2, r-1; taps -2..+2)
    "vertical_layer1": _case(PC_GATE, 48, 3, 3, 4, {"r0": (3, 512), "r1": (3, 512)}, _vertical(48, ("r0", "r1"), (-1, 0, 1)),
                             pre=True, cond=True),
    "vertical_layer0": _case(PC_GATE, 32, 3, 3, 4, {"r0": (3, 512), "r1": (3, 512)}, _vertical(32, ("r0", "r1"), (-2, -1, 0, 1, 2)),
                             pre=True, cond=True),
    # horizontal stack at n = 1, 2, 3 columns: v2h (K = 1024) + taps -1, 0
    "horizontal_n1": _horizontal(1),
    "horizontal_n2": _horizontal(2),
    "horizontal_n3": _horizontal(3),
    # 1x1 residual convolution, 512 -> 512: 576 tiles
    "residual_in0": _case(PC_RES, 96, 3, 3, 2, {"out": (3, 512)}, [("out", 512, 0, 0)], res_in=0),
    "residual_in1": _case(PC_RES, 96, 3, 3, 2, {"out": (3, 512)}, [("out", 512, 0, 0)], res_in=1),
    # 12 segments: every ks, partial-width reads (a_kd > ks), images read several times, per-column K lengths differ
    "max_segments": _case(PC_LOGITS, _MAXSEG_T, 3, 3, 2,
                          {"i1024": (3, 1024), "i512": (3, 512), "i256": (3, 256), "i192": (3, 192), "i64": (3, 64)},
                          [(name, ks, cs, cs * _MAXSEG_T) for name, ks, cs in (
                              ("i1024", 1024, 0), ("i1024", 64, 1), ("i512", 512, -1), ("i512", 192, 0), ("i256", 256, 1),
                              ("i256", 128, 0), ("i192", 192, -1), ("i64", 64, 0), ("i1024", 512, -1), ("i512", 128, 1),
                              ("i256", 64, -1), ("i192", 128, 0))]),
    "skipped_taps_logits": _skipped(PC_LOGITS),
    "skipped_taps_res": _skipped(PC_RES),
    # 5100 tiles: a CTA of a 148-SM B200 handles 34 or 35, so its tiles past the 32nd reach column 2 as well
    "skipped_taps_long": _skipped(PC_LOGITS, T=1700, n_tiles=1, ks=64),
}
# tile counts around grid = min(tiles, SMs): resolved against the device's SM count at run time
TILE_COUNTS = {"tiles_1": (0, 1), "tiles_sm-1": (1, -1), "tiles_sm": (1, 0), "tiles_sm+1": (1, 1), "tiles_2sm+1": (2, 1),
               "tiles_3sm+1": (3, 1)}


def _tile_count_case(name):
    sms = _cabi.device_info()[0]
    k, r = TILE_COUNTS[name]
    tiles = k * sms + r
    n_tiles = next(n for n in (3, 2, 1) if tiles % n == 0)
    m_tiles = tiles // n_tiles
    return _case(PC_LOGITS, m_tiles, 1, 1, n_tiles, {"a": (1, 256)}, [("a", 256, 0, 0)])


def _get_case(name):
    return _tile_count_case(name) if name in TILE_COUNTS else CASES[name]


def _names(mode):
    return [n for n, c in CASES.items() if c["mode"] == mode] + (list(TILE_COUNTS) if mode == PC_LOGITS else [])


# ---- one launch configuration: inputs, launches, float64 reference ---------------------------------------------

class GemmCase:
    def __init__(self, c, dev="cuda", seed=0):
        self.c, self.dev = c, torch.device(dev)
        T, cols = c["T"], c["cols"]
        self.Bp, self.B = 128 * T, 128 * T - PAD
        self.M, self.N = cols * T * 128, c["n_tiles"] * 256
        self.gate = c["mode"] == PC_GATE
        self.d_gate = self.N // 2 if self.gate else 0
        self.out_kd = self.d_gate if self.gate else self.N
        for name, ks, cs, ts in c["segs"]:     # the kernel reads rows (mt + tile_shift) of every tile with a valid segment
            ncol_img, kd = c["images"][name]
            assert ks <= kd
            for col in range(cols):
                if 0 <= col + cs < c["ncols_src"]:
                    assert 0 <= col * T + ts and (col + 1) * T + ts <= ncol_img * T, (name, col)
        self.gen = torch.Generator(device=self.dev).manual_seed(seed)
        q = lambda shape, n, den: _q(self.gen, shape, n, den, self.dev)
        self.A = {name: q((ncol * T * 128, kd), 4, 8) for name, (ncol, kd) in c["images"].items()}
        self.W = [q((ks, self.N), 4, 16) for (_, ks, _, _) in c["segs"]]
        self.bias = q((self.N,), 64, 128)
        self.cond = q((self.Bp, self.N), 8, 64) if c["cond"] else None
        self.res = q((self.M, self.N), 64, 128) if c["mode"] == PC_RES else None
        perm = gate_perm(self.d_gate, self.dev) if self.gate else None
        self.w_img = [_w_image(w, perm) for w in self.W]
        self.bias_tiles = self.bias[perm].contiguous() if self.gate else self.bias
        self.err = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self._upload()
        h16 = lambda n: torch.empty(n, dtype=torch.float16, device=self.dev)
        self.out = h16(self.M * self.out_kd) if c["mode"] != PC_LOGITS else None
        self.pre = h16(self.M * 2 * self.d_gate) if c["pre"] else None
        self.res_img = torch.empty(self.M * self.N, dtype=torch.float32, device=self.dev) if self.res is not None else None
        self.logits = torch.empty((self.M, self.N), dtype=torch.float32, device=self.dev) if c["mode"] == PC_LOGITS else None

    def _upload(self):
        self.a16 = {name: to_image16(a) for name, a in self.A.items()}
        self.cond16 = to_image16(self.cond) if self.cond is not None else None
        self.res32 = to_image32(self.res) if self.res is not None else None

    def perturb_padding(self):
        """New values in every input row of a padding batch slot (b >= B); valid rows must not notice."""
        q = lambda shape, n, den: _q(self.gen, shape, n, den, self.dev)
        for t, n, den in [(a, 4, 8) for a in self.A.values()] + [(t, n, d) for t, n, d in ((self.cond, 8, 64), (self.res, 64, 128)) if t is not None]:
            pad = torch.arange(t.shape[0], device=self.dev) % self.Bp >= self.B
            t[pad] = q((int(pad.sum()), t.shape[1]), n, den)
        self._upload()

    def valid_rows(self):
        return torch.arange(self.M, device=self.dev) % self.Bp < self.B

    def descriptor(self):
        c, g = self.c, _Gemm()
        for i, (name, ks, cs, ts) in enumerate(c["segs"]):
            g.seg[i].a_img, g.seg[i].w_img = self.a16[name].data_ptr(), self.w_img[i].data_ptr()
            g.seg[i].a_kd, g.seg[i].ks, g.seg[i].tile_shift, g.seg[i].col_shift = c["images"][name][1], ks, ts, cs
        g.nseg, g.m_tiles, g.n_tiles, g.tiles_per_col = len(c["segs"]), c["cols"] * c["T"], c["n_tiles"], c["T"]
        g.ncols_src, g.mode = c["ncols_src"], c["mode"]
        ptr = lambda t: t.data_ptr() if t is not None else None
        g.bias, g.cond_img, g.out_img, g.pre_img = ptr(self.bias_tiles), ptr(self.cond16), ptr(self.out), ptr(self.pre)
        g.res_img, g.logits, g.out_kd, g.res_in, g.d_gate, g.err = ptr(self.res_img), ptr(self.logits), self.out_kd, c["res_in"], self.d_gate, ptr(self.err)
        return g

    def launch(self):
        """One launch on freshly poisoned outputs (NaN: anything the kernel does not write shows); decoded [rows, K] results."""
        for t in (self.out, self.pre, self.res_img, self.logits):
            if t is not None:
                t.fill_(float("nan"))
        if self.res_img is not None and self.c["res_in"]:
            self.res_img.copy_(self.res32.view(-1))
        g = self.descriptor()
        n0 = _cabi.launch_count()
        with torch.cuda.device(self.dev):
            _cabi.check(_cabi.lib.dvq_pcnn_gemm(C.byref(g), torch.cuda.current_stream(self.dev).cuda_stream), "dvq_pcnn_gemm")
        assert _cabi.launch_count() == n0 + 1
        torch.cuda.synchronize(self.dev)
        assert int(self.err.item()) == 0, "pipeline time-out %d" % int(self.err.item())
        got = {}
        if self.logits is not None:
            got["logits"] = self.logits.clone()
        if self.out is not None:
            got["out"] = from_image16(self.out, self.out_kd).clone()
        if self.pre is not None:
            got["pre"] = from_image16(self.pre, 2 * self.d_gate).clone()
        if self.res_img is not None:
            got["res"] = from_image32(self.res_img, self.N).clone()
        return got

    def reference(self):
        """float64: C = sum over the segments valid for a row's grid column of A[row + 128 tile_shift, :ks] @ W, then the
        epilogue.  Exact, so the FP32 / FP16 outputs are its roundings."""
        c, T = self.c, self.c["T"]
        rows = torch.arange(self.M, device=self.dev)
        col = rows // (128 * T)
        acc = torch.zeros((self.M, self.N), dtype=torch.float64, device=self.dev)
        for (name, ks, cs, ts), w in zip(c["segs"], self.W):
            r = rows[(col + cs >= 0) & (col + cs < c["ncols_src"])]
            acc.index_add_(0, r, self.A[name][r + 128 * ts, :ks].double() @ w.double())
        x = acc + self.bias.double()
        if c["mode"] == PC_LOGITS:
            return {"logits": x.float()}
        if c["mode"] == PC_RELU:
            return {"out": x.clamp_min(0).float().half()}
        if c["mode"] == PC_RES:
            if c["res_in"]:
                x = x + self.res.double()
            return {"res": x.float(), "out": x.float().half()}
        d = self.d_gate
        cond = self.cond.double()[rows % self.Bp] if self.cond is not None else torch.zeros_like(x)
        ref = {"gate": torch.tanh(x[:, :d] + cond[:, :d]) * torch.sigmoid(x[:, d:] + cond[:, d:])}
        if c["pre"]:
            ref["pre"] = x.float().half()
        return ref


def _assert_bits(got, ref, what, case):
    same = _bits(got) == _bits(ref)
    if bool(same.all()):
        return
    bad_rows = (~same).any(1).nonzero().squeeze(1)
    cols = sorted(set((bad_rows // case.Bp).tolist()))
    diff = (got.double() - ref.double()).abs()
    raise AssertionError("%s: %d of %d elements differ, in rows of grid columns %s (first row %d); max |diff| %s" % (
        what, int((~same).sum()), same.numel(), cols, int(bad_rows[0]), float(diff.nan_to_num(float("inf")).max())))


def _run_case(name, dev="cuda"):
    """Reference check, repeat determinism and padding-row independence of one case; returns the case and first outputs."""
    case = GemmCase(_get_case(name), dev)
    got = case.launch()
    ref = case.reference()
    for k, r in ref.items():
        if k == "gate":
            err = float((got["out"].double() - r).abs().max())
            print("%s: gated output, worst |out - float64| = %.3e (bar 2^-9 = %.3e)" % (name, err, GATE_BAR))
            assert err <= GATE_BAR, (name, err)
        else:
            _assert_bits(got[k], r, "%s %s" % (name, k), case)
    again = case.launch()
    for k in got:
        _assert_bits(again[k], got[k], "%s %s (repeat launch)" % (name, k), case)
    case.perturb_padding()
    moved = case.launch()
    valid = case.valid_rows()
    for k in got:
        _assert_bits(moved[k][valid], got[k][valid], "%s %s (padding rows changed)" % (name, k), case)
    return case, got


@pytest.mark.parametrize("name", _names(PC_GATE))
def test_gate_epilogue(name):
    _run_case(name)


@pytest.mark.parametrize("name", _names(PC_RES))
def test_res_epilogue(name):
    _run_case(name)


@pytest.mark.parametrize("name", _names(PC_RELU))
def test_relu_epilogue(name):
    _run_case(name)


@pytest.mark.parametrize("name", _names(PC_LOGITS))
def test_logits_epilogue(name):
    _run_case(name)


def test_second_device_in_the_same_process():
    """The dynamic shared-memory opt-in is per device: the first launch on cuda:1 after cuda:0 must succeed."""
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    outs = [_run_case("tiles_sm+1", dev)[1]["logits"].cpu() for dev in ("cuda:0", "cuda:1")]
    assert torch.equal(_bits(outs[0]), _bits(outs[1]))


# ---- argument validation: rejected on the host, nothing launched -------------------------------------------------

def _seg0(field, value):
    return lambda g: setattr(g.seg[0], field, value)


def _set(**kw):
    def f(g):
        for k, v in kw.items():
            setattr(g, k, v)
    return f


GEMM_BAD = {
    "nseg_0": (_set(nseg=0), BAD_SHAPE, "K-segments"),
    "nseg_13": (_set(nseg=13), BAD_SHAPE, "K-segments"),
    "ks_0": (_seg0("ks", 0), BAD_SHAPE, "segment 0"),
    "ks_not_multiple_of_64": (_seg0("ks", 96), BAD_SHAPE, "segment 0"),
    "a_kd_below_ks": (_seg0("a_kd", 192), BAD_SHAPE, "segment 0"),
    "a_kd_not_multiple_of_8": (lambda g: (_seg0("a_kd", 260)(g), _seg0("ks", 192)(g)), BAD_SHAPE, "segment 0"),
    "a_img_misaligned": (lambda g: setattr(g.seg[0], "a_img", g.seg[0].a_img + 8), BAD_ALIGN, "16-byte"),
    "w_img_misaligned": (lambda g: setattr(g.seg[0], "w_img", g.seg[0].w_img + 8), BAD_ALIGN, "16-byte"),
    "bias_null": (_set(bias=None), BAD_ARG, "bias is NULL"),
    "logits_null": (_set(logits=None), BAD_ARG, "output buffer is NULL"),
    "gate_out_null": (_set(mode=PC_GATE, out_img=None), BAD_ARG, "output buffer is NULL"),
    "res_out_null": (_set(mode=PC_RES, out_img=None), BAD_ARG, "output buffer is NULL"),
    "relu_out_null": (_set(mode=PC_RELU, out_img=None), BAD_ARG, "output buffer is NULL"),
    "res_without_res_img": (_set(mode=PC_RES, res_img=None), BAD_ARG, "residual image"),
    "mode_4": (_set(mode=4), BAD_ARG, "epilogue mode"),
    "mode_negative": (_set(mode=-1), BAD_ARG, "epilogue mode"),
    "m_tiles_0": (_set(m_tiles=0), BAD_SHAPE, "empty tile grid"),
    "n_tiles_0": (_set(n_tiles=0), BAD_SHAPE, "empty tile grid"),
    "tiles_per_col_0": (_set(tiles_per_col=0), BAD_SHAPE, "empty tile grid"),
}


def _expect_rejected(call, code, words):
    _cabi.lib.dvq_vq_set_refine(-1, 0)            # leaves an unrelated message: the one read below must be fresh
    n0 = _cabi.launch_count()
    assert call() == code
    assert words in _cabi.last_error(), _cabi.last_error()
    assert _cabi.launch_count() == n0


@pytest.mark.parametrize("name", list(GEMM_BAD))
def test_gemm_rejects_bad_arguments(name):
    mutate, code, words = GEMM_BAD[name]
    case = GemmCase(_case(PC_LOGITS, 1, 1, 1, 1, {"a": (1, 256)}, [("a", 256, 0, 0)]))
    case.out = torch.zeros(128 * 256, dtype=torch.float16, device="cuda")        # an output image for the other modes
    case.res_img = torch.zeros(128 * 256, dtype=torch.float32, device="cuda")
    g = case.descriptor()
    mutate(g)
    _expect_rejected(lambda: _cabi.lib.dvq_pcnn_gemm(C.byref(g), torch.cuda.current_stream().cuda_stream), code, words)
    torch.cuda.synchronize()
    assert int(case.err.item()) == 0


# ---- dvq_pcnn_embed / dvq_pcnn_rows_to_image ---------------------------------------------------------------------

def _embed_args(**kw):
    a = dict(W=3, x_stride=5, B=200, Bp=256, n_emb=512, d=512)
    a.update(kw)
    return a


def _embed_call(a, x, emb, img16, img32):
    ptr = lambda t: t.data_ptr() if t is not None else None
    return _cabi.lib.dvq_pcnn_embed(ptr(x), a["x_stride"], a["W"], a["B"], a["Bp"], ptr(emb), a["n_emb"], a["d"], ptr(img16), ptr(img32),
                                    torch.cuda.current_stream().cuda_stream)


def _rows_call(a, label, table, img16):
    ptr = lambda t: t.data_ptr() if t is not None else None
    return _cabi.lib.dvq_pcnn_rows_to_image(ptr(label), a["B"], a["Bp"], ptr(table), a["n_rows"], a["kd"], ptr(img16),
                                            torch.cuda.current_stream().cuda_stream)


def test_embed_matches_torch_packing():
    """Rows m = c Bp + b of emb[clamp(x[b, c])] (indices clamped to [0, n_emb)), zero for b >= B, as the FP16 operand
    image and the FP32 residual image; x read with a row stride wider than the grid."""
    a = _embed_args()
    W, S, B, Bp, n_emb, d = a["W"], a["x_stride"], a["B"], a["Bp"], a["n_emb"], a["d"]
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randint(-3, n_emb + 3, (B, S), generator=gen, device="cuda")
    x[:4, :W] = torch.tensor([[-1, 0, n_emb - 1], [n_emb, n_emb + 7, -100], [5, 6, 7], [1, 2, 3]], device="cuda")
    emb = torch.randn((n_emb, d), generator=gen, device="cuda")
    rows = torch.zeros((W, Bp, d), device="cuda")
    rows[:, :B] = emb[x[:, :W].clamp(0, n_emb - 1)].permute(1, 0, 2)
    rows = rows.reshape(W * Bp, d)
    for with32 in (True, False):
        img16 = torch.full((W * Bp * d,), float("nan"), dtype=torch.float16, device="cuda")
        img32 = torch.full((W * Bp * d,), float("nan"), device="cuda") if with32 else None
        _cabi.check(_embed_call(a, x, emb, img16, img32), "dvq_pcnn_embed")
        torch.cuda.synchronize()
        assert torch.equal(_bits(img16), _bits(to_image16(rows).view(-1)))
        if with32:
            assert torch.equal(_bits(img32), _bits(to_image32(rows).view(-1)))


def test_rows_to_image_matches_torch_packing():
    """table[clamp(label[b])] as an FP16 operand image [Bp, kd], zero rows for b >= B."""
    B, Bp, n_rows, kd = 200, 256, 128, 1024
    gen = torch.Generator(device="cuda").manual_seed(4)
    label = torch.randint(-2, n_rows + 2, (B,), generator=gen, device="cuda")
    label[:3] = torch.tensor([-5, n_rows, n_rows + 100], device="cuda")
    table = torch.randn((n_rows, kd), generator=gen, device="cuda")
    rows = torch.zeros((Bp, kd), device="cuda")
    rows[:B] = table[label.clamp(0, n_rows - 1)]
    img16 = torch.full((Bp * kd,), float("nan"), dtype=torch.float16, device="cuda")
    _cabi.check(_rows_call(dict(B=B, Bp=Bp, n_rows=n_rows, kd=kd), label, table, img16), "dvq_pcnn_rows_to_image")
    torch.cuda.synchronize()
    assert torch.equal(_bits(img16), _bits(to_image16(rows).view(-1)))


EMBED_BAD = {
    "B_0": (dict(B=0), BAD_SHAPE), "Bp_below_B": (dict(Bp=128), BAD_SHAPE), "Bp_not_multiple_of_128": (dict(Bp=320), BAD_SHAPE),
    "d_0": (dict(d=0), BAD_SHAPE), "d_not_multiple_of_8": (dict(d=508), BAD_SHAPE), "W_0": (dict(W=0), BAD_SHAPE),
    "n_emb_0": (dict(n_emb=0), BAD_SHAPE), "x_null": ("x", BAD_ARG), "emb_null": ("emb", BAD_ARG), "img16_null": ("img16", BAD_ARG),
}
ROWS_BAD = {
    "B_0": (dict(B=0), BAD_SHAPE), "Bp_below_B": (dict(Bp=128), BAD_SHAPE), "Bp_not_multiple_of_128": (dict(Bp=320), BAD_SHAPE),
    "kd_0": (dict(kd=0), BAD_SHAPE), "kd_not_multiple_of_8": (dict(kd=1020), BAD_SHAPE), "n_rows_0": (dict(n_rows=0), BAD_SHAPE),
    "label_null": ("label", BAD_ARG), "table_null": ("table", BAD_ARG), "img16_null": ("img16", BAD_ARG),
}


@pytest.mark.parametrize("name", list(EMBED_BAD))
def test_embed_rejects_bad_arguments(name):
    change, code = EMBED_BAD[name]
    t = dict(x=torch.zeros((200, 5), dtype=torch.int64, device="cuda"), emb=torch.zeros((512, 512), device="cuda"),
             img16=torch.zeros(3 * 256 * 512, dtype=torch.float16, device="cuda"))
    a = _embed_args(**change) if isinstance(change, dict) else _embed_args()
    if isinstance(change, str):
        t[change] = None
    _expect_rejected(lambda: _embed_call(a, t["x"], t["emb"], t["img16"], None), code, "NULL" if code == BAD_ARG else "Bp")


@pytest.mark.parametrize("name", list(ROWS_BAD))
def test_rows_to_image_rejects_bad_arguments(name):
    change, code = ROWS_BAD[name]
    t = dict(label=torch.zeros(200, dtype=torch.int64, device="cuda"), table=torch.zeros((128, 1024), device="cuda"),
             img16=torch.zeros(256 * 1024, dtype=torch.float16, device="cuda"))
    a = dict(B=200, Bp=256, n_rows=128, kd=1024)
    if isinstance(change, dict):
        a.update(change)
    else:
        t[change] = None
    _expect_rejected(lambda: _rows_call(a, t["label"], t["table"], t["img16"]), code, "NULL" if code == BAD_ARG else "Bp")
