"""The tensor-core entry points at every shape and schedule they accept, against plain high-precision references.

- Convolutions (fprop, dgrad, wgrad) on integer-valued data: activations in {-2..2}, weights in {-1, 0, 1}, integer bias
  and residual.  Every product and partial sum is then an integer below 2^24, exact in fp32 in any order, and the
  epilogue rounds to nearest even: the kernel must EQUAL the float64 result rounded to bf16 (fp32 for wgrad).
- Every caller-owned output sits inside a larger buffer whose guard bytes hold a sentinel and must be unchanged; every
  caller-owned input is a view into a buffer whose neighbours hold NaN, so a read outside its extent shows up in the
  (exact) results.
- Train-mode BatchNorm at every C against float64 with per-element bounds derived from the fp32 evaluation.
- The inference network at every accepted architecture and tower schedule against a float64 copy of its graph, layer by
  layer, and the search-mode evaluator's values against the network's.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import helpers as H
from oracle import kv_oracle as O

pytestmark = pytest.mark.gpu
TOL = 2e-2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SENT16, SENT32 = 0x5A5A, 0x5A5A5A5A          # guard fill of bf16 / fp32 outputs (finite, unlikely as a result)
BOARD_GUARD = 4                              # boards of guard on each side of a board-shaped buffer
VEC_GUARD = 256                              # fp32 elements (1 KB) of guard on each side of a vector


@pytest.fixture(scope="module")
def eng():
    from knightvision_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _check(eng, rc, what):
    from knightvision_b200 import _native as N
    N.check(eng.ctx, rc, what)


# ---- guarded outputs and NaN-framed inputs -------------------------------------------------------------------------
def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _guarded(shape, dtype, guard):
    """(buffer, view): the view [shape] starts `guard` rows into a buffer filled with the sentinel bit pattern."""
    buf = torch.empty((shape[0] + 2 * guard,) + tuple(shape[1:]), dtype=dtype, device="cuda")
    _bits(buf).fill_(SENT16 if buf.element_size() == 2 else SENT32)
    return buf, buf[guard:guard + shape[0]]


def _guards_intact(buf, guard, n):
    s = SENT16 if buf.element_size() == 2 else SENT32
    return bool((_bits(buf[:guard]) == s).all()) and bool((_bits(buf[guard + n:]) == s).all())


def _nan_framed(t, guard):
    """A copy of t as a (contiguous) view into a buffer whose other rows are NaN."""
    buf = torch.full((t.shape[0] + 2 * guard,) + tuple(t.shape[1:]), float("nan"), dtype=t.dtype, device=t.device)
    buf[guard:guard + t.shape[0]] = t
    return buf[guard:guard + t.shape[0]]


# ---- float64 references -----------------------------------------------------------------------------------------------
def _im2col(x):
    """NHWC [n,8,8,c] -> float64 [n*64, 9*c], column (tap, c) = x[b, y+ky-1, x+kx-1, c] (zero outside the board)."""
    n, c = x.shape[0], x.shape[3]
    xp = F.pad(x.double(), (0, 0, 1, 1, 1, 1))
    return torch.stack([xp[:, ky:ky + 8, kx:kx + 8, :] for ky in range(3) for kx in range(3)], dim=3).reshape(n * 64, 9 * c)


def _conv_ref(x, w, bias=None, res=None, relu=False):
    """float64 [relu](conv3x3(x, w) + bias [+ res]) on NHWC, w [Cout,Cin,3,3] (cross-correlation, zero padding)."""
    n, cout = x.shape[0], w.shape[0]
    y = _im2col(x) @ w.double().permute(0, 2, 3, 1).reshape(cout, -1).T
    if bias is not None:
        y = y + bias.double()
    y = y.reshape(n, 8, 8, cout)
    if res is not None:
        y = y + res.double()
    return y.clamp(min=0) if relu else y


def _wgrad_ref(x, dy):
    """float64 dW[co][ci][ky][kx] = sum over pixels of dy[p][co] * x[p + (ky-1, kx-1)][ci]."""
    cout, cin = dy.shape[3], x.shape[3]
    g = dy.reshape(-1, cout).double().T @ _im2col(x)
    return g.reshape(cout, 3, 3, cin).permute(0, 3, 1, 2)


def _ints(shape, lo, hi, g, dtype=torch.bfloat16):
    return torch.randint(lo, hi + 1, shape, device="cuda", generator=g).to(dtype)


# ---- 1 + 2. convolutions: exact arithmetic at every accepted shape, outputs within their extent ----------------------
FPROP_CIN = (64, 128, 192, 256, 320, 384, 448, 512)
FPROP_N = (1, 2, 3, 5, 8, 9, 37, 301)         # 301: ceil(n/4) * cout/256 > 74 CTA pairs -> the pairs loop over tiles


def _fprop_raw(eng, x, wp, bias, res, y, relu):
    _check(eng, eng._lib.kv_conv3x3_fprop(eng.ctx, _ptr(x), _ptr(wp), _ptr(bias), _ptr(res), _ptr(y), int(x.shape[0]),
                                          int(x.shape[3]), int(wp.shape[0]), int(relu), eng._stream()), "kv_conv3x3_fprop")


def check_conv_case(eng, cin, cout, n, flags, seed, dgrad=False):
    """One fprop (or dgrad: fprop on the flip-transposed pack) on NaN-framed integer inputs into a guarded output.
    flags: bit 0 bias, bit 1 residual, bit 2 relu (fprop only).  Asserts bit equality with float64 and intact guards."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = _ints((cout, cin, 3, 3), -1, 1, g, torch.float32)
    if dgrad:         # dx = conv(dy, W'), W'[ci][co] = W[co][ci] with the taps mirrored; cin <-> cout
        x = _nan_framed(_ints((n, 8, 8, cout), -2, 2, g), BOARD_GUARD)
        wp = _nan_framed(eng.conv3x3_pack(w, flip_transpose=True), 8)
        bias = res = None
        relu = False
        cout_out = cin
        ref = _conv_ref(x, w.transpose(0, 1).flip(2, 3))
    else:
        x = _nan_framed(_ints((n, 8, 8, cin), -2, 2, g), BOARD_GUARD)
        wp = _nan_framed(eng.conv3x3_pack(w), 8)
        bias = _nan_framed(_ints((cout,), -3, 3, g, torch.float32), VEC_GUARD) if flags & 1 else None
        res = _nan_framed(_ints((n, 8, 8, cout), -2, 2, g), BOARD_GUARD) if flags & 2 else None
        relu = bool(flags & 4)
        cout_out = cout
        ref = _conv_ref(x, w, bias, res, relu)
    ybuf, y = _guarded((n, 8, 8, cout_out), torch.bfloat16, BOARD_GUARD)
    _fprop_raw(eng, x, wp, bias, res, y, relu)
    torch.cuda.synchronize()
    what = f"{'dgrad' if dgrad else 'fprop'} cin={cin} cout={cout} n={n} flags={flags}"
    assert _guards_intact(ybuf, BOARD_GUARD, n), what + ": write outside the output"
    assert torch.isfinite(y.float()).all(), what + ": read outside an input"
    exp = ref.to(torch.bfloat16)
    bad = (y.float() != exp.float())
    assert not bad.any(), f"{what}: {int(bad.sum())} elements differ from float64 rounded to bf16"


@pytest.mark.parametrize("cout", [256, 512])
@pytest.mark.parametrize("cin", FPROP_CIN)
def test_fprop_exact_every_shape(eng, cin, cout):
    """kv_conv3x3_fprop at every accepted cin (cin % 64 == 0, one to eight channel blocks per tap) and cout, board counts
    with partial 4-board tiles and one large enough that the CTA pairs loop; bias / residual / relu cycled."""
    shape = FPROP_CIN.index(cin) * 2 + (cout == 512)
    for i, n in enumerate(FPROP_N):
        check_conv_case(eng, cin, cout, n, (shape + i) % 8, seed=1000 * cin + cout + n)


@pytest.mark.parametrize("cin,cout", [(256, 256), (256, 512), (512, 256), (512, 512)])
def test_dgrad_exact(eng, cin, cout):
    for n in (1, 3, 5, 9, 37, 301):
        check_conv_case(eng, cin, cout, n, 0, seed=7 * cin + cout + n, dgrad=True)


def test_fprop_exact_without_halo_operand():
    """The 9-fetch fprop path (KV_CONV_HALO=0 is read once per process) in a child interpreter: same exact equality."""
    code = ("import sys; sys.path[:0] = [{root!r}, {tests!r}]\n"
            "import test_gpu_shapes as S\n"
            "from knightvision_b200.engine import Engine\n"
            "e = Engine(0)\n"
            "for i, cin in enumerate(S.FPROP_CIN):\n"
            "    for j, n in enumerate((1, 5, 37)):\n"
            "        S.check_conv_case(e, cin, (256, 512)[(i + j) % 2], n, (3 * i + j) % 8, seed=31 * cin + n)\n"
            "e.close()\n"
            "print('halo-less fprop exact')\n").format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    env = dict(os.environ, KV_CONV_HALO="0")
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "halo-less fprop exact" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def _wgrad_splits(sm_count, cin, cout, n):
    """Split-K rule of kv_conv3x3_wgrad: (splits, boards per split)."""
    tiles = (cout // 128) * (cin // 256) * 9
    s = max(sm_count // tiles, 1)
    s = min(s, n)
    return s, -(-n // s)


def _wgrad_raw(eng, x, dy, dw):
    _check(eng, eng._lib.kv_conv3x3_wgrad(eng.ctx, _ptr(x), _ptr(dy), _ptr(dw), int(x.shape[0]), int(x.shape[3]),
                                          int(dy.shape[3]), eng._stream()), "kv_conv3x3_wgrad")


def _wgrad_case(eng, cin, cout, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = _nan_framed(_ints((n, 8, 8, cin), -2, 2, g), BOARD_GUARD)
    dy = _nan_framed(_ints((n, 8, 8, cout), -2, 2, g), BOARD_GUARD)
    buf, dw = _guarded((cout, cin, 3, 3), torch.float32, 1)      # one row of guard = 9 * cin floats
    _wgrad_raw(eng, x, dy, dw)
    torch.cuda.synchronize()
    return x, dy, buf, dw


@pytest.mark.parametrize("cout", [128, 256, 384, 512])
@pytest.mark.parametrize("cin", [256, 512])
def test_wgrad_exact_split_cases(eng, cin, cout):
    """kv_conv3x3_wgrad at every cout tile count (odd ones included) and both cin, with board counts chosen from the
    split rule: one split; fewer boards than splits; a trailing split without boards; a long K (~1000 boards)."""
    S0 = _wgrad_splits(eng.sm_count, cin, cout, 1 << 30)[0]
    ns = {"one split": 1, "long K": 997}
    if S0 >= 3:
        ns["fewer boards than splits"] = S0 - 1
        ns["empty trailing split"] = next(n for n in range(S0 + 1, 4096) if (S0 - 1) * (-(-n // S0)) >= n)
    for kind, n in ns.items():
        s, bps = _wgrad_splits(eng.sm_count, cin, cout, n)
        if kind == "empty trailing split":
            assert (s - 1) * bps >= n
        x, dy, buf, dw = _wgrad_case(eng, cin, cout, n, seed=cin + cout + n)
        what = f"wgrad cin={cin} cout={cout} n={n} ({kind}, {s} splits of {bps} boards)"
        assert _guards_intact(buf, 1, cout), what + ": write outside the output"
        assert torch.isfinite(dw).all(), what + ": read outside an input"
        assert torch.equal(dw, _wgrad_ref(x, dy).float()), what
        dw2 = eng.conv3x3_wgrad(x, dy)
        assert torch.equal(dw2, dw), what + ": not deterministic"


def test_wgrad_workspace_reuse(eng):
    """Large shape, small shape, large again: the split workspace is reused without stale partial sums."""
    x, dy, _, dw = _wgrad_case(eng, 512, 512, 301, seed=1)
    first = dw.clone()
    xs, dys, _, dws = _wgrad_case(eng, 256, 128, 7, seed=2)
    assert torch.equal(dws, _wgrad_ref(xs, dys).float())
    assert torch.equal(eng.conv3x3_wgrad(x, dy), first)
    assert torch.equal(first, _wgrad_ref(x, dy).float())


# ---- 3. BatchNorm at every C against float64 -------------------------------------------------------------------------
def _ulp_bf16(a):
    """bf16 unit in the last place at |a| (8 significant bits)."""
    _, e = torch.frexp(a.abs().clamp(min=1e-30))
    return torch.ldexp(torch.ones_like(a), e - 8)


def _bn_inputs(n, C, seed):
    """z with four kinds of channel: ordinary (mean 0.3, std 1.7), large mean / small spread (32, 0.1), exactly
    constant, and channels whose pre-activations are all negative (beta -30)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    kind = torch.arange(C, device="cuda") % 4
    z = torch.randn(n, 8, 8, C, device="cuda", generator=g, dtype=torch.float64)
    z = torch.where(kind == 1, 32.0 + 0.1 * z, torch.where(kind == 2, torch.full_like(z, 0.75), 0.3 + 1.7 * z))
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.2
    beta = torch.where(kind == 3, torch.full_like(beta, -30.0), beta)
    res = torch.randn(n, 8, 8, C, device="cuda", generator=g).to(torch.bfloat16)
    dy = torch.randn(n, 8, 8, C, device="cuda", generator=g).to(torch.bfloat16)
    rm = torch.randn(C, device="cuda", generator=g)
    rv = torch.rand(C, device="cuda", generator=g) + 0.5
    return kind, z.to(torch.bfloat16), gamma, beta, res, dy, rm, rv


BN_CASES = [(n, C) for C in (64, 128, 256, 512, 1024) for n in (1, 3, 33, 600)]


@pytest.mark.parametrize("n,C", BN_CASES)
def test_bn_relu_against_float64(eng, n, C):
    """kv_bn_relu_fwd / kv_bn_relu_bwd / kv_channel_sum against float64, per element, with NaN-framed inputs and
    guarded outputs.  600 boards makes the reduction grid reach its 4-CTAs-per-SM cap.  Bounds:
      save_mean: 1e-6 of the mean |z|, save_rstd: 1e-6 relative, against two-pass float64 statistics of the bf16 z;
      running statistics: 1e-6 of the magnitudes of their two terms (momentum blend in fp32);
      y:  1/2 bf16 ulp + 2^-21 (|z s| + |mean s| + |beta| + |res|), s = gamma * rstd (fp32 evaluation of the folded
          affine transform, six roundings);
      dz: 1/2 bf16 ulp + 4 * 2^-23 |gamma rstd| (|g| + |dbeta/N| + |zhat dgamma/N|);
      dgamma, dbeta, channel_sum: 1e-5 of the per-channel sum of |terms|.
    The backward takes the saved statistics as inputs, so its references use them; the ReLU mask is the kernel's own
    bf16 y > 0 (what the backward reads), so every element is compared."""
    ci = BN_CASES.index((n, C))
    relu, with_res = ci % 2 == 0, ci % 3 != 1
    kind, z0, gamma0, beta0, res0, dy0, rm0, rv0 = _bn_inputs(n, C, seed=C + n)
    z, dy = _nan_framed(z0, BOARD_GUARD), _nan_framed(dy0, BOARD_GUARD)
    res = _nan_framed(res0, BOARD_GUARD) if with_res else None
    gamma, beta = _nan_framed(gamma0, VEC_GUARD), _nan_framed(beta0, VEC_GUARD)
    mom, eps = 0.1, 1e-5
    mom32, eps32 = float(np.float32(mom)), float(np.float32(eps))
    rows = n * 64
    ybuf, y = _guarded(z.shape, torch.bfloat16, BOARD_GUARD)
    vec = {k: _guarded((C,), torch.float32, VEC_GUARD) for k in ("mean", "rstd", "rm", "rv", "dg", "db", "cs")}
    vec["rm"][1].copy_(rm0)
    vec["rv"][1].copy_(rv0)
    mean, rstd, rm, rv, dg, db, cs = (vec[k][1] for k in ("mean", "rstd", "rm", "rv", "dg", "db", "cs"))
    _check(eng, eng._lib.kv_bn_relu_fwd(eng.ctx, _ptr(z), _ptr(res), _ptr(gamma), _ptr(beta), _ptr(rm), _ptr(rv), mom, eps,
                                        _ptr(y), _ptr(mean), _ptr(rstd), rows, C, int(relu), eng._stream()), "kv_bn_relu_fwd")
    dzbuf, dz = _guarded(z.shape, torch.bfloat16, BOARD_GUARD)
    drbuf, dres = _guarded(z.shape, torch.bfloat16, BOARD_GUARD)
    _check(eng, eng._lib.kv_bn_relu_bwd(eng.ctx, _ptr(dy), _ptr(y), _ptr(z), _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dz),
                                        _ptr(dres) if with_res else None, _ptr(dg), _ptr(db), rows, C, int(relu),
                                        eng._stream()), "kv_bn_relu_bwd")
    _check(eng, eng._lib.kv_channel_sum(eng.ctx, _ptr(dy), _ptr(cs), rows, C, eng._stream()), "kv_channel_sum")
    torch.cuda.synchronize()
    what = f"bn n={n} C={C} relu={relu} res={with_res}"
    for b in (ybuf, dzbuf) + ((drbuf,) if with_res else ()):
        assert _guards_intact(b, BOARD_GUARD, n), what + ": write outside a board-shaped output"
    if not with_res:
        assert (_bits(drbuf) == SENT16).all(), what + ": dres written although it was not asked for"
    for k, (b, _) in vec.items():
        assert _guards_intact(b, VEC_GUARD, C), f"{what}: write outside {k}"

    zd = z.double().reshape(rows, C)
    # statistics: two-pass float64 mean, biased variance for rstd, unbiased for the running variance
    m64 = zd.mean(0)
    var64 = ((zd - m64) ** 2).mean(0)
    rstd64 = 1.0 / torch.sqrt(var64 + eps32)
    assert ((mean.double() - m64).abs() <= 1e-6 * zd.abs().mean(0)).all(), what + ": save_mean"
    assert ((rstd.double() - rstd64).abs() <= 1e-6 * rstd64).all(), what + ": save_rstd"
    unb = var64 * rows / (rows - 1) if rows > 1 else var64
    for got, r0, new in ((rm, rm0, m64), (rv, rv0, unb)):
        exp = (1 - mom32) * r0.double() + mom32 * new
        assert ((got.double() - exp).abs() <= 1e-6 * ((1 - mom32) * r0.double().abs() + mom32 * new.abs())).all(), \
            what + ": running statistics"
    assert torch.isfinite(torch.stack([mean, rstd, rm, rv, dg, db, cs])).all(), what + ": read outside an input"

    # forward output, with the saved statistics
    s = gamma.double() * rstd.double()
    rd = res.double().reshape(rows, C) if with_res else torch.zeros_like(zd)
    pre = (zd - mean.double()) * s + beta.double() + rd
    y_ref = pre.clamp(min=0) if relu else pre
    e32 = 2.0 ** -21 * ((zd * s).abs() + (mean.double() * s).abs() + beta.double().abs() + rd.abs())
    yd = y.double().reshape(rows, C)
    assert ((yd - y_ref).abs() <= 0.5 * _ulp_bf16(y_ref.abs() + e32) + e32).all(), \
        f"{what}: y, max error {(yd - y_ref).abs().max().item():.3e}"

    # backward with the kernel's mask and saved statistics
    dyd = dy.double().reshape(rows, C)
    gg = dyd * (yd > 0) if relu else dyd
    zhat = (zd - mean.double()) * rstd.double()
    db_ref, dg_ref = gg.sum(0), (gg * zhat).sum(0)
    assert ((db.double() - db_ref).abs() <= 1e-5 * gg.abs().sum(0)).all(), what + ": dbeta"
    assert ((dg.double() - dg_ref).abs() <= 1e-5 * (gg * zhat).abs().sum(0)).all(), what + ": dgamma"
    dz_ref = s * (gg - db.double() / rows - zhat * dg.double() / rows)
    e32 = 4 * 2.0 ** -23 * s.abs() * (gg.abs() + (db.double() / rows).abs() + (zhat * dg.double() / rows).abs())
    dzd = dz.double().reshape(rows, C)
    assert ((dzd - dz_ref).abs() <= 0.5 * _ulp_bf16(dz_ref.abs() + e32) + e32).all(), \
        f"{what}: dz, max error {(dzd - dz_ref).abs().max().item():.3e}"
    if with_res:
        assert torch.equal(dres.double().reshape(rows, C), gg), what + ": dres"
    if relu:      # channels whose pre-activations are all negative pass no gradient at all
        neg = kind == 3
        assert (yd[:, neg] == 0).all()
        assert (dzd[:, neg] == 0).all() and (dg[neg] == 0).all() and (db[neg] == 0).all(), what + ": dead channels"
        if with_res:
            assert (dres.reshape(rows, C)[:, neg].float() == 0).all()
    assert ((cs.double() - dyd.sum(0)).abs() <= 1e-5 * dyd.abs().sum(0)).all(), what + ": channel_sum"


# ---- 4. the network at every accepted architecture and schedule ------------------------------------------------------
def bnrand_net(seed=0, **kw):
    """ChessNet with the weights of oracle/gen_golden.py's recipe: non-trivial BN statistics, so folding is exercised."""
    from knightvision_b200.model import ChessNet
    torch.manual_seed(seed)
    net = ChessNet(**kw).eval()
    g = torch.Generator().manual_seed(1)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.05)
            m.running_var.copy_(1.0 + 0.2 * torch.rand(m.running_var.shape, generator=g))
            m.weight.data.copy_(1.0 + 0.1 * torch.randn(m.weight.shape, generator=g))
            m.bias.data.copy_(0.05 * torch.randn(m.bias.shape, generator=g))
    return net


def live_heads(net):
    """Shift the BatchNorm of both 1x1 heads up by 0.5: with the default initialisation their two / one channels are
    often negative at every square after the ReLU, and policy and value then do not depend on the tower at all."""
    with torch.no_grad():
        net.policy_bn.bias.add_(0.5)
        net.value_bn.bias.add_(0.5)
    return net


class Fp64Net:
    """float64 copy of model._fp32_graph (the graph of ai/model.py:51-77, eval-mode BatchNorm) on `device`."""

    def __init__(self, net, device):
        self.sd = {k: v.detach().to(device, torch.float64) for k, v in net.state_dict().items()}
        self.arch = net.arch
        self.eps = {n + ".": m.eps for n, m in net.named_modules() if isinstance(m, torch.nn.BatchNorm2d)}

    def bn(self, p, t):
        s = self.sd
        return F.batch_norm(t, s[p + ".running_mean"], s[p + ".running_var"], s[p + ".weight"], s[p + ".bias"], False, 0.0,
                            self.eps[p + "."])

    def conv(self, p, t, pad=1):
        return F.conv2d(t, self.sd[p + ".weight"], self.sd[p + ".bias"], padding=pad)

    def tower_layers(self):
        """[(conv, bn, residual input = k convs back or None)] in the order of kv_net_forward_partial."""
        L = [("conv2", "bn2", None)] if self.arch[3] else []
        for i in range(self.arch[2]):
            L += [(f"res_blocks.{i}.conv1", f"res_blocks.{i}.bn1", None), (f"res_blocks.{i}.conv2", f"res_blocks.{i}.bn2", 2)]
        return L

    def stem(self, x):
        return F.relu(self.bn("bn1", self.conv("conv1", x.double())))

    def layer(self, k, h, res=None):
        conv, bn, _ = self.tower_layers()[k]
        t = self.bn(bn, self.conv(conv, h))
        return F.relu(t + res if res is not None else t)

    def heads(self, h):
        s = self.sd
        p = F.relu(self.bn("policy_bn", self.conv("policy_conv", h, 0))).flatten(1)
        p = F.linear(p, s["policy_fc.weight"], s["policy_fc.bias"])
        v = F.relu(self.bn("value_bn", self.conv("value_conv", h, 0))).flatten(1)
        v = F.relu(F.linear(v, s["value_fc1.weight"], s["value_fc1.bias"]))
        v = torch.tanh(F.linear(v, s["value_fc2.weight"], s["value_fc2.bias"]))
        return p, v

    def forward(self, x):
        h = self.stem(x)
        acts = [h]
        for k, (_, _, r) in enumerate(self.tower_layers()):
            h = self.layer(k, h, acts[-r] if r else None)
            acts.append(h)
        return self.heads(h)


ARCHS = [(64, 256, True, 1), (128, 256, True, 0), (192, 256, True, 1), (320, 512, True, 1), (448, 512, True, 2),
         (64, 512, True, 1), (512, 512, False, 1), (256, 256, False, 0)]
NET_N = (1, 5, 130)


def _arch_kw(a):
    return dict(stem=a[0], tower=a[1], conv2=a[2], blocks=a[3])


def _lines(n, seed):
    lines = H.random_playout_positions(n_games=max(2, n // 40 + 1), max_plies=80, seed=seed)
    idx = np.random.default_rng(seed).permutation(len(lines))[:n]
    assert len(idx) == n
    return lines[idx]


def _nchw(t):
    return t.double().permute(0, 3, 1, 2)


def _layer_errors(eng, net, ref, d):
    """[(kind, max rel, rms rel)] of every tower conv fed the kernel's own bf16 input (and residual) in float64, and
    the stem's error in bf16 ulps."""
    nconv = len(ref.tower_layers())
    acts = [_nchw(eng.net_forward_partial(d, k)) for k in range(nconv + 1)]
    out = []
    for k, (conv, _, r) in enumerate(ref.tower_layers()):
        kind = "stem->tower" if conv == "conv2" else ("block conv1" if conv.endswith("conv1") else "block conv2")
        exp = ref.layer(k, acts[k], acts[k + 1 - r] if r else None)
        err = acts[k + 1] - exp
        out.append((kind, (err.abs().max() / exp.abs().max()).item(),
                    (err.pow(2).mean().sqrt() / exp.pow(2).mean().sqrt()).item()))
    return acts[0], out


@pytest.fixture(scope="module")
def layer_baseline(eng):
    """Per layer kind, the largest max / RMS relative error of the known-good reference architecture (256, 512, 5)."""
    net = bnrand_net(seed=3).attach(eng, max_batch=130)
    eng.net_geometry = None
    lines = _lines(130, seed=40)
    from knightvision_b200.engine import lines_to_device
    _, errs = _layer_errors(eng, net, Fp64Net(net, "cuda"), lines_to_device(lines, eng.device))
    base = {}
    for kind, emax, erms in errs:
        b = base.get(kind, (0.0, 0.0))
        base[kind] = (max(b[0], emax), max(b[1], erms))
    return base


def _outputs(eng, net, d, nconv):
    mid = eng.net_forward_partial(d, nconv).clone()
    pol, val = (t.clone() for t in net.forward_lines(d))
    return mid, pol, val


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _forward_guarded(eng, d, n):
    """kv_net_forward into guarded policy / value buffers, the lines a view between boards of garbage."""
    lbuf = torch.full((n + 2 * BOARD_GUARD, 16), -1, dtype=torch.int64, device="cuda")
    lbuf[BOARD_GUARD:BOARD_GUARD + n] = d
    lines = lbuf[BOARD_GUARD:BOARD_GUARD + n]
    pbuf, pol = _guarded((n, 4096), torch.float32, BOARD_GUARD)
    vbuf, val = _guarded((n,), torch.float32, VEC_GUARD)
    _check(eng, eng._lib.kv_net_forward(eng.ctx, _ptr(lines), n, _ptr(pol), _ptr(val), eng._stream()), "kv_net_forward")
    torch.cuda.synchronize()
    assert _guards_intact(pbuf, BOARD_GUARD, n) and _guards_intact(vbuf, VEC_GUARD, n), "kv_net_forward wrote outside"
    return pol, val


@pytest.mark.parametrize("arch", ARCHS, ids=lambda a: f"{a[0]}-{a[1]}-{'T' if a[2] else 'F'}-{a[3]}")
def test_network_every_architecture(eng, arch, layer_baseline, capsys, monkeypatch):
    """Layer by layer against float64, final outputs within 2e-2 of float64, and every tower schedule: conv mode 1 ==
    mode 2 per-layer == whole-tower launch; halo kernel (fused 2) == its 4-CTA-cluster variants (3, 4) and within the
    accumulation-order bound of fused 0; every depth-first chunk size == the default chunk, bit for bit."""
    from knightvision_b200.engine import lines_to_device
    nmax = max(NET_N)
    net = live_heads(bnrand_net(seed=sum(arch[:2]) + arch[3], **_arch_kw(arch)))
    ref = Fp64Net(net, "cuda")
    nconv = len(ref.tower_layers())
    clusters = None
    report = []
    for n in NET_N:
        eng.net_geometry = None
        net.attach(eng, max_batch=nmax)
        clusters = eng.net_tower_clusters4()
        lines = _lines(n, seed=n + arch[0])
        d = lines_to_device(lines, eng.device)
        x = torch.from_numpy(O.encode(lines)).cuda()
        # layer by layer (default schedule)
        stem, errs = _layer_errors(eng, net, ref, d)
        exp = ref.stem(x)
        floor = torch.full_like(exp, 2.0 ** -12)
        ulps = ((stem - exp).abs() / _ulp_bf16(torch.maximum(exp.abs(), floor))).max().item()
        assert ulps <= 1.0, (arch, n, "stem", ulps)
        for kind, emax, erms in errs:
            bmax, brms = layer_baseline[kind]
            report.append((n, kind, emax, 2 * bmax, erms, 2 * brms))
            assert emax <= 2 * bmax and erms <= 2 * brms, (arch, n, kind, emax, bmax, erms, brms)
        rp, rv = ref.forward(x)
        if n > 1:         # the outputs depend on the position, i.e. on the tower
            assert rp.std(0).max().item() > 2e-3 and rv.std().item() > 2e-4, (arch, n, "heads independent of the tower")
        pol, val = _forward_guarded(eng, d, n)
        dp, dv = (pol - rp).abs().max().item(), (val - rv[:, 0]).abs().max().item()
        report.append((n, "policy/value", max(dp, dv), TOL, None, None))
        assert dp < TOL and dv < TOL, (arch, n, dp, dv)
        # schedules
        eng.net_set_conv_mode(1)
        o_m1 = _outputs(eng, net, d, nconv)
        eng.net_set_conv_mode(2)
        eng.net_set_tower_fused(0)
        o_f0 = _outputs(eng, net, d, nconv)
        eng.net_set_tower_fused(1)
        o_f1 = _outputs(eng, net, d, nconv)
        assert _same(o_m1, o_f0) and _same(o_f0, o_f1), (arch, n, "conv mode 1 / per-layer / whole-tower")
        eng.net_set_tower_fused(2)
        o_f2 = _outputs(eng, net, d, nconv)
        modes = (3, 4) if clusters >= 8 else ()
        for mode in modes:
            eng.net_set_tower_fused(mode)
            assert _same(_outputs(eng, net, d, nconv), o_f2), (arch, n, f"fused {mode} vs 2")
        m0, m2 = o_f0[0].float(), o_f2[0].float()
        assert ((m0 - m2).abs() <= 0.02 * m0.abs().clamp(min=1.0)).all(), (arch, n, "fused 2 vs 0")
        assert (o_f0[1] - o_f2[1]).abs().max().item() < 5e-3 and (o_f0[2] - o_f2[2]).abs().max().item() < 5e-3
        # depth-first chunk sizes (read by kv_net_create): bit-identical to the default chunking
        for chunk in ("1", "2", "3"):
            monkeypatch.setenv("KV_TOWER_CHUNK", chunk)
            eng.net_geometry = None
            net.attach(eng, max_batch=nmax)
            for mode, want in ((1, o_f1), (2, o_f2)):
                eng.net_set_tower_fused(mode)
                assert _same(_outputs(eng, net, d, nconv), want), (arch, n, f"chunk {chunk} fused {mode}")
        monkeypatch.delenv("KV_TOWER_CHUNK")
    eng.net_geometry = None
    with capsys.disabled():
        print(f"\n[arch stem {arch[0]} tower {arch[1]} conv2 {arch[2]} blocks {arch[3]}] max error / bound "
              f"(relative to max |float64| per tower layer; absolute for policy / value); 4-CTA clusters {clusters}")
        for n, kind, e, b, r, rb in report:
            print(f"  n={n:4d} {kind:12s} max {e:.3e} / {b:.3e}" + (f"   rms {r:.3e} / {rb:.3e}" if r is not None else ""))


def test_network_many_chunks_256_tower(eng, capsys):
    """The 256-wide tower at 1 201 boards (301 board tiles): the default depth-first chunking makes two unequal chunks
    (151 + 150 tiles); every schedule against float64 and against each other."""
    from knightvision_b200.engine import lines_to_device
    n = 1201
    arch = (64, 256, True, 1)
    net = live_heads(bnrand_net(seed=77, **_arch_kw(arch)))
    eng.net_geometry = None
    net.attach(eng, max_batch=n)
    ref = Fp64Net(net, "cuda")
    nconv = len(ref.tower_layers())
    lines = _lines(n, seed=5)
    d = lines_to_device(lines, eng.device)
    eng.net_set_tower_fused(0)
    o_f0 = _outputs(eng, net, d, nconv)
    eng.net_set_tower_fused(1)
    assert _same(_outputs(eng, net, d, nconv), o_f0)
    eng.net_set_tower_fused(2)
    o_f2 = _outputs(eng, net, d, nconv)
    if eng.net_tower_clusters4() >= 8:
        for mode in (3, 4):
            eng.net_set_tower_fused(mode)
            assert _same(_outputs(eng, net, d, nconv), o_f2), f"fused {mode}"
    m0, m2 = o_f0[0].float(), o_f2[0].float()
    assert ((m0 - m2).abs() <= 0.02 * m0.abs().clamp(min=1.0)).all()
    rp, rv = ref.forward(torch.from_numpy(O.encode(lines)).cuda())
    dp, dv = (o_f2[1] - rp).abs().max().item(), (o_f2[2] - rv).abs().max().item()
    eng.net_geometry = None
    with capsys.disabled():
        print(f"\n[256-wide tower, {n} boards] max |kernel - float64|: policy {dp:.3e}, value {dv:.3e} (bound {TOL:.0e})")
    assert dp < TOL and dv < TOL


# ---- 5. search-mode evaluator values equal the network's ------------------------------------------------------------
@pytest.mark.parametrize("arch", [(256, 256, False, 2), (256, 512, True, 5)], ids=["256x2", "reference"])
@pytest.mark.parametrize("split", [0, 1])
def test_search_root_value_equals_network(eng, arch, split):
    """After one wave, each root's value in the tree (the evaluator's own heads + value MLP, kv_mcts.cu) equals the
    value kv_net_forward gives for that position, from the side to move's point of view (kv_mcts.cuh: v = wtm ? v :
    -v): the same device functions with the same association, so bit for bit."""
    G = 16
    net = bnrand_net(seed=9, **_arch_kw(arch))
    eng.net_geometry = None
    net.attach(eng, max_batch=G)
    roots = eng.random_positions(G, max_plies=30, seed=11 + split)
    eng.mcts_create(G, 4, max_plies=4, temp_plies=0, seed=3, eval_mode=1)
    eng.mcts_set_eval_split(split)
    try:
        eng.mcts_reset(roots.clone(), 0)
        eng.mcts_run_sims(1)
        torch.cuda.synchronize()
        _, val = net.forward_lines(roots)
        val = val[:, 0].cpu().numpy()
        for g in range(G):
            nv, _, _, root = eng.mcts_dump_tree(g)
            assert np.array_equal(root.view(np.int64)[:12], roots[g, :12].cpu().numpy()), g
            wtm = bool(int(root[12]) & 1)
            exp = val[g] if wtm else -val[g]
            assert nv[0].view(np.uint32) == np.float32(exp).view(np.uint32), (g, nv[0], exp)
    finally:
        eng.mcts_set_eval_split(-1)
        eng.net_geometry = None
