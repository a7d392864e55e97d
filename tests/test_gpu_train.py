"""Training-side convolution operators (SURVEY 8f-2) on the B200 against plain PyTorch fp32 of the same op
(`F.conv2d` and its input / weight gradients): fprop, dgrad and the MN-major tcgen05 wgrad kernel, the autograd
function built from them, and one optimisation step of the reference's loss (scripts/train.py:158-190) through them.
Tolerances: outputs are bf16 (rel 2^-8 per element) with fp32 accumulation; wgrad is fp32 end to end."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from knightvision_b200.engine import Engine
    e = Engine(0)
    yield e
    e.close()


def _rel(a, r):
    return ((a.float() - r).abs().max() / r.abs().max()).item()


@pytest.mark.parametrize("n,cin,cout", [(1, 256, 256), (6, 256, 512), (101, 512, 512), (300, 512, 256)])
def test_fprop_dgrad_wgrad_match_torch_fp32(eng, n, cin, cout):
    g = torch.Generator(device="cuda").manual_seed(n)
    x = (torch.randn(n, 8, 8, cin, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    dy = (torch.randn(n, 8, 8, cout, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    w = torch.randn(cout, cin, 3, 3, device="cuda", generator=g) * 0.02
    b = torch.randn(cout, device="cuda", generator=g) * 0.1
    wb = w.to(torch.bfloat16).float()                       # the kernels see the bf16-rounded parameter
    xf, dyf = x.float().permute(0, 3, 1, 2), dy.float().permute(0, 3, 1, 2)
    ref_y = F.conv2d(xf, wb, b, padding=1).permute(0, 2, 3, 1)
    ref_dx = torch.nn.grad.conv2d_input(xf.shape, wb, dyf, padding=1).permute(0, 2, 3, 1)
    ref_dw = torch.nn.grad.conv2d_weight(xf, w.shape, dyf, padding=1)
    y = eng.conv3x3_fprop(x, eng.conv3x3_pack(w), b)
    dx = eng.conv3x3_fprop(dy, eng.conv3x3_pack(w, flip_transpose=True))
    dw = eng.conv3x3_wgrad(x, dy)
    assert y.shape == (n, 8, 8, cout) and dx.shape == (n, 8, 8, cin) and dw.shape == (cout, cin, 3, 3)
    assert _rel(y, ref_y) < 8e-3 and _rel(dx, ref_dx) < 8e-3        # bf16 output rounding
    assert _rel(dw, ref_dw) < 1e-4                                   # fp32 accumulate, fp32 out
    # relu / residual epilogue flags on caller-owned tensors
    res = (torch.randn(n, 8, 8, cout, device="cuda", generator=g)).to(torch.bfloat16)
    y2 = eng.conv3x3_fprop(x, eng.conv3x3_pack(w), b, residual=res, relu=True)
    assert _rel(y2, F.relu(ref_y + res.float())) < 8e-3
    # deterministic: split-K partials are added in a fixed order
    assert torch.equal(dw, eng.conv3x3_wgrad(x, dy))


def test_wgrad_taps_and_borders_exact(eng):
    """Integer-valued inputs make every product and partial sum exact in fp32: the nine taps, the zero padding at the
    board edges and the split-K reduction must then reproduce torch bit for bit."""
    n, cin, cout = 37, 256, 256
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randint(-2, 3, (n, 8, 8, cin), device="cuda", generator=g).to(torch.bfloat16)
    dy = torch.randint(-2, 3, (n, 8, 8, cout), device="cuda", generator=g).to(torch.bfloat16)
    ref = torch.nn.grad.conv2d_weight(x.float().permute(0, 3, 1, 2), (cout, cin, 3, 3), dy.float().permute(0, 3, 1, 2),
                                      padding=1)
    assert torch.equal(eng.conv3x3_wgrad(x, dy), ref)
    w = torch.randint(-1, 2, (cout, cin, 3, 3), device="cuda", generator=g).float()
    refx = torch.nn.grad.conv2d_input((n, cout, 8, 8)[:1] + (cin, 8, 8), w, dy.float().permute(0, 3, 1, 2), padding=1)
    dx = eng.conv3x3_fprop(dy, eng.conv3x3_pack(w, flip_transpose=True))
    # |dx| <= 2 * 9 * 256 = 4608 would not fit bf16 exactly; compare after the same rounding
    assert torch.equal(dx.float(), refx.permute(0, 2, 3, 1).to(torch.bfloat16).float())


def test_autograd_function_matches_torch(eng):
    from knightvision_b200.train_ops import conv3x3_b200
    torch.manual_seed(1)
    n = 48
    x0 = torch.randn(n, 256, 8, 8, device="cuda")
    w1 = (torch.randn(512, 256, 3, 3, device="cuda") * 0.02).requires_grad_()
    b1 = (torch.randn(512, device="cuda") * 0.1).requires_grad_()
    w2 = (torch.randn(512, 512, 3, 3, device="cuda") * 0.02).requires_grad_()
    tgt = torch.randn(n, 512, 8, 8, device="cuda")

    def run(conv):
        x = x0.clone().requires_grad_()
        h = F.relu(conv(x, w1, b1))
        y = conv(h, w2, None)
        loss = ((y.float() - tgt) ** 2).mean()
        gx, g1, gb, g2 = torch.autograd.grad(loss, (x, w1, b1, w2))
        return loss.item(), gx, g1, gb, g2

    ref = run(lambda x, w, b: F.conv2d(x, w, b, padding=1))                       # plain fp32
    def cudnn_bf16(x, w, b):                                                     # what autocast would run
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return F.conv2d(x, w, b, padding=1)
    lib = run(cudnn_bf16)
    got = run(lambda x, w, b: conv3x3_b200(x, w, b, eng))
    assert abs(got[0] - ref[0]) < 5e-3 * abs(ref[0])
    for a, r, l in zip(got[1:], ref[1:], lib[1:]):
        assert a.shape == r.shape
        # two bf16 layers deep with bf16 gradients: no further from fp32 than the library's bf16 path is (x 1.5 + eps)
        assert _rel(a, r) < max(1.5 * _rel(l, r), 1e-2), (_rel(a, r), _rel(l, r))


def test_training_step_native_vs_cudnn(eng, monkeypatch):
    """One optimisation step of the reference loss on the 20x256-style tower (2 blocks here) with the tower convolutions
    on the tcgen05 kernels vs on cuDNN: same loss and the same parameter update within bf16 noise."""
    from knightvision_b200 import learn as LR
    from knightvision_b200.model import ChessNet
    from knightvision_b200 import layout as L
    torch.manual_seed(7)
    lines = torch.from_numpy(np.stack([L.start_line()] * 96).view(np.int64)).cuda()
    moves = torch.randint(0, 4096, (96,), device="cuda")
    rewards = torch.tensor([1.0, 0.2, -1.0] * 32, device="cuda")
    results = {}
    for native in ("1", "0"):
        monkeypatch.setenv("KV_TRAIN_NATIVE", native)
        torch.manual_seed(3)
        net = ChessNet(stem=256, tower=256, blocks=2, conv2=False, max_batch=96).cuda()
        opt = torch.optim.SGD(net.parameters(), lr=0.05)
        data = LR.ReplayData(eng)
        data.extend_packed(lines, moves, rewards)
        l0 = eng.launches
        loss = LR.train_epochs(net, opt, data, epochs=1, batch_size=96, accumulate_steps=1)
        results[native] = (loss, net.weight_blob().clone(), eng.launches - l0)
    assert np.isfinite(results["1"][0]) and abs(results["1"][0] - results["0"][0]) < 2e-2 * abs(results["0"][0])
    assert results["1"][2] >= 4 * 3 and results["0"][2] == 1          # 4 tower convs x (fprop, dgrad, wgrad) + encode
    d = (results["1"][1] - results["0"][1]).abs().max().item()
    assert d < 5e-3, d


@pytest.mark.parametrize("rows_boards,C,with_res,relu", [
    pytest.param(3, 256, False, True, id="3-256-False"), pytest.param(77, 512, True, True, id="77-512-True"),
    pytest.param(512, 256, True, True, id="512-256-True"), pytest.param(5, 64, True, True, id="5-64-True"),
    pytest.param(33, 128, False, True, id="33-128-False"), pytest.param(9, 1024, True, True, id="9-1024-True"),
    pytest.param(40, 256, True, False, id="40-256-True-norelu"), pytest.param(7, 1024, False, False, id="7-1024-False-norelu")])
def test_bn_relu_fwd_bwd_match_torch_fp32(eng, rows_boards, C, with_res, relu):
    """Fused train-mode BatchNorm + ReLU (+ residual) against torch fp32 on the same bf16 inputs: outputs, input / skip /
    affine gradients, saved and running statistics, at every supported C and with the ReLU on or off."""
    n = rows_boards
    g = torch.Generator(device="cuda").manual_seed(C + n)
    z = (torch.randn(n, 8, 8, C, device="cuda", generator=g) * 1.7 + 0.3).to(torch.bfloat16)
    res = torch.randn(n, 8, 8, C, device="cuda", generator=g).to(torch.bfloat16) if with_res else None
    dy = torch.randn(n, 8, 8, C, device="cuda", generator=g).to(torch.bfloat16)
    gamma = (torch.rand(C, device="cuda", generator=g) + 0.5)
    beta = torch.randn(C, device="cuda", generator=g) * 0.2
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    y, mean, rstd = eng.bn_relu_fwd(z, gamma, beta, rm, rv, 0.1, 1e-5, residual=res, relu=relu)
    dz, dres, dgamma, dbeta = eng.bn_relu_bwd(dy, y, z, gamma, mean, rstd, relu=relu, want_dres=with_res)
    # torch fp32 reference
    zf = z.float().permute(0, 3, 1, 2).clone().requires_grad_()
    gf, bf = gamma.clone().requires_grad_(), beta.clone().requires_grad_()
    rf = res.float().permute(0, 3, 1, 2).clone().requires_grad_() if with_res else None
    rm2, rv2 = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    pre = F.batch_norm(zf, rm2, rv2, gf, bf, True, 0.1, 1e-5)
    out = pre + rf if with_res else pre
    if relu:
        out = F.relu(out)
    # the kernel masks with its own bf16 output; use the same mask for the reference gradient where out is within rounding of 0
    out.backward(dy.float().permute(0, 3, 1, 2))
    assert _rel(y.permute(0, 3, 1, 2), out.detach()) < 6e-3
    assert torch.allclose(rm, rm2, atol=1e-5, rtol=1e-4) and torch.allclose(rv, rv2, atol=1e-5, rtol=1e-4)
    assert torch.allclose(mean, zf.detach().mean(dim=(0, 2, 3)), atol=1e-5, rtol=1e-4)
    assert _rel(dgamma, gf.grad) < 5e-3 and _rel(dbeta, bf.grad) < 5e-3
    # the ReLU mask of an element whose pre-activation is within fp32 rounding of 0 may differ between two correct
    # implementations; such elements (a handful in millions) are excluded from the element-wise gradient comparison
    pre_act = (pre + rf if with_res else pre).detach()
    safe = pre_act.abs() > 1e-4
    assert safe.float().mean().item() > 0.999
    def rel_safe(a, r):
        return (((a.float() - r).abs() * safe).max() / r.abs().max()).item()
    assert rel_safe(dz.permute(0, 3, 1, 2), zf.grad) < 1.2e-2
    if with_res:
        assert rel_safe(dres.permute(0, 3, 1, 2), rf.grad) < 6e-3
    # column sums (conv bias gradient): exact for these magnitudes up to fp32 summation order
    cs = eng.channel_sum(dy)
    assert torch.allclose(cs, dy.float().sum(dim=(0, 1, 2)), atol=2e-3, rtol=1e-5)
    assert torch.equal(cs, eng.channel_sum(dy))


def test_residual_block_node_matches_the_chained_operators(eng, monkeypatch):
    """The one-node residual block (skip gradient fused into the dgrad epilogue) against the same block built from the
    separate conv / bn_relu autograd functions, and against plain PyTorch fp32."""
    from knightvision_b200 import train_ops as T
    from knightvision_b200.model import _Block
    torch.manual_seed(11)
    blk = _Block(256).cuda().train()
    with torch.no_grad():
        for p in blk.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    x0 = torch.randn(40, 256, 8, 8, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    tgt = torch.randn(40, 256, 8, 8, device="cuda")

    def run(kind):
        import copy
        b = copy.deepcopy(blk)
        x = x0.clone().requires_grad_()
        if kind == "node":
            y = T.residual_block_b200(x, b, eng)
        elif kind == "chain":
            t = T.bn_relu_b200(T.conv3x3_b200(x, b.conv1.weight, b.conv1.bias, eng), b.bn1, eng)
            y = T.bn_relu_b200(T.conv3x3_b200(t, b.conv2.weight, b.conv2.bias, eng), b.bn2, eng, residual=x)
        elif kind == "lib":           # what the reference runs: autocast + cuDNN + torch BatchNorm
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = F.relu(b.bn2(b.conv2(F.relu(b.bn1(b.conv1(x))))) + x)
        else:
            xf = x.float()
            y = F.relu(b.bn2(b.conv2(F.relu(b.bn1(b.conv1(xf))))) + xf)
        loss = ((y.float() - tgt) ** 2).mean()
        params = [b.conv1.weight, b.bn1.weight, b.bn1.bias, b.conv2.weight, b.bn2.weight, b.bn2.bias]
        grads = torch.autograd.grad(loss, [x] + params)
        return loss.item(), [g.float() for g in grads], b
    ln, gn, bn_ = run("node")
    lc, gc, bc = run("chain")
    lf, gf, _ = run("fp32")
    ll, gl, _ = run("lib")
    assert ln == pytest.approx(lc, rel=1e-3) and ln == pytest.approx(lf, rel=2e-2)
    l2 = lambda a, r: ((a - r).norm() / r.norm()).item()
    for a, c, f, l in zip(gn, gc, gf, gl):
        assert _rel(a, c) < 1.5e-2                 # same kernels; dx differs by one bf16 rounding (fused add)
        # bf16 vs fp32: ReLU masks of pre-activations within bf16 rounding of 0 legitimately differ, so the error is
        # judged in the L2 norm and against what the library's own bf16 path (autocast + cuDNN) makes of the same block
        assert l2(a, f) < max(1.5 * l2(l, f), 1e-2), (l2(a, f), l2(l, f))
    for a, c in zip(bn_.buffers(), bc.buffers()):
        assert torch.equal(a, c)                   # running statistics and num_batches_tracked
