"""TRAINING-path kernels (SURVEY.md 8 f-2): every backward / staging kernel against the float64 torch stand-ins of
oracle/train_ops.py on seeded inputs, then the whole training step (MatcherTrainFn forward + backward on the kernels, the
CUDA match loss) against the gradients of the unmodified reference (tests/golden/train_backward_*.npz)."""
import json
import os

import numpy as np
import pytest
import torch

from tests import emul_ops

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _rel(got, ref):
    ref = ref.double()
    return float((got.double().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize('variant', [1, 0])       # 1 = mma.sync TF32x3 (default), 0 = fp32 CUDA cores
@pytest.mark.parametrize('is_cross,counts', [(0, [128, 128]), (1, [128, 128, 128]), (1, [100, 100, 100, 100]), (0, [70, 128, 33]),
                                             (1, [70, 128, 33]), (1, [150, 192, 101])])
def test_attention_backward_vs_torch(is_cross, counts, variant):
    from e2e_multi_view_matching_b200 import ops, _lib
    _lib.lib().mvm_debug_set_attention_backward_variant(variant)
    g = torch.Generator().manual_seed(5 + is_cross + len(counts))
    T, B, n_pad = len(counts), 2, (max(counts) + 63) // 64 * 64          # (192 = three 64-row tiles: not a multiple of 128)
    qkv = torch.randn(B * T, n_pad, 768, generator=g) * 1.5
    dout = torch.randn(B * T, n_pad, 256, generator=g)
    for v in range(B * T):
        dout[v, counts[v % T]:] = 0          # the gradient of padding rows is zero by construction
    out = emul_ops.attention(qkv, B, T, counts, is_cross)
    ref = emul_ops.attention_backward(qkv, out, dout, B, T, counts, is_cross)
    try:
        got = ops.attention_backward(qkv.cuda(), out.cuda(), dout.cuda(), B, T, counts, is_cross)
        torch.cuda.synchronize()
    finally:
        _lib.lib().mvm_debug_set_attention_backward_variant(1)
    for name, lo in (('dq', 0), ('dk', 256), ('dv', 512)):
        e = _rel(got[:, :, lo:lo + 256], ref[:, :, lo:lo + 256])
        print('attention backward variant', variant, 'cross' if is_cross else 'self', counts, name, 'rel err %.2e' % e)
        assert e < 2e-5, (name, e)
    for v in range(B * T):
        assert float(got[v, counts[v % T]:].abs().max()) == 0.0 if counts[v % T] < n_pad else True


@pytest.mark.parametrize('groups,relu', [(1, True), (2, True), (1, False)])
def test_batchnorm_train_forward_backward_vs_torch(groups, relu):
    from e2e_multi_view_matching_b200 import ops
    g = torch.Generator().manual_seed(11)
    n_pad, n_valid, slots, C = 128, 100, 6, 96
    rows = slots * n_pad
    x = torch.randn(rows, C, generator=g) * 3 + 1
    w, b = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    dy = torch.randn(rows, C, generator=g)
    dy.view(slots, n_pad, C)[:, n_valid:] = 0
    rm, rv = torch.zeros(C), torch.ones(C)
    y_ref, st_ref = emul_ops.batchnorm_train(x, w, b, rm, rv, 0.1, 1e-5, n_pad, n_valid, relu=relu, groups=groups,
                                             out=torch.zeros_like(x), save=True)
    dx_ref = dy.clone()
    dg_ref, db_ref = emul_ops.batchnorm_train_backward(x, y_ref, dx_ref, w, st_ref, n_pad, n_valid, relu=relu)
    rmc, rvc = torch.zeros(C).cuda(), torch.ones(C).cuda()
    xc = x.cuda()
    y, st = ops.batchnorm_train(xc, w.cuda(), b.cuda(), rmc, rvc, 0.1, 1e-5, n_pad, n_valid, relu=relu, groups=groups,
                                out=torch.zeros_like(xc), save=True)
    dx = dy.cuda()
    dg, db = ops.batchnorm_train_backward(xc, y, dx, w.cuda(), st, n_pad, n_valid, relu=relu)
    torch.cuda.synchronize()
    assert _rel(y, y_ref) < 1e-5 and _rel(st, st_ref) < 1e-5
    assert _rel(rmc, rm) < 1e-5 and _rel(rvc, rv) < 1e-5
    assert _rel(dx, dx_ref) < 2e-5, _rel(dx, dx_ref)
    assert _rel(dg, dg_ref) < 2e-5 and _rel(db, db_ref) < 2e-5


@pytest.mark.parametrize('m,n,spread', [(64, 64, 3.0), (100, 100, 30.0), (37, 90, 10.0), (450, 520, 10.0)])     # last: > 415 columns (KC = 33 kernels)
def test_sinkhorn_train_vs_autograd(m, n, spread):
    from e2e_multi_view_matching_b200 import ops
    g = torch.Generator().manual_seed(m + n)
    B, iters = (3, 100) if n <= 415 else (2, 100)
    scores = torch.randn(B, m, n, generator=g) * spread
    alpha = torch.tensor([1.3])
    G = torch.randn(B, m + 1, n + 1, generator=g)
    Z_ref, _ = emul_ops.sinkhorn_train_forward(scores, alpha, iters)
    dZ_ref, da_ref = emul_ops.sinkhorn_train_backward(scores, alpha, None, iters, G)
    Z, pot = ops.sinkhorn_train_forward(scores.cuda(), alpha.cuda(), iters)
    dZ, da = ops.sinkhorn_train_backward(scores.cuda(), alpha.cuda(), pot, iters, G.cuda())
    torch.cuda.synchronize()
    ez = float((Z.cpu().double() - Z_ref.double()).abs().max())
    eg = _rel(dZ[:, :m, :n], dZ_ref[:, :m, :n])
    ea = abs(float(da) - float(da_ref)) / max(abs(float(da_ref)), 1e-12)
    print('sinkhorn train %dx%d spread %.0f: couplings abs err %.2e, d scores rel err %.2e, d alpha rel err %.2e' % (m, n, spread, ez, eg, ea))
    assert ez < 2e-4 * max(1.0, spread) and eg < 2e-4 and ea < 2e-4


@pytest.mark.parametrize('rows,n_out,k_in,k2', [(384, 256, 256, 0), (896, 512, 256, 256), (384, 768, 256, 0), (384, 64, 32, 0),
                                                (384, 32, 16, 0), (384, 256, 128, 0), (17920, 256, 256, 0), (8960, 512, 256, 256),
                                                (4480, 768, 256, 0)])     # the last three: split-K weight gradients
def test_backward_gemms_vs_fp64(rows, n_out, k_in, k2):
    from e2e_multi_view_matching_b200 import ops
    g = torch.Generator().manual_seed(rows + n_out)
    dy = torch.randn(rows, n_out, generator=g) * 1e-3          # gradients are small: the 3xTF32 path keeps the fp32 range
    x = torch.randn(rows, k_in, generator=g)
    x2 = torch.randn(rows, k2, generator=g) if k2 else None
    w = torch.randn(n_out, k_in + k2, generator=g) * 0.1
    res = torch.randn(rows, k_in + k2, generator=g) * 1e-4
    dx = ops.gemm_dx(dy.cuda(), w.cuda(), residual=res.cuda())
    dw = ops.gemm_dw(dy.cuda(), x.cuda(), x2.cuda() if k2 else None)
    torch.cuda.synchronize()
    dx_ref = dy.double() @ w.double() + res.double()
    dw_ref = dy.double().t() @ (torch.cat([x, x2], 1) if k2 else x).double()
    assert _rel(dx, dx_ref) < 1e-5, _rel(dx, dx_ref)
    assert _rel(dw, dw_ref) < 1e-5, _rel(dw, dw_ref)
    cs = ops.colsum(dy.cuda())
    assert _rel(cs, dy.double().sum(0)) < 1e-5


def _golden_case(name):
    from oracle.make_train_backward_golden import build
    from e2e_multi_view_matching_b200.models.multi_view_matcher import MultiViewMatcher
    z = np.load(os.path.join(GOLDEN, 'train_backward_%s.npz' % name))
    case = json.loads(str(z['meta']))
    data_np, sd = build(case)
    model = MultiViewMatcher({'multi_frame_matching': case['multi'], 'GNN_layers': case['layers'], 'conf_mlp': True,
                              'full_output': False})
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    data = {k: (torch.from_numpy(v).cuda() if isinstance(v, np.ndarray) else v) for k, v in data_np.items()}
    return z, case, model.cuda().train(), data


def _loss(case, model, data):
    from e2e_multi_view_matching_b200.training import compute_match_loss
    result = model(data)
    loss = 0.0
    for b in range(case['views']):
        for a in range(b):
            key = '%d_%d' % (a, b)
            loss = loss + compute_match_loss(result['scores_' + key], data['gt_indices_' + key], data['gt_weights_' + key])
    return loss


def test_pair_scores_and_augmented_sinkhorn_layout():
    """Score matrices of every (pair, tuple) in one launch (score mode of the persistent GEMM) into [B, N+1, N+1] buffers,
    read in place by the Sinkhorn training kernels."""
    from e2e_multi_view_matching_b200 import ops
    g = torch.Generator().manual_seed(3)
    B, T, N, n_pad = 2, 3, 100, 128
    md = torch.randn(B, T, n_pad, 256, generator=g)
    pairs = [(0, 1), (0, 2), (1, 2)]
    ref = emul_ops.pair_scores(md, pairs, N)
    got = ops.pair_scores(md.cuda(), pairs, N)
    assert _rel(got[:, :N, :N], ref[:, :N, :N]) < 1e-5
    alpha = torch.tensor([0.7])
    Z_ref, _ = emul_ops.sinkhorn_train_forward(ref, alpha, 100, augmented=True)
    Z, pot = ops.sinkhorn_train_forward(got, alpha.cuda(), 100, augmented=True)
    G = torch.randn(Z_ref.shape, generator=g)
    dZ_ref, da_ref = emul_ops.sinkhorn_train_backward(ref, alpha, None, 100, G, augmented=True)
    dZ, da = ops.sinkhorn_train_backward(got, alpha.cuda(), pot, 100, G.cuda(), augmented=True)
    torch.cuda.synchronize()
    assert float((Z.cpu().double() - Z_ref.double()).abs().max()) < 5e-4
    assert _rel(dZ[:, :N, :N], dZ_ref[:, :N, :N]) < 2e-4 and abs(float(da) - float(da_ref)) <= 2e-4 * abs(float(da_ref)) + 1e-6


def _to_cpu(o):
    if torch.is_tensor(o):
        return o.detach().cpu()
    if isinstance(o, (list, tuple)):
        return type(o)(_to_cpu(x) for x in o)
    return o


@pytest.mark.parametrize('name', ['mv3_64', 'mv4_100', 'pair_96'])
def test_backward_system_vs_standins_on_the_gpu_forward_state(name, monkeypatch):
    """The whole backward (every kernel in sequence, 100+ launches) against the float64 stand-ins run on the SAME saved
    forward state (the GPU's activations, BatchNorm statistics and ReLU masks): isolates the backward kernels from the
    rounding of the forward -- a pre-ReLU activation within ~1e-5 of zero flips its mask between two correct forwards,
    which moves the gradient by far more than rounding does (profiles/r02_train_kink.txt)."""
    import copy
    from e2e_multi_view_matching_b200 import ops, _lib
    from e2e_multi_view_matching_b200.models import train_forward as TF
    from e2e_multi_view_matching_b200.training import compute_match_loss
    from tests.test_train_host_logic import PATCHED
    z, case, model, data = _golden_case(name)
    ids = None if case['multi'] else [0, 1]
    with torch.no_grad():
        result, S = TF._forward(model, data, ids, save=True)
    grads = {}
    for k, Z in result.items():
        key = k[len('scores_'):]
        leaf = Z.detach().clone().requires_grad_(True)
        compute_match_loss(leaf, data['gt_indices_' + key], data['gt_weights_' + key]).backward()
        grads[k] = leaf.grad
    with torch.no_grad():
        G = TF._backward(model, S, grads)
    torch.cuda.synchronize()
    names = {p: n for n, p in model.named_parameters()}
    got = {names[p]: g.detach().cpu().double() for p, g in G.items()}
    # the same backward on the CPU stand-ins, fed with the GPU's saved state
    model_c = copy.deepcopy(model).cpu()
    S_c = TF._Saved()
    for k, v in vars(S).items():
        setattr(S_c, k, _to_cpu(v))
    S_c.dev = torch.device('cpu')
    for f in PATCHED:
        monkeypatch.setattr(ops, f, getattr(emul_ops, f))
    with torch.no_grad():
        G_c = TF._backward(model_c, S_c, {k: v.cpu() for k, v in grads.items()})
    names_c = {p: n for n, p in model_c.named_parameters()}
    ref = {names_c[p]: g.detach().double() for p, g in G_c.items()}
    assert sorted(got) == sorted(ref) and len(got) > 50
    scale = max(float(v.abs().max()) for v in ref.values())
    worst = (0.0, None)
    for k in ref:
        e = float((got[k] - ref[k]).abs().max()) / max(float(ref[k].abs().max()), 1e-3 * scale)
        worst = max(worst, (e, k))
        assert e < 5e-4, (k, e)      # the fp32 Sinkhorn recursion alone contributes up to 5e-5 (test_sinkhorn_train_vs_autograd)
    print(name, 'backward on the kernels vs float64 stand-ins on the same forward state: worst relative error %.2e at %s' % worst)


@pytest.mark.parametrize('name', ['mv3_64', 'mv4_100', 'pair_96'])
def test_train_step_vs_reference_golden(name):
    """loss.backward() through the kernels against the reference's autograd (its fp64 run).  The loss matches to the
    reference's own fp32 deviation.  The gradients are bounded by what ONE flipped ReLU mask does (the measured error /
    reference-deviation ratios are printed: median 2-11, i.e. most parameters sit within a few times the reference's own
    fp32-vs-fp64 deviation when no mask flips upstream of them) (an activation within ~1e-5 of zero has a different sign in two correctly rounded forwards: measured
    on the float64 stand-ins with a 1e-6 forward perturbation, profiles/r02_train_kink.txt: up to 7e-3 of the gradient's
    scale) -- 2e-2 of the parameter's gradient scale.  The backward itself is pinned tighter by the test above."""
    from oracle.make_train_backward_golden import sample_index
    from tests.test_train_host_logic import check_gradients
    z, case, model, data = _golden_case(name)
    model._train_debug = {}
    loss = _loss(case, model, data)
    noise = abs(float(z['loss_f32']) - float(z['loss_f64']))
    assert abs(float(loss) - float(z['loss_f64'])) <= 8 * noise + 2e-5 * abs(float(z['loss_f64'])), (float(loss), float(z['loss_f64']))
    loss.backward()
    torch.cuda.synchronize()
    for k, g in model._train_debug.items():        # gradients at the stage boundaries (reference layout [T, B, 256, N])
        if k in ('g_gnn', 'g_kenc') and 'inter__' + k in z.files:
            ref = z['inter__' + k].astype(np.float64)          # at the seeded positions of oracle/make_train_backward_golden.py
            got = g.cpu().numpy().transpose(1, 0, 3, 2).reshape(-1)
            err = float(np.abs(got[sample_index('inter__' + k, got.size)] - ref).max())
            print(name, k, 'max err %.3g = %.1f x the reference\'s fp32-vs-fp64 deviation (%.3g), |ref| max %.3g'
                  % (err, err / float(z['inter_noise__' + k]), float(z['inter_noise__' + k]), float(np.abs(ref).max())))
    worst, ratios = check_gradients(model, z, tol_noise=0.0, tol_rel=2e-2, what=name, return_ratios=True)
    print(name, 'loss %.6f (reference fp64 %.6f, fp32 %.6f); worst gradient error / (2e-2 of its scale) %.3f at %s'
          % (float(loss), float(z['loss_f64']), float(z['loss_f32']), worst[0], worst[1]))


def test_training_loop_reduces_the_loss():
    """A few optimiser steps on one batch through model(data) / loss.backward() / torch.optim: the loss goes down and the
    eval forward afterwards runs on the updated weights."""
    z, case, model, data = _golden_case('mv3_64')
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    losses = []
    for _ in range(6):
        opt.zero_grad(set_to_none=True)
        loss = _loss(case, model, data)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    print('match loss over 6 Adam steps:', ['%.1f' % v for v in losses])
    assert losses[-1] < 0.9 * losses[0] and all(np.isfinite(losses))
    out = model.eval()(data)
    assert torch.isfinite(out['scores_0_1']).all()
