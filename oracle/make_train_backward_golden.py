"""Golden gradients for the TRAINING step of the matcher (SURVEY.md 8 f-2, BASELINE cfg5 stage 1): the unmodified
reference MultiViewMatcher in .train() (batch-statistics BatchNorm, stacked views, combined cross attention), the
reference's OWN helpers.compute_match_loss (helpers.py:228-241) summed over the pairs like helpers.run_matcher
(:243-260), loss.backward() -- in fp32 and (yardstick) fp64 -> tests/golden/train_backward_*.npz: the loss and, per
parameter, the gradient (fp64 run stored as float32: in full up to 1024 elements, else 1024 seeded samples; its L2 norm; the largest
deviation of the reference's own fp32 run from its fp64 run over the WHOLE gradient = the yardstick `noise`), plus the gradients w.r.t.
the output of final_proj, of the GNN and of the keypoint encoder for stage-level diagnosis.
TEST INFRASTRUCTURE ONLY (needs /root/reference); the GPU test rebuilds inputs and weights from the seeds."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402
from oracle.make_validation_golden import gt_from_landmarks  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
CASES = [dict(name='mv3_64', multi=True, views=3, kpts=64, batch=2, layers=['self', 'cross', 'cross', 'self', 'cross'], wseed=61, iseed=71, gain=10.0),
         dict(name='mv4_100', multi=True, views=4, kpts=100, batch=2, layers=['self', 'cross'] * 2, wseed=62, iseed=72, gain=10.0),
         dict(name='pair_96', multi=False, views=2, kpts=96, batch=2, layers=['self', 'cross'] * 2, wseed=63, iseed=73, gain=10.0)]
N_SAMPLE = 1024


def build(case):
    from e2e_multi_view_matching_b200.synthetic import make_scene_tuple_inputs, make_state_dict
    data = make_scene_tuple_inputs(case['iseed'], n_views=case['views'], n_kpts=case['kpts'], batch=case['batch'])
    for b_ in range(case['views']):
        for a_ in range(b_):
            pairs = [gt_from_landmarks(data['landmark%d' % a_][b], data['landmark%d' % b_][b]) for b in range(case['batch'])]
            data['gt_indices_%d_%d' % (a_, b_)] = np.stack([p[0] for p in pairs])
            data['gt_weights_%d_%d' % (a_, b_)] = np.stack([p[1] for p in pairs])
    sd = make_state_dict(len(case['layers']), seed=case['wseed'], final_proj_gain=case['gain'], conf_head='score')
    return data, sd


def sample_index(name, numel):
    """Seeded sample positions of a large gradient (the same in the generator and in the test)."""
    if numel <= N_SAMPLE:
        return np.arange(numel)
    seed = sum(ord(c) * (i + 1) for i, c in enumerate(name)) % (2 ** 31)
    return np.sort(np.random.default_rng(seed).choice(numel, N_SAMPLE, replace=False))


def main():
    ref_shim.load()
    import helpers
    from models.models.multi_view_matcher import MultiViewMatcher
    assert helpers.__file__.startswith('/root/reference')
    torch.set_num_threads(8)
    report = {}
    for case in CASES:
        data_np, sd = build(case)
        out = {}
        for dtype, tag in ((torch.float32, 'f32'), (torch.float64, 'f64')):
            torch.manual_seed(0)
            model = MultiViewMatcher({'multi_frame_matching': case['multi'], 'GNN_layers': case['layers'], 'conf_mlp': True,
                                      'full_output': False})
            model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
            model = model.to(dtype).train()
            data = {k: (torch.from_numpy(v).to(dtype) if isinstance(v, np.ndarray) and v.dtype.kind == 'f' else
                        (torch.from_numpy(v) if isinstance(v, np.ndarray) else v)) for k, v in data_np.items()}
            inter = {}
            hooks = []

            def keep(name):
                def fn(mod, inp, outp):
                    outp.register_hook(lambda g: inter.__setitem__(name, g.detach().numpy().copy()))
                return fn
            hooks.append(model.final_proj.register_forward_hook(keep('g_mdesc')))
            if case['multi']:
                hooks.append(model.gnn.register_forward_hook(keep('g_gnn')))
                hooks.append(model.kenc.register_forward_hook(keep('g_kenc')))
            result = model(data)
            loss = 0.0
            for b_ in range(case['views']):
                for a_ in range(b_):
                    key = '%d_%d' % (a_, b_)
                    loss = loss + helpers.compute_match_loss(result['scores_' + key], data['gt_indices_' + key], data['gt_weights_' + key])
            loss.backward()
            for h_ in hooks:
                h_.remove()
            out['%s__loss' % tag] = np.float64(loss.item())
            for k, v in inter.items():
                out['%s__inter__%s' % (tag, k)] = v
            for k, p in model.named_parameters():
                if p.grad is not None:
                    out['%s__full__%s' % (tag, k)] = p.grad.detach().numpy().reshape(-1).astype(np.float64)
        small = {'meta': json.dumps(case), 'loss_f64': out['f64__loss'], 'loss_f32': out['f32__loss']}
        names = [k[len('f64__full__'):] for k in out if k.startswith('f64__full__')]
        rel = {}
        for k in names:
            g64, g32 = out['f64__full__' + k], out['f32__full__' + k]
            small['grad__' + k] = g64[sample_index(k, g64.size)].astype(np.float32)
            small['noise__' + k] = np.float64(np.abs(g32 - g64).max())
            small['norm__' + k] = np.float64(np.linalg.norm(g64))
            rel[k] = float(small['noise__' + k] / max(np.abs(g64).max(), 1e-30))
        for k in [k[len('f64__inter__'):] for k in out if k.startswith('f64__inter__')]:
            flat = out['f64__inter__' + k].reshape(-1)
            small['inter__' + k] = flat[sample_index('inter__' + k, flat.size)].astype(np.float32)
            small['inter_noise__' + k] = np.float64(np.abs(out['f32__inter__' + k].astype(np.float64) - out['f64__inter__' + k]).max())
        worst = max(rel, key=rel.get)
        report[case['name']] = {'loss_f64': float(out['f64__loss']), 'loss_f32': float(out['f32__loss']), 'n_params_with_grad': len(names),
                                'max_rel_ref32_vs_ref64': rel[worst], 'at': worst,
                                'median_rel_ref32_vs_ref64': float(np.median(list(rel.values())))}
        print(case['name'], report[case['name']])
        np.savez_compressed(os.path.join(OUT, 'train_backward_%s.npz' % case['name']), **small)
    json.dump(report, open(os.path.join(OUT, 'train_backward_report.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
