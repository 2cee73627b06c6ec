"""Golden vectors for the TRAIN-MODE forward of the matcher (SURVEY.md 8 a8 / a13 / f-2): the unmodified reference
MultiViewMatcher in .train() with config['full_output'] = True -- batch-statistics BatchNorm in the keypoint encoder,
every GNN layer and the confidence head, stacked views, combined cross attention -- on seeded inputs and weights, in
fp32 and (yardstick) fp64 -> tests/golden/train_forward_*.npz, including the BatchNorm running statistics after the
call.  TEST INFRASTRUCTURE ONLY (needs /root/reference); the GPU test rebuilds inputs and weights from the seeds."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = '/root/reference'
OUT = os.path.join(ROOT, 'tests', 'golden')

CASES = [dict(name='mv3_64', multi=True, views=3, kpts=64, batch=2, layers=['self', 'cross', 'cross', 'self', 'cross'], wseed=41, iseed=51, gain=10.0),
         dict(name='pair_128', multi=False, views=2, kpts=128, batch=2, layers=['self', 'cross'] * 2, wseed=42, iseed=52, gain=10.0)]
STATS = ['kenc.encoder.1.running_mean', 'kenc.encoder.10.running_var', 'gnn.layers.0.mlp.1.running_mean',
         'gnn.layers.3.mlp.1.running_var', 'conf_mlp.layers_f.1.running_mean', 'conf_mlp.layers_c.4.running_var',
         'conf_mlp.layers_f.4.num_batches_tracked']


def build(case):
    from oracle.weights import make_state_dict, make_correlated_view_inputs
    sd = make_state_dict(len(case['layers']), seed=case['wseed'], final_proj_gain=case['gain'])
    data = make_correlated_view_inputs(case['iseed'], case['views'], case['kpts'], batch=case['batch'])
    return sd, data


def main():
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from models.models.multi_view_matcher import MultiViewMatcher
    torch.set_num_threads(8)
    report = {}
    for case in CASES:
        sd, data_np = build(case)
        out = {}
        for dtype, tag in ((torch.float32, 'f32'), (torch.float64, 'f64')):
            torch.manual_seed(0)
            model = MultiViewMatcher({'multi_frame_matching': case['multi'], 'GNN_layers': case['layers'], 'conf_mlp': True,
                                      'full_output': True})
            model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
            model = model.to(dtype).train()
            data = {k: (torch.from_numpy(v).to(dtype) if isinstance(v, np.ndarray) and v.dtype.kind == 'f' else v)
                    for k, v in data_np.items()}
            res = model(data)
            st = model.state_dict()
            for k, v in res.items():
                if v is not None:
                    out['%s__%s' % (tag, k)] = v.detach().numpy()
            for k in STATS:
                if k in st:
                    out['%s__stat__%s' % (tag, k)] = st[k].detach().numpy()
        noise = max(float(np.abs(out['f32__' + k[5:]].astype(np.float64) - v).max()) for k, v in out.items()
                    if k.startswith('f64__scores_'))  # noqa
        report[case['name']] = {'max_abs_ref32_vs_ref64_scores': noise}
        print(case['name'], report[case['name']], sorted(k for k in out if k.startswith('f32__') and 'stat' not in k)[:6])
        np.savez_compressed(os.path.join(OUT, 'train_forward_%s.npz' % case['name']), meta=json.dumps(case), **out)
    json.dump(report, open(os.path.join(OUT, 'train_forward_report.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
