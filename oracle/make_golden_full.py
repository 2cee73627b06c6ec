"""Full-size reference fixtures for the BASELINE.json configurations (cfg2 / cfg3 / cfg4).

Run in the authoring container only (needs /root/reference):
    python -m oracle.make_golden_full [case ...]
The UNMODIFIED reference ``MultiViewMatcher`` is run on the seeded inputs bench.py uses, at the sizes the
headline numbers are quoted on: 5 views x 1024 keypoints x 28 layers (cfg3), 2 x 1024 x 18 layers (cfg2) and
2 x 2048 x 18 layers (cfg4).  A coupling matrix is 4.2 MB (16.8 MB at 2048), so the fixture keeps, per pair:
the match indices and scores and the confidences in full, N_ROWS sampled rows of the coupling matrix (seeded
row ids, plus the dustbin row; cfg3, with ten pairs, keeps the first `n_rows` of the drawn rows so that the fixture
stays under 1 MB), and float64 checksums of the whole matrix (sum, sum of squares, sum of the
row arg-max indices).  The reference is also run in DOUBLE precision (``model.double()``): the distance of
its shipped fp32 run to its own fp64 run is the arithmetic noise of the reference, stored per pair
(``noise_*``) and used by the GPU tests as the yardstick for the tolerance on the log-scores.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np
import torch

REF = '/root/reference'
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
N_ROWS = 24

CASES = {
    # the bench workload (bench.py: weights seed 0 / gain 12, tuples 1000 + k)
    'cfg3_5x1024_28l': dict(views=5, kpts=1024, layers=(['self'] + ['cross'] * 3) * 7, multi=True, batch=1,
                            wseed=0, gain=12.0, iseed=1000, width=640, height=480, f=577.87, n_rows=8),
    'cfg2_2x1024_18l_b2': dict(views=2, kpts=1024, layers=['self', 'cross'] * 9, multi=False, batch=2,
                               wseed=0, gain=12.0, iseed=2000, width=720, height=537, f=650.0),
    'cfg4_2x2048_18l': dict(views=2, kpts=2048, layers=['self', 'cross'] * 9, multi=False, batch=1,
                            wseed=0, gain=12.0, iseed=4000, width=1600, height=1200, f=1400.0),
}


def build(case):
    from e2e_multi_view_matching_b200.synthetic import make_state_dict, make_scene_tuple_inputs
    sd = make_state_dict(len(case['layers']), seed=case['wseed'], final_proj_gain=case['gain'])
    data = make_scene_tuple_inputs(case['iseed'], case['views'], case['kpts'], batch=case['batch'],
                                   width=case['width'], height=case['height'], f=case['f'])
    return sd, data


def input_digest(sd, data):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(np.ascontiguousarray(sd[k]).tobytes())
    for k in sorted(data):
        if isinstance(data[k], np.ndarray) and k.startswith(('keypoints', 'scores', 'descriptors')):
            h.update(np.ascontiguousarray(data[k]).tobytes())
    return h.hexdigest()


def run_reference(case, sd, data, double):
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from models.models.multi_view_matcher import MultiViewMatcher  # the unmodified reference
    model = MultiViewMatcher({'multi_frame_matching': case['multi'], 'GNN_layers': case['layers'], 'conf_mlp': True}).eval()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    dt = torch.float64 if double else torch.float32
    if double:
        model = model.double()
    keys = [k for k in data if k.startswith(('keypoints', 'descriptors', 'scores', 'image'))]
    d = {k: torch.from_numpy(data[k]).to(dt) for k in keys}
    d['ids'] = data['ids']
    with torch.no_grad():
        out = model(d)
    return {k: v.numpy() for k, v in out.items() if v is not None}


def summarize(case, ref, ref64, seed):
    rng = np.random.default_rng(seed)
    out, noise = {}, {}
    for k, v in ref.items():
        if k.startswith('matches'):
            assert v.max() < 32768
            out[k] = v.astype(np.int16)
        elif k.startswith('matching_scores') or k.startswith('conf_scores'):
            out[k] = v.astype(np.float32)
        elif k.startswith('scores_'):
            B, m1, n1 = v.shape
            drawn = rng.choice(m1 - 1, N_ROWS, replace=False)[:case.get('n_rows', N_ROWS)]
            rows = np.sort(np.concatenate([drawn, [m1 - 1]]))
            out['rows_' + k] = rows.astype(np.int32)
            out['sample_' + k] = v[:, rows, :].astype(np.float32)
            out['sample64_' + k] = ref64[k][:, rows, :].astype(np.float32)
            z = v.astype(np.float64)
            out['chk_' + k] = np.stack([z.sum((1, 2)), (z * z).sum((1, 2)),
                                        v[:, :-1, :-1].argmax(2).astype(np.float64).sum(1)], 1)
            d = np.abs(z - ref64[k])
            inner = np.sort(v[:, :-1, :-1], axis=2)
            margin = inner[..., -1] - inner[..., -2]
            noise[k] = {'max_abs_ref32_vs_ref64': float(d.max()), 'p999': float(np.quantile(d, 0.999)),
                        'rel_excess_1e-5': float((d - 1e-5 * np.abs(ref64[k])).max()),
                        'frac_rows_margin_gt_2e-3': float((margin > 2e-3).mean()),
                        'min_margin': float(margin.min()),
                        'match_flips_ref32_vs_ref64': int((v[:, :-1, :-1].argmax(2) != ref64[k][:, :-1, :-1].argmax(2)).sum())}
    return out, noise


def main():
    torch.set_num_threads(os.cpu_count())
    names = sys.argv[1:] or list(CASES)
    os.makedirs(OUT, exist_ok=True)
    rep_path = os.path.join(OUT, 'matcher_full_report.json')
    report = json.load(open(rep_path)) if os.path.exists(rep_path) else {}
    for name in names:
        case = CASES[name]
        sd, data = build(case)
        t0 = time.time()
        ref = run_reference(case, sd, data, double=False)
        t1 = time.time()
        ref64 = run_reference(case, sd, data, double=True)
        t2 = time.time()
        out, noise = summarize(case, ref, ref64, seed=case['iseed'] + 99)
        meta = dict(case)
        meta['digest'] = input_digest(sd, data)
        np.savez_compressed(os.path.join(OUT, 'matcher_full_%s.npz' % name), meta=json.dumps(meta), **out)
        report[name] = {'seconds_fp32': t1 - t0, 'seconds_fp64': t2 - t1, 'noise': noise}
        worst = max(v['max_abs_ref32_vs_ref64'] for v in noise.values())
        print(name, 'ok: reference fp32 %.0fs, fp64 %.0fs; max |ref32 - ref64| on log-scores %.2e; flips %d' %
              (t1 - t0, t2 - t1, worst, sum(v['match_flips_ref32_vs_ref64'] for v in noise.values())), flush=True)
        with open(rep_path, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
