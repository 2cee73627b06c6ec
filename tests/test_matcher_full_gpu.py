"""Full-size parity at the BASELINE.json configurations: the CUDA matcher against fixtures produced by the
UNMODIFIED reference at 5 x 1024 kpts x 28 layers (cfg3, the bench workload), 2 x 1024 x 18 layers (cfg2, batch 2)
and 2 x 2048 x 18 layers (cfg4) -- oracle/make_golden_full.py.  Per pair the fixture holds the matches, matching
scores and confidences in full, 25 rows of the coupling matrix (9 for cfg3) and float64 checksums of the whole matrix, plus
the same rows from the reference's own double-precision run, whose distance to the fp32 run (`noise`) is the
yardstick for the score tolerance."""
import json
import os

import numpy as np
import pytest
import torch

from tests.util import GOLDEN

pytestmark = pytest.mark.gpu

CASES = ['cfg3_5x1024_28l', 'cfg2_2x1024_18l_b2', 'cfg4_2x2048_18l']
TAU = 2e-3


@pytest.mark.parametrize('name', CASES)
def test_full_size_matcher_vs_reference(name):
    from oracle.make_golden_full import build, input_digest
    from e2e_multi_view_matching_b200.models.multi_view_matcher import MultiViewMatcher
    z = np.load(os.path.join(GOLDEN, 'matcher_full_%s.npz' % name))
    meta = json.loads(str(z['meta']))
    noise = json.load(open(os.path.join(GOLDEN, 'matcher_full_report.json')))[name]['noise']
    sd, data = build(meta)
    assert input_digest(sd, data) == meta['digest'], 'seeded inputs differ from the ones the reference saw'
    model = MultiViewMatcher({'multi_frame_matching': meta['multi'], 'GNN_layers': meta['layers'], 'conf_mlp': True}).eval()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, strict=True)
    model = model.cuda()
    keys = [k for k in data if k.startswith(('keypoints', 'descriptors', 'scores'))]
    d = {k: torch.from_numpy(data[k]).cuda() for k in keys}
    d.update({k: torch.empty(data[k].shape, device='meta') for k in data if k.startswith('image')})
    d['ids'] = data['ids']
    out = model(d)
    torch.cuda.synchronize()
    T = meta['views']
    worst32 = worst64 = 0.0
    rows_total = rows_stable = mism0 = 0
    for b in range(T):
        for a in range(b):
            sk = 'scores_%d_%d' % (a, b)
            Z = out[sk].double()
            Zc = Z.cpu().numpy()
            n_ab = noise[sk]['max_abs_ref32_vs_ref64']
            # ---- sampled rows of the coupling matrix ----
            rows = z['rows_' + sk]
            got = Zc[:, rows, :]
            e32 = np.abs(got - z['sample_' + sk])
            e64 = np.abs(got - z['sample64_' + sk])
            worst32, worst64 = max(worst32, float(e32.max())), max(worst64, float(e64.max()))
            # as close to the reference's double-precision run as the reference's own fp32 run is (x1.5), and
            # within two fp32-class noises of the fp32 run
            assert e64.max() <= max(1e-4, 1.5 * n_ab) + 3e-5 * np.abs(got).max(), (sk, float(e64.max()), n_ab)
            assert (e32 <= max(3e-4, 2.5 * n_ab) + 3e-5 * np.abs(got)).all(), (sk, float(e32.max()), n_ab)
            # ---- whole-matrix checksums: mean signed error and mean square ----
            chk = z['chk_' + sk]
            numel = Zc[0].size
            # (the split-operand arithmetic carries a systematic +1e-5 .. +1e-4 bias, profiles/r02_score_ab.txt: this is a
            # gross-error check -- a dropped row or column shifts the mean by far more)
            assert np.abs(Zc.sum((1, 2)) - chk[:, 0]).max() / numel < 2e-4, sk
            assert np.abs((Zc * Zc).sum((1, 2)) - chk[:, 1]).max() / np.abs(chk[:, 1]).max() < 1e-4, sk
            # ---- matches: exact on every row whose top-2 margin (ours) exceeds tau ----
            inner = Z[:, :-1, :-1]
            top2 = torch.topk(inner, 2, dim=2).values
            m_row = (top2[..., 0] - top2[..., 1]).cpu().numpy()
            top2c = torch.topk(inner, 2, dim=1).values
            m_col = (top2c[:, 0] - top2c[:, 1]).cpu().numpy()
            for vid, margin, other in ((a, m_row, m_col), (b, m_col, m_row)):
                mk = 'matches%d_%d_%d' % (vid, a, b)
                g, r = out[mk].cpu().numpy(), z[mk].astype(np.int64)
                assert g.dtype == np.int64 and g.shape == r.shape
                # a match decision involves the row's arg-max and the mutual check through the column's arg-max
                j = np.where(r >= 0, r, 0)
                stable = (margin > TAU) & ((r < 0) | (np.take_along_axis(other, j, 1) > TAU))
                unmatched_unstable = (r < 0) & (margin > TAU)     # a -1 may hinge on the partner's near-tie
                stable &= ~unmatched_unstable | (g == r)
                assert np.array_equal(g[stable], r[stable]), (mk, int((g[stable] != r[stable]).sum()))
                rows_total += g.size
                rows_stable += int(stable.sum())
                mism0 += int((g != r).sum())
                same = g == r
                ms = 'matching_scores%d_%d_%d' % (vid, a, b)
                np.testing.assert_allclose(out[ms].cpu().numpy()[same], z[ms][same], rtol=2e-3, atol=1e-6)
            ck = 'conf_scores_%d_%d' % (a, b)
            same = out['matches%d_%d_%d' % (a, a, b)].cpu().numpy() == z['matches%d_%d_%d' % (a, a, b)]
            cerr = np.abs(out[ck].cpu().numpy()[..., 0] - z[ck][..., 0])[same]
            assert cerr.max() < 3e-4, (ck, float(cerr.max()))
    frac = rows_stable / rows_total
    print('%s: max |cuda - ref32| %.2e, |cuda - ref64| %.2e on the sampled rows; %d of %d keypoints compared exactly '
          '(%.2f %%); mismatches at margin 0: %d' % (name, worst32, worst64, rows_stable, rows_total, 100 * frac, mism0))
    assert frac >= 0.9, frac
    assert mism0 <= 0.005 * rows_total, mism0
