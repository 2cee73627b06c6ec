"""Golden vectors for the ground-truth match computation (SURVEY.md 8 f-2): the reference's OWN
compute_gt_matches_of_image_pair (helpers.py:121-203), imported unmodified through oracle/ref_shim.py (helpers.py pulls
in coloredlogs and the two-view pose files), run on seeded synthetic scenes -> tests/golden/gt_matches_*.npz.
TEST INFRASTRUCTURE ONLY; needs /root/reference, runs in the authoring container.

Scene: a depth map for view 0 (smooth surface 1.5-4 m with holes of zero depth), keypoints of view 0 at integer
pixels, a second camera (rotation <= 12 deg, baseline <= 0.4 m); a share of the view-1 keypoints are the rounded
reprojections of view-0 keypoints (true matches, depth map 1 consistent at those pixels), the rest are random.
Besides the outputs the fixture stores, per keypoint, the margin between the best and second-best reprojection
error in the reference's float32 error matrix, so the GPU test can require exact indices wherever the decision
is not a rounding-level tie.  The stored depth maps keep only the pixels the computation reads (depth0 at the
truncated view-0 keypoints, depth1 at the truncated view-1 keypoints, helpers.py:125-128); every other pixel is
zero, which leaves the outputs unchanged and keeps the fixtures small."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_shim  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')


def rot(axis, deg):
    a = np.asarray(axis, float); a /= np.linalg.norm(a)
    t = np.deg2rad(deg)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(t) * K + (1 - np.cos(t)) * K @ K


def scene(seed, bs, n, H, W, hole_frac, match_frac):
    rng = np.random.default_rng(seed)
    f = 0.9 * W
    K = np.eye(4, dtype=np.float32); K[0, 0] = K[1, 1] = f; K[0, 2] = (W - 1) / 2; K[1, 2] = (H - 1) / 2
    out = {k: [] for k in ('kpts0', 'kpts1', 'K0', 'K1', 'T', 'depth0', 'depth1')}
    yy, xx = np.mgrid[0:H, 0:W]
    for b in range(bs):
        a, c = rng.uniform(0.5, 1.5, 2)
        depth0 = (2.75 + 1.2 * np.sin(a * xx / W * 3.0) * np.cos(c * yy / H * 2.0)).astype(np.float32)
        holes = rng.random((H, W)) < hole_frac
        depth0[holes] = 0.0
        R = rot(rng.normal(size=3), rng.uniform(2, 12)); t = rng.normal(size=3); t *= rng.uniform(0.05, 0.4) / np.linalg.norm(t)
        T = np.eye(4); T[:3, :3] = R; T[:3, 3] = t
        k0 = np.stack([rng.integers(0, W, n), rng.integers(0, H, n)], 1).astype(np.float32)
        d = depth0[k0[:, 1].astype(int), k0[:, 0].astype(int)]
        X = np.linalg.inv(K[:3, :3].astype(float)) @ np.stack([k0[:, 0] * d, k0[:, 1] * d, d])
        Y = R @ X + t[:, None]
        p = K[:3, :3].astype(float) @ Y
        uv = p[:2] / np.where(np.abs(p[2]) > 1e-9, p[2], 1.0)
        depth1 = rng.uniform(1.5, 4.0, (H, W)).astype(np.float32)
        depth1[rng.random((H, W)) < hole_frac] = 0.0
        k1 = np.stack([rng.integers(0, W, n), rng.integers(0, H, n)], 1).astype(np.float32)
        order = rng.permutation(n)
        n_true = 0
        for i in order:
            if n_true >= int(match_frac * n):
                break
            u, v = np.rint(uv[0, i]), np.rint(uv[1, i])
            if d[i] > 0 and Y[2, i] > 0.1 and 0 <= u < W and 0 <= v < H:
                j = order[n_true]
                k1[j] = (u, v)
                depth1[int(v), int(u)] = Y[2, i] * rng.uniform(0.97, 1.03)
                n_true += 1
        # a few sub-pixel offsets so that .long() truncation is exercised
        k0 += rng.uniform(0, 0.9, k0.shape).astype(np.float32) * (rng.random((n, 1)) < 0.3)
        k1 += rng.uniform(0, 0.9, k1.shape).astype(np.float32) * (rng.random((n, 1)) < 0.3)
        for key, val in (('kpts0', k0), ('kpts1', k1), ('K0', K), ('K1', K), ('T', T.astype(np.float32)),
                         ('depth0', depth0), ('depth1', depth1)):
            out[key].append(val)
    return {k: np.stack(v) for k, v in out.items()}


def keep_read_pixels(z):
    """z with depth0 / depth1 zero everywhere except at the pixels of the truncated keypoints of their view."""
    z = dict(z)
    for v in (0, 1):
        k = z['kpts%d' % v].astype(np.int64)
        bi = np.arange(k.shape[0])[:, None]
        d = np.zeros_like(z['depth%d' % v])
        d[bi, k[..., 1], k[..., 0]] = z['depth%d' % v][bi, k[..., 1], k[..., 0]]
        z['depth%d' % v] = d
    return z


def margins(helpers, z):
    """best / second-best error per row and column of the reference's float32 error matrix (recomputed with its code)."""
    t = {k: torch.from_numpy(v) for k, v in z.items()}
    bs, n, _ = t['kpts0'].shape
    bi = torch.arange(bs).unsqueeze(-1).expand(bs, n)
    k0, k1 = t['kpts0'].long(), t['kpts1'].long()
    d0 = t['depth0'][bi, k0[..., 1], k0[..., 0]].unsqueeze(-1)
    d1 = t['depth1'][bi, k1[..., 1], k1[..., 0]].unsqueeze(-1)
    K0, K1, T = t['K0'].unsqueeze(1), t['K1'].unsqueeze(1), t['T'].unsqueeze(1)
    _, k0to1 = helpers.transform_kpts(k0, d0, K0, K1, T)
    _, k1to0 = helpers.transform_kpts(k1, d1, K1, K0, torch.linalg.inv(T))
    e = torch.sqrt(((k1to0.unsqueeze(2).expand(bs, n, n, 2) - k0.unsqueeze(1)) ** 2).sum(3)).transpose(1, 2)
    e = e + torch.sqrt(((k0to1.unsqueeze(2).expand(bs, n, n, 2) - k1.unsqueeze(1)) ** 2).sum(3))
    e = e / 2.0
    r2 = torch.topk(e, 2, dim=2, largest=False).values
    c2 = torch.topk(e, 2, dim=1, largest=False).values
    return (r2[..., 1] - r2[..., 0]).numpy(), (c2[:, 1] - c2[:, 0]).numpy(), r2[..., 0].numpy(), c2[:, 0].numpy()


def main():
    ref_shim.load()
    import helpers                       # the reference's helpers.py, unmodified
    assert helpers.__file__.startswith('/root/reference')
    report = {}
    for name, (seed, bs, n, H, W, holes, frac, e_match, e_unmatch) in {
            'small': (1, 2, 96, 60, 80, 0.05, 0.5, 5.0, 15.0),
            'scannet_like': (2, 3, 400, 240, 320, 0.08, 0.45, 5.0, 15.0),
            'dense_1024': (3, 2, 1024, 240, 320, 0.02, 0.6, 3.0, 10.0),
            'no_matches': (4, 1, 64, 48, 64, 0.6, 0.0, 5.0, 15.0)}.items():
        z = keep_read_pixels(scene(seed, bs, n, H, W, holes, frac))
        t = {k: torch.from_numpy(v) for k, v in z.items()}
        idx, w = helpers.compute_gt_matches_of_image_pair(t['kpts0'], t['kpts1'], t['K0'], t['K1'], t['T'], t['depth0'],
                                                          t['depth1'], e_match, e_unmatch)
        rm, cm, rmin, cmin = margins(helpers, z)
        np.savez_compressed(os.path.join(OUT, 'gt_matches_%s.npz' % name), **z, indices=idx.numpy(), weights=w.numpy(),
                            row_margin=rm, col_margin=cm, row_min=rmin, col_min=cmin,
                            thresholds=np.array([e_match, e_unmatch], np.float32))
        nm = int((idx[:, 0, :-1] >= 0).sum())
        report[name] = {'bs': bs, 'n': n, 'matches': nm, 'dropped': int((w[:, :, :-1] == 0).sum()),
                        'rows_with_margin_below_1e-4': int((rm < 1e-4).sum() + (cm < 1e-4).sum())}
        print(name, report[name])
    import json
    json.dump(report, open(os.path.join(OUT, 'gt_matches_report.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
