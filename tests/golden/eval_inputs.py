"""Seeded synthetic inputs of the fixtures (shared by make_golden.py and the tests): Redwood-format ground-truth
scenes, perturbed estimates, ModelNet-style batches, loss inputs, 3DMatch-layout pair files, sequences for the
padding helpers and the clouds of the C++ pre-processing cross-check."""
import os
import pickle

import numpy as np


def _rot(rng, max_deg):
    axis = rng.normal(size=3); axis /= np.linalg.norm(axis)
    a = np.deg2rad(rng.uniform(0, max_deg))
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def _pose(rng, max_deg, max_t):
    T = np.eye(4)
    T[:3, :3] = _rot(rng, max_deg)
    T[:3, 3] = rng.uniform(-max_t, max_t, size=3)
    return T


SCENES = ['scene-a', 'scene-b', 'scene-c']


def make_scenes(seed=123):
    """-> {scene: dict(n_frag, pairs [(i,j)], gt (n,4,4), info (n,6,6), est [(src, tgt, pose44)])}.
    Estimated pairs are a subset of the ground-truth pairs (the reference benchmark requires it); consecutive
    pairs (j - i == 1) are present and must be ignored by the recall."""
    rng = np.random.default_rng(seed)
    out = {}
    for s, scene in enumerate(SCENES):
        n_frag = 12 + 5 * s
        pairs = [(i, j) for i in range(n_frag) for j in range(i + 1, n_frag) if rng.random() < 0.35]
        gt = np.stack([_pose(rng, 120, 2.0) for _ in pairs])
        info = []
        for _ in pairs:
            A = rng.normal(size=(6, 6))
            info.append(A @ A.T * 50 + np.eye(6) * rng.uniform(200, 2000))
        est = []
        for (i, j), T in zip(pairs, gt):
            r = rng.random()
            if r < 0.1:
                continue                                            # pair not estimated at all
            noise = _pose(rng, 1.5, 0.02) if r < 0.75 else _pose(rng, 40, 0.8)   # good / failed registration
            est.append((j, i, T @ noise))                           # est.log header is "tgt src": src=j, tgt=i
        out[scene] = dict(n_frag=n_frag, pairs=pairs, gt=gt, info=np.stack(info), est=est)
    return out


def write_gt(scenes, folder):
    for scene, d in scenes.items():
        os.makedirs(os.path.join(folder, scene), exist_ok=True)
        with open(os.path.join(folder, scene, 'gt.log'), 'w') as f:
            for (i, j), T in zip(d['pairs'], d['gt']):
                f.write(f'{i}\t{j}\t{d["n_frag"]}\n')
                for r in range(4):
                    f.write('\t'.join('{0:.12e}'.format(v) for v in T[r]) + '\n')
        with open(os.path.join(folder, scene, 'gt.info'), 'w') as f:
            for (i, j), M in zip(d['pairs'], d['info']):
                f.write(f'{i}\t{j}\t{d["n_frag"]}\n')
                for r in range(6):
                    f.write('\t'.join('{0:.12e}'.format(v) for v in M[r]) + '\n')


def modelnet_batch(seed=7, B=5, N=64):
    import torch
    rng = np.random.default_rng(seed)
    raw = rng.uniform(-1, 1, size=(B, N, 3))
    gt = np.stack([_pose(rng, 45, 0.5)[:3] for _ in range(B)])
    pred = np.stack([(np.vstack([g, [0, 0, 0, 1]]) @ _pose(rng, 3, 0.03))[:3] for g in gt])
    src = raw + rng.normal(scale=0.01, size=raw.shape)
    ref = np.einsum('bij,bnj->bni', gt[:, :, :3], raw) + gt[:, None, :, 3] + rng.normal(scale=0.01, size=raw.shape)
    t = lambda a: torch.from_numpy(a.astype(np.float32))
    return dict(points_src=t(src), points_ref=t(ref), points_raw=t(np.einsum('bij,bnj->bni', gt[:, :, :3], raw) + gt[:, None, :, 3]),
                transform_gt=t(gt)), t(pred)


def pose_batches(seed=9, n_batches=3, L=6, B=4):
    """Per batch: pred['pose'] (L,B,3,4) and gt pose (B,3,4) for compute_metrics / aggregate_metrics."""
    import torch
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_batches):
        gt = np.stack([_pose(rng, 60, 1.0)[:3] for _ in range(B)])
        pred = np.stack([[(np.vstack([g, [0, 0, 0, 1]]) @ _pose(rng, 25.0 / (l + 1), 0.3 / (l + 1)))[:3] for g in gt]
                         for l in range(L)])
        out.append((torch.from_numpy(pred.astype(np.float32)), torch.from_numpy(gt.astype(np.float32))))
    return out


def loss_state_dict(sd, seed=31):
    """The benchmark state_dicts initialise the InfoNCE matrices to identity; use a seeded dense W so that the
    symmetrisation (triu + triu^T) matters."""
    import torch
    rng = np.random.default_rng(seed)
    sd = dict(sd)
    for k in ('feature_criterion.W', 'feature_criterion_un.W'):
        sd[k] = torch.from_numpy((rng.normal(size=tuple(sd[k].shape)) * 0.1).astype(np.float32))
    return sd


def loss_inputs(pairs, src_lens, tgt_lens, seed=33):
    """Ground-truth pose (3,4) per pair from the generator + seeded level-0 overlap masks."""
    import torch
    rng = np.random.default_rng(seed)
    pose = np.stack([np.asarray(p['pose'], dtype=np.float32)[:3] for p in pairs])
    return {'pose': torch.from_numpy(pose),
            'src_overlap': [torch.from_numpy(rng.random(n) < 0.6) for n in src_lens],
            'tgt_overlap': [torch.from_numpy(rng.random(n) < 0.5) for n in tgt_lens]}


def grad_sample_index(name, numel, k=32):
    """Deterministic sample positions of a parameter's gradient (shared by make_golden.py:grad_fixture and tests/test_oracle_grad.py)."""
    import zlib
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    return np.sort(rng.choice(numel, size=min(k, numel), replace=False))


def write_pair_files(folder, n_pairs=11, seed=0):
    """A small dataset in the 3DMatch layout: `<folder>/test/scene/cloud_bin_<i>.pth` (float64 ndarrays, like the
    real files) and `<folder>/info.pkl`; returns the info dict."""
    import torch
    rng = np.random.default_rng(seed)
    infos = dict(rot=[], trans=[], src=[], tgt=[], overlap=[])
    os.makedirs(os.path.join(folder, 'test', 'scene'), exist_ok=True)
    for i in range(n_pairs + 1):
        pts = rng.normal(size=(int(rng.integers(50, 400)), 3))
        torch.save(pts, os.path.join(folder, 'test', 'scene', f'cloud_bin_{i}.pth'))
    for i in range(n_pairs):
        q, _ = np.linalg.qr(rng.normal(size=(3, 3)))
        infos['rot'].append(q); infos['trans'].append(rng.normal(size=(3, 1)))
        infos['src'].append(f'test/scene/cloud_bin_{i + 1}.pth'); infos['tgt'].append(f'test/scene/cloud_bin_{i}.pth')
        infos['overlap'].append(float(rng.uniform(0.1, 0.9)))
    with open(os.path.join(folder, 'info.pkl'), 'wb') as f:
        pickle.dump(infos, f)
    return infos


def seq_inputs(seed=2):
    """Ragged (N, 5) sequences for pad_sequence / unpad_sequences / split_src_tgt, and a padded (6, 11, 4, 5) stack."""
    import torch
    rng = np.random.default_rng(seed)
    seqs = [torch.from_numpy(rng.normal(size=(n, 5)).astype(np.float32)) for n in (7, 3, 11, 1)]
    six = torch.from_numpy(rng.normal(size=(6, 11, 4, 5)).astype(np.float32))
    return seqs, six


def refcpp_inputs(seed=9):
    """Two clouds (400 + 500 points) for the radius-search / grid-subsampling cross-check of the C++ core."""
    rng = np.random.default_rng(seed)
    pts = rng.uniform(-0.5, 0.5, size=(900, 3)).astype(np.float32)
    return pts, np.array([400, 500])
