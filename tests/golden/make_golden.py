"""Generate the committed golden fixtures by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    make -C oracle ref                      # refcpp_fixture binds the reference's C++ core (oracle/_ref)
    python tests/golden/make_golden.py      # every fixture; `... make_golden.py data`: data.npz + refcpp.npz

Every fixture is produced by the reference's own modules, imported through
oracle/ref_bridge.py (third-party stubs per SURVEY.md Appendix A), on seeded
inputs from regtr_b200.synthetic and seeded weights from regtr_b200.weights.
Tests regenerate the same inputs/weights from the seeds and compare:
  * `-m "not gpu"`: oracle (oracle/regtr_oracle.py) vs these fixtures  -> pins the oracle;
  * `-m gpu`      : CUDA product vs these fixtures and vs the oracle.
Fixtures are kept small: full integer metadata, but only a strided sample of the
large float tensors plus their fp64 checksums.
"""
from __future__ import annotations

import hashlib
import os
import re
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import ref_bridge  # noqa: E402
from regtr_b200.config import get_config  # noqa: E402
from regtr_b200.synthetic import make_3dmatch_pair, make_modelnet_pair  # noqa: E402
from regtr_b200.weights import random_state_dict  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

# (fixture name, config, weight seed, list of pair makers[, config overrides])
FORWARD_CASES = {
    'fwd_modelnet_b1': ('modelnet', 11, [lambda: make_modelnet_pair(1000)]),
    'fwd_3dmatch_small_b1': ('3dmatch', 12, [lambda: make_3dmatch_pair(2000, 3000)]),
    'fwd_3dmatch_small_b2': ('3dmatch', 13, [lambda: make_3dmatch_pair(2001, 2500),
                                             lambda: make_3dmatch_pair(2002, 4000)]),
    # alternative config branches (SURVEY.md 8f N4); float outputs only (the pyramid is the modelnet one)
    'var_modelnet_attndec_b1': ('modelnet', 14, [lambda: make_modelnet_pair(1001)],
                                dict(direct_regress_coor=False)),
    'var_modelnet_postnorm_b1': ('modelnet', 15, [lambda: make_modelnet_pair(1002)], dict(pre_norm=False)),
    'var_modelnet_learnedpe_attndec_b2': ('modelnet', 16, [lambda: make_modelnet_pair(1003),
                                                           lambda: make_modelnet_pair(1004)],
                                          dict(pos_emb_type='learned', direct_regress_coor=False)),
}


# The reference's own sample inputs (src/demo.py:154-192 runs exactly these files): real 3DMatch fragments sit
# on a 6 mm sensor lattice where voxel-boundary hits are common (SURVEY.md 7-H1), which no synthetic cloud
# exercises.  The clouds are copied (fp32: the files hold fp32 values stored as fp64, the demo casts with
# .float()) into tests/golden/real/ as INPUT fixtures; outputs come from the unmodified reference.
REF_DATA = '/root/reference/data'
REAL_CASES = {
    'real_3dmatch_redkitchen_0_5': ('3dmatch', 31, 'indoor/test/7-scenes-redkitchen/cloud_bin_0.pth',
                                    'indoor/test/7-scenes-redkitchen/cloud_bin_5.pth'),
    'real_3dmatch_sun3d_home_38_41': ('3dmatch', 32,
                                      'indoor/test/sun3d-home_at-home_at_scan1_2013_jan_1/cloud_bin_38.pth',
                                      'indoor/test/sun3d-home_at-home_at_scan1_2013_jan_1/cloud_bin_41.pth'),
    'real_3dmatch_sun3d_hotel3_8_15': ('3dmatch', 33, 'indoor/test/sun3d-hotel_umd-maryland_hotel3/cloud_bin_8.pth',
                                       'indoor/test/sun3d-hotel_umd-maryland_hotel3/cloud_bin_15.pth'),
    'real_modelnet_2': ('modelnet', 34, 'modelnet_demo_data/modelnet_test_2_0.ply',
                        'modelnet_demo_data/modelnet_test_2_1.ply'),
    'real_modelnet_630': ('modelnet', 35, 'modelnet_demo_data/modelnet_test_630_0.ply',
                          'modelnet_demo_data/modelnet_test_630_1.ply'),
}


def _np(t):
    return t.detach().cpu().numpy()


def load_point_cloud(fname):
    """demo.py:140-151 without open3d: .pth = pickled ndarray, .ply = binary little-endian xyz doubles."""
    if fname.endswith('.pth'):
        data = torch.load(fname, weights_only=False)
    else:
        raw = open(fname, 'rb').read()
        head, body = raw.split(b'end_header\n', 1)
        assert b'format binary_little_endian' in head and b'property double x' in head
        n = int(re.search(rb'element vertex (\d+)', head).group(1))
        data = np.frombuffer(body, dtype='<f8', count=3 * n).reshape(n, 3)
    return np.asarray(data)[:, :3]


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def real_fixture(name):
    """Forward of the unmodified reference on one of its own sample pairs.  Keeps the fixture small: exact
    level sizes and level >= 1 points, SHA-256 (+ a strided row sample) of every int64 index array, strided
    feature rows with fp64 checksums, correspondences, overlap logits and poses in full."""
    cfg_name, wseed, src_rel, tgt_rel = REAL_CASES[name]
    cfg = get_config(cfg_name)
    sd = random_state_dict(cfg, wseed)
    src = load_point_cloud(os.path.join(REF_DATA, src_rel)).astype(np.float32)   # demo.py:180 `.float()`
    tgt = load_point_cloud(os.path.join(REF_DATA, tgt_rel)).astype(np.float32)
    os.makedirs(os.path.join(OUT, 'real'), exist_ok=True)
    np.savez_compressed(os.path.join(OUT, 'real', name + '_input.npz'), src_xyz=src, tgt_xyz=tgt,
                        src_file=np.array(src_rel), tgt_file=np.array(tgt_rel))
    model = ref_bridge.build_reference_model(cfg, sd)
    out = ref_bridge.reference_forward(model, [src], [tgt])
    meta = out['kpconv_meta']
    step = 13
    fx = {'pose': _np(out['pose']), 'row_step': np.array(step)}
    for lvl in range(len(meta['points'])):
        fx[f'stack_lengths_{lvl}'] = _np(meta['stack_lengths'][lvl]).astype(np.int64)
        for key in ('neighbors', 'pools', 'upsamples'):
            a = _np(meta[key][lvl]).astype(np.int64)
            fx[f'{key}_{lvl}_shape'] = np.array(a.shape, dtype=np.int64)
            fx[f'{key}_{lvl}_sha256'] = sha(a)
            fx[f'{key}_{lvl}_rows'] = a[::97].astype(np.int32)
        if lvl > 0:
            fx[f'points_{lvl}'] = _np(meta['points'][lvl])
    for side in ('src', 'tgt'):
        fx[f'{side}_kp_warped_0'] = _np(out[f'{side}_kp_warped'][0])
        fx[f'{side}_overlap_0'] = _np(out[f'{side}_overlap'][0])
        fu, fc = _np(out[f'{side}_feat_un'][0]), _np(out[f'{side}_feat'][0])
        fx[f'{side}_feat_un_0_rows'] = fu[::step]
        fx[f'{side}_feat_0_rows'] = fc[:, ::step]
        fx[f'{side}_feat_un_0_sum'] = np.array(fu.astype(np.float64).sum())
        fx[f'{side}_feat_0_sum'] = np.array(fc.astype(np.float64).sum())
        fx[f'{side}_feat_un_0_absmax'] = np.array(np.abs(fu).max())
        fx[f'{side}_feat_0_absmax'] = np.array(np.abs(fc).max())
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **fx)
    print(name, [int(fx[f'stack_lengths_{l}'].sum()) for l in range(len(meta['points']))],
          'pose[-1]', fx['pose'][-1, 0, 0])


def benchmark_fixture():
    """Category-b fixtures for the end-to-end benchmark test (SURVEY.md 8f N1 + N2): the `gt.log` / `gt.info`
    entries (src/datasets/3dmatch/benchmarks/3DMatch/<scene>/) and the `test_3DMatch_info.pkl` rows
    (src/datasets/3dmatch/) of the two shipped sample pairs that belong to the 3DMatch benchmark."""
    import json
    import pickle
    ref = '/root/reference/src/datasets/3dmatch'
    info = pickle.load(open(os.path.join(ref, 'test_3DMatch_info.pkl'), 'rb'))
    want = {('7-scenes-redkitchen', 5, 0): 'real_3dmatch_redkitchen_0_5',
            ('sun3d-hotel_umd-maryland_hotel3', 15, 8): 'real_3dmatch_sun3d_hotel3_8_15'}
    rows = []
    for i, (sp, tp) in enumerate(zip(info['src'], info['tgt'])):
        scene = sp.split('/')[1]
        key = (scene, int(sp.split('_')[-1][:-4]), int(tp.split('_')[-1][:-4]))
        if key in want:
            rows.append(dict(src=sp, tgt=tp, rot=np.asarray(info['rot'][i]).tolist(), trans=np.asarray(info['trans'][i]).tolist(),
                             overlap=float(info['overlap'][i]), fixture=want[key]))
    out_dir = os.path.join(OUT, 'real', 'benchmarks', '3DMatch')
    for scene, si, ti in want:
        os.makedirs(os.path.join(out_dir, scene), exist_ok=True)
        for fname, n_rows in (('gt.log', 4), ('gt.info', 6)):
            lines = open(os.path.join(ref, 'benchmarks', '3DMatch', scene, fname)).read().split('\n')
            for k, ln in enumerate(lines):
                f = ln.split()
                if len(f) == 3 and int(f[0]) == ti and int(f[1]) == si:
                    open(os.path.join(out_dir, scene, fname), 'w').write('\n'.join(lines[k:k + 1 + n_rows]) + '\n')
                    break
            else:
                raise RuntimeError((scene, fname))
    json.dump(rows, open(os.path.join(OUT, 'real', 'test_3DMatch_info_rows.json'), 'w'), indent=1)
    print('benchmark fixture', [r['src'] for r in rows])


def forward_fixture(name):
    cfg_name, wseed, makers, *rest = FORWARD_CASES[name]
    variant = bool(rest)
    cfg = get_config(cfg_name, **(rest[0] if rest else {}))
    sd = random_state_dict(cfg, wseed)
    model = ref_bridge.build_reference_model(cfg, sd)
    pairs = [mk() for mk in makers]
    out = ref_bridge.reference_forward(model, [p['src_xyz'] for p in pairs], [p['tgt_xyz'] for p in pairs])
    meta = out['kpconv_meta']
    step = 29 if variant else 7
    fx = {'pose': _np(out['pose']), 'row_step': np.array(step)}
    for lvl in range(len(meta['points'])):
        fx[f'stack_lengths_{lvl}'] = _np(meta['stack_lengths'][lvl]).astype(np.int64)
        if variant:            # index parity is pinned by the three base cases; keep these fixtures small
            continue
        fx[f'neighbors_{lvl}'] = _np(meta['neighbors'][lvl]).astype(np.int32)
        fx[f'pools_{lvl}'] = _np(meta['pools'][lvl]).astype(np.int32)
        fx[f'upsamples_{lvl}'] = _np(meta['upsamples'][lvl]).astype(np.int32)
        if lvl > 0:
            fx[f'points_{lvl}'] = _np(meta['points'][lvl])
    for b in range(len(pairs)):
        for side in ('src', 'tgt'):
            fx[f'{side}_kp_warped_{b}'] = _np(out[f'{side}_kp_warped'][b])
            fx[f'{side}_overlap_{b}'] = _np(out[f'{side}_overlap'][b])
            fu, fc = _np(out[f'{side}_feat_un'][b]), _np(out[f'{side}_feat'][b])
            fx[f'{side}_feat_un_{b}_rows'] = fu[::step]
            fx[f'{side}_feat_{b}_rows'] = fc[:, ::step]
            fx[f'{side}_feat_un_{b}_sum'] = np.array(fu.astype(np.float64).sum())
            fx[f'{side}_feat_{b}_sum'] = np.array(fc.astype(np.float64).sum())
            fx[f'{side}_feat_un_{b}_absmax'] = np.array(np.abs(fu).max())
            fx[f'{side}_feat_{b}_absmax'] = np.array(np.abs(fc).max())
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **fx)
    print(name, {k: v.shape for k, v in fx.items() if k.startswith(('pose', 'stack'))})


def op_fixtures():
    """Small known-answer vectors for the individual reference ops on the hot path."""
    m = ref_bridge.modules()
    rng = np.random.default_rng(77)
    fx = {}

    # KPConv.forward (kpconv_blocks.py:269-414) incl. shadow neighbours and zero-sum rows
    Nq, Ns, K, Cin, Cout, P = 37, 53, 11, 8, 12, 15
    q = rng.normal(size=(Nq, 3)).astype(np.float32) * 0.1
    s = rng.normal(size=(Ns, 3)).astype(np.float32) * 0.1
    inds = rng.integers(0, Ns + 1, size=(Nq, K)).astype(np.int64)        # Ns == shadow
    inds[3] = Ns                                                          # fully shadow row
    x = rng.normal(size=(Ns, Cin)).astype(np.float32)
    x[5] = -np.abs(x[5])                                                  # row with negative sum
    conv = m.blocks.KPConv(P, 3, Cin, Cout, 0.12, 0.15, fixed_kernel_points='center',
                           KP_influence='linear', aggregation_mode='sum')
    W = rng.normal(size=(P, Cin, Cout)).astype(np.float32) * 0.3
    kp = rng.normal(size=(P, 3)).astype(np.float32) * 0.08
    kp[0] = 0
    with torch.no_grad():
        conv.weights.copy_(torch.from_numpy(W))
        conv.kernel_points.copy_(torch.from_numpy(kp))
        y = conv(torch.from_numpy(q), torch.from_numpy(s), torch.from_numpy(inds), torch.from_numpy(x))
    fx.update(kp_q=q, kp_s=s, kp_inds=inds, kp_x=x, kp_W=W, kp_kp=kp, kp_extent=np.float32(0.12),
              kp_out=_np(y))

    # max_pool (127-143) and per-cloud InstanceNorm block (474-530)
    with torch.no_grad():
        fx['maxpool_out'] = _np(m.blocks.max_pool(torch.from_numpy(x), torch.from_numpy(inds)))
        bn = m.blocks.BatchNormBlock(Cin, True, 0.02)
        lens = torch.tensor([20, 33])
        fx['inorm_lens'] = lens.numpy()
        fx['inorm_out'] = _np(bn(torch.from_numpy(x), lens))

    # PositionEmbeddingCoordsSine (position_embedding.py:7-50)
    pe = m.posemb.PositionEmbeddingCoordsSine(3, 256, scale=1.0)
    xyz = rng.normal(size=(29, 3)).astype(np.float32)
    fx['pe_xyz'] = xyz
    fx['pe_out'] = _np(pe(torch.from_numpy(xyz)))

    # compute_rigid_transform (se3_torch.py:108-154), batched, incl. a reflection case
    a = rng.normal(size=(4, 60, 3)).astype(np.float32)
    R = np.stack([np.linalg.qr(rng.normal(size=(3, 3)))[0] for _ in range(4)]).astype(np.float32)
    R[0] *= np.sign(np.linalg.det(R[0]))
    R[1] *= -np.sign(np.linalg.det(R[1]))                                 # improper: exercises det fix
    b = np.einsum('bij,bnj->bni', R, a) + rng.normal(size=(4, 1, 3)).astype(np.float32)
    b += rng.normal(size=b.shape).astype(np.float32) * 0.01
    w = rng.uniform(0, 1, size=(4, 60)).astype(np.float32)
    w[2, :50] = 0
    with torch.no_grad():
        T = m.se3.compute_rigid_transform(torch.from_numpy(a), torch.from_numpy(b), torch.from_numpy(w))
    fx.update(kabsch_a=a, kabsch_b=b, kabsch_w=w, kabsch_T=_np(T))

    # TransformerCrossEncoder on a PADDED batch of 2 pairs (transformers.py:18-59, 183-244)
    cfg = get_config('3dmatch')
    sd = random_state_dict(cfg, 21)
    layer = m.transformers.TransformerCrossEncoderLayer(
        256, 8, 1024, 0.0, activation='relu', normalize_before=True,
        sa_val_has_pos_emb=True, ca_val_has_pos_emb=True, attention_type='dot_prod')
    enc = m.transformers.TransformerCrossEncoder(layer, 6, torch.nn.LayerNorm(256), return_intermediate=True)
    enc.load_state_dict({k[len('transformer_encoder.'):]: v for k, v in sd.items()
                         if k.startswith('transformer_encoder.')}, strict=True)
    enc.eval()
    S, T_ = [23, 17], [19, 31]
    src = [torch.from_numpy(rng.normal(size=(n, 256)).astype(np.float32)) for n in S]
    tgt = [torch.from_numpy(rng.normal(size=(n, 256)).astype(np.float32)) for n in T_]
    sxyz = [torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32)) for n in S]
    txyz = [torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32)) for n in T_]
    pad = torch.nn.utils.rnn.pad_sequence

    def mask(lens):
        mk = torch.zeros((len(lens), max(lens)), dtype=torch.bool)
        for i, l in enumerate(lens):
            mk[i, l:] = True
        return mk
    with torch.no_grad():
        so, to = enc(pad(src), pad(tgt), src_key_padding_mask=mask(S), tgt_key_padding_mask=mask(T_),
                     src_pos=pad([pe(v) for v in sxyz]), tgt_pos=pad([pe(v) for v in txyz]))
    for b in range(2):
        fx[f'xenc_src_{b}'] = _np(src[b]); fx[f'xenc_tgt_{b}'] = _np(tgt[b])
        fx[f'xenc_sxyz_{b}'] = _np(sxyz[b]); fx[f'xenc_txyz_{b}'] = _np(txyz[b])
        fx[f'xenc_src_out_{b}'] = _np(so[:, :S[b], b]); fx[f'xenc_tgt_out_{b}'] = _np(to[:, :T_[b], b])
    np.savez_compressed(os.path.join(OUT, 'ops.npz'), **fx)
    print('ops', len(fx), 'arrays')


def eval_fixtures():
    """Registration metrics (SURVEY.md 8f N1): the reference's own est.log writer, 3DMatch benchmark, ModelNet
    metrics and metric aggregation on seeded synthetic trajectories (tests/golden/eval_inputs.py)."""
    import tempfile
    import types
    from scipy.spatial.transform import Rotation
    import eval_inputs as ei
    # environment shims only: numpy aliases removed after the reference's pinned numpy, and nibabel's
    # mat2quat (absent here) restated with scipy -- the benchmark only uses q's vector part in a quadratic form
    np.float, np.int = float, int
    m = ref_bridge.modules()
    import nibabel.quaternions as nq
    nq.mat2quat = lambda M: Rotation.from_matrix(np.asarray(M)).as_quat()[[3, 0, 1, 2]]
    with ref_bridge._in_ref_dir():
        import benchmark.benchmark_predator as bp
        import benchmark.benchmark_modelnet as bm
        import models.generic_reg_model as grm
    bp.nq = nq
    fx = {}
    scenes = ei.make_scenes()
    with tempfile.TemporaryDirectory() as tmp:
        gt_dir, log_dir = os.path.join(tmp, 'gt'), os.path.join(tmp, 'log')
        ei.write_gt(scenes, gt_dir)
        fake = types.SimpleNamespace(_log_path=log_dir, cfg=types.SimpleNamespace(benchmark='3DMatch'))
        for scene, d in scenes.items():
            for src, tgt, T in d['est']:                                  # the reference's own writer, one pair per call
                batch = {'src_xyz': [None], 'src_path': [f'x/{scene}/cloud_bin_{src}.pth'],
                         'tgt_path': [f'x/{scene}/cloud_bin_{tgt}.pth']}
                grm.GenericRegModel._save_3DMatch_log(fake, batch, {'pose': torch.from_numpy(T[None, None, :3].copy())})
        est_dir = os.path.join(log_dir, '3DMatch')
        s, recall = bp.benchmark(est_dir, gt_dir)
        fx['bench_str'] = np.frombuffer(s.encode('utf-8'), dtype=np.uint8)
        fx['bench_recall'] = np.array(recall)
        for scene in scenes:
            fx[f'flags_{scene}'] = np.load(os.path.join(est_dir, scene, 'flag.npy'))
            fx[f'errors_{scene}'] = np.load(os.path.join(est_dir, scene, 'errors.npy'))
        fx['est_log_scene_a'] = np.frombuffer(open(os.path.join(est_dir, 'scene-a', 'est.log'), 'rb').read(), dtype=np.uint8)
    data, pred = ei.modelnet_batch()
    met = bm.compute_metrics(data, pred)
    for k, v in met.items():
        fx[f'mn_{k}'] = np.asarray(v)
    for k, v in bm.summarize_metrics(met).items():
        fx[f'mns_{k}'] = np.asarray(v)
    fake = types.SimpleNamespace(reg_success_thresh_rot=10, reg_success_thresh_trans=0.1,
                                 logger=types.SimpleNamespace(info=lambda *a, **k: None))
    per = [grm.GenericRegModel._compute_metrics(fake, {'pose': p}, {'pose': g}) for p, g in ei.pose_batches()]
    agg = grm.GenericRegModel._aggregate_metrics(fake, per)
    for k, v in agg.items():
        fx[f'agg_{k}'] = _np(v)
    np.savez_compressed(os.path.join(OUT, 'eval.npz'), **fx)
    print('eval', len(fx), 'arrays; recall', recall)
    print(s)


def loss_fixture():
    """RegTR.compute_loss of the unmodified reference on the `fwd_modelnet_b1` forward with seeded overlap
    masks and ground-truth pose (tests/golden/eval_inputs.py:loss_inputs)."""
    import eval_inputs as ei
    cfg_name, wseed, makers = FORWARD_CASES['fwd_modelnet_b1'][:3]
    cfg = get_config(cfg_name)
    sd = random_state_dict(cfg, wseed)
    sd = ei.loss_state_dict(sd)
    model = ref_bridge.build_reference_model(cfg, sd)
    pairs = [mk() for mk in makers]
    batch = {'src_xyz': [torch.from_numpy(p['src_xyz']) for p in pairs], 'tgt_xyz': [torch.from_numpy(p['tgt_xyz']) for p in pairs]}
    with torch.no_grad():
        pred = model(batch)
        batch.update(ei.loss_inputs(pairs, [int(x.shape[0]) for x in batch['src_xyz']], [int(x.shape[0]) for x in batch['tgt_xyz']]))
        losses = model.compute_loss(pred, batch)
    fx = {f'loss_{k}': _np(v) for k, v in losses.items()}
    for lvl in range(len(batch['kpconv_meta']['points'])):
        fx[f'overlap_pyr_{lvl}'] = _np(batch['overlap_pyr'][f'pyr_{lvl}'])
    np.savez_compressed(os.path.join(OUT, 'loss.npz'), **fx)
    print('loss', {k: float(v) for k, v in fx.items() if k.startswith('loss_')})


def grad_fixture():
    """d(total loss)/d(parameters) of the unmodified reference (eval mode: dropout off, autograd on) on the
    `fwd_modelnet_b1` forward with the seeded loss inputs of loss_fixture: per parameter the l2 norm, the sum and 32
    sampled entries.  Pins the ORACLE's backward (tests/test_oracle_grad.py) -- the checker a CUDA backward (SURVEY.md
    8f N3) will be tested against."""
    import eval_inputs as ei
    grad_sample_index = ei.grad_sample_index
    cfg_name, wseed, makers = FORWARD_CASES['fwd_modelnet_b1'][:3]
    cfg = get_config(cfg_name)
    sd = ei.loss_state_dict(random_state_dict(cfg, wseed))
    model = ref_bridge.build_reference_model(cfg, sd)
    model.eval()
    for p_ in model.parameters():
        p_.requires_grad_(p_.is_floating_point())
    pairs = [mk() for mk in makers]
    batch = {'src_xyz': [torch.from_numpy(p['src_xyz']) for p in pairs], 'tgt_xyz': [torch.from_numpy(p['tgt_xyz']) for p in pairs]}
    pred = model(batch)
    batch.update(ei.loss_inputs(pairs, [int(x.shape[0]) for x in batch['src_xyz']], [int(x.shape[0]) for x in batch['tgt_xyz']]))
    losses = model.compute_loss(pred, batch)
    losses['total'].backward()
    fx = {'loss_total': _np(losses['total'].detach())}
    n = 0
    for name, p_ in model.named_parameters():
        if p_.grad is None:
            continue
        g = p_.grad.detach().double().reshape(-1)
        idx = grad_sample_index(name, g.numel())
        fx[f'g|{name}'] = np.concatenate([[float(g.norm()), float(g.sum())], g[torch.from_numpy(idx)].numpy()])
        n += 1
    np.savez_compressed(os.path.join(OUT, 'grad.npz'), **fx)
    print('grad: parameters with a gradient', n, 'total loss', float(fx['loss_total']))


def _ref_module(rel):
    """One reference source file imported on its own (its package __init__ pulls in h5py and friends)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('ref_' + os.path.basename(rel)[:-3], os.path.join(ref_bridge.REF_SRC, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def data_fixture():
    """Input side (tests/test_data.py): the reference's `collate_pair` on three items of the seeded pair files, its
    sequence helpers on seeded sequences, the full 3DMatch benchmark pickle (`test_3DMatch_info.pkl`, every row) and
    the SHA-256 of the shipped sample clouds, whose fp32 values the real_*_input.npz fixtures hold."""
    import pickle
    import tempfile
    import eval_inputs as ei
    from regtr_b200 import data as D
    collate = _ref_module(os.path.join('data_loaders', 'collate_functions.py')).collate_pair
    R = _ref_module(os.path.join('utils', 'seq_manipulation.py'))
    fx = {}
    with tempfile.TemporaryDirectory() as tmp:
        ei.write_pair_files(tmp)
        ds = D.ThreeDMatchPairs(tmp, os.path.join(tmp, 'info.pkl'))
        out = collate([ds[i] for i in (4, 0, 7)])
    fx['collate_keys'] = np.array(list(out))
    for k, v in out.items():
        if torch.is_tensor(v):
            fx[f'collate|{k}'] = _np(v)
        else:
            for b, x in enumerate(v):
                fx[f'collate|{k}|{b}'] = _np(x) if torch.is_tensor(x) else np.array(x)
    seqs, six = ei.seq_inputs()
    for i, kw in enumerate((dict(), dict(require_padding_mask=True, require_lens=True))):
        padded, mask, lens = R.pad_sequence(seqs, **kw)
        fx[f'pad{i}_padded'] = _np(padded)
        if mask is not None:
            fx[f'pad{i}_mask'] = _np(mask)
        if lens is not None:
            fx[f'pad{i}_lens'] = np.array(lens)
    lens = [s.shape[0] for s in seqs]
    for b, x in enumerate(R.unpad_sequences(six, lens)):
        fx[f'unpad_{b}'] = _np(x)
    src, tgt = R.split_src_tgt(torch.cat(seqs), lens)
    for b, x in enumerate(list(src) + list(tgt)):
        fx[f'split_{b}'] = _np(x)
    info = pickle.load(open(os.path.join(ref_bridge.REF_SRC, 'datasets', '3dmatch', 'test_3DMatch_info.pkl'), 'rb'))
    fx.update(info_rot=np.stack(info['rot']), info_trans=np.stack(info['trans']), info_src=np.array(info['src']),
              info_tgt=np.array(info['tgt']), info_overlap=np.array(info['overlap'], dtype=np.float64))
    for case, (_, _, src_rel, tgt_rel) in REAL_CASES.items():
        if src_rel.startswith('indoor/'):
            for rel in (src_rel, tgt_rel):
                fx[f'cloud_sha256|{rel}'] = sha(torch.load(os.path.join(REF_DATA, rel), weights_only=False))
    np.savez_compressed(os.path.join(OUT, 'data.npz'), **fx)
    print('data', len(fx), 'arrays;', len(info['rot']), 'benchmark rows')


def refcpp_fixture():
    """The reference's C++ pre-processing core (nanoflann radius search, hash-map grid subsampling; built into
    oracle/_ref by `make -C oracle ref`) on the clouds of eval_inputs.refcpp_inputs: every query's in-radius
    neighbours in the order returned (ragged: counts + concatenated ids) and the subsampled level sizes."""
    import eval_inputs as ei
    from oracle import pre
    ref = pre.RefCpp()
    pts, lens = ei.refcpp_inputs()
    b = ref.batch_neighbors(pts, pts, lens, lens, 0.11, 64)
    valid = b < len(pts)
    _, len_r = ref.batch_subsample(pts, lens, 0.1)
    np.savez_compressed(os.path.join(OUT, 'refcpp.npz'), neighbor_counts=valid.sum(1).astype(np.int32),
                        neighbor_ids=b[valid].astype(np.int32), subsample_lens=len_r)
    print('refcpp', int(valid.sum()), 'neighbours; level sizes', len_r.tolist())


if __name__ == '__main__':
    torch.manual_seed(0)
    np.random.seed(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'real':          # only the real-data fixtures (minutes of CPU)
        benchmark_fixture()
        for case in (sys.argv[2:] or REAL_CASES):
            real_fixture(case)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'bench':
        benchmark_fixture()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'grad':
        grad_fixture()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == 'data':
        data_fixture()
        refcpp_fixture()
        sys.exit(0)
    data_fixture()
    refcpp_fixture()
    eval_fixtures()
    loss_fixture()
    grad_fixture()
    op_fixtures()
    for case in FORWARD_CASES:
        forward_fixture(case)
    benchmark_fixture()
    for case in REAL_CASES:
        real_fixture(case)
    for f in sorted(os.listdir(OUT)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, 'KiB')
