"""CPU tests of the input pipeline (SURVEY.md 8f N2, regtr_b200/data.py): file formats of the reference's
3DMatch loader, collate layout, size bucketing, read-ahead stream.  What the unmodified reference computed or
shipped is read from tests/golden/data.npz (tests/golden/make_golden.py:data_fixture)."""
import os
import pickle
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, REAL_CASES, load_golden, sha256_of

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
import eval_inputs as ei  # noqa: E402
from regtr_b200 import data as D  # noqa: E402


@pytest.fixture(scope='module')
def fx():
    return load_golden('data')


def _make_dataset(tmp_path, n_pairs=11, seed=0):
    infos = ei.write_pair_files(str(tmp_path), n_pairs, seed)
    return D.ThreeDMatchPairs(str(tmp_path), str(tmp_path / 'info.pkl')), infos


def test_dataset_items_and_collate(tmp_path):
    ds, infos = _make_dataset(tmp_path)
    assert len(ds) == 11
    it = ds[3]
    assert it['src_xyz'].dtype == torch.float32 and it['src_xyz'].shape[1] == 3
    assert it['pose'].shape == (3, 4) and it['idx'] == 3 and it['src_path'].endswith('cloud_bin_4.pth')
    np.testing.assert_allclose(it['pose'][:, :3].numpy(), infos['rot'][3], atol=1e-6)
    np.testing.assert_allclose(it['pose'][:, 3:].numpy(), infos['trans'][3], atol=1e-6)
    b = D.collate_pair([ds[0], ds[1], ds[2]])
    assert isinstance(b['src_xyz'], list) and len(b['tgt_xyz']) == 3 and b['pose'].shape == (3, 3, 4)
    assert b['overlap_p'].shape == (3,) and b['idx'] == [0, 1, 2]


def test_collate_matches_reference_function(tmp_path, fx):
    """collate_pair vs what the reference's data_loaders/collate_functions.py returned for the same three items."""
    ds, _ = _make_dataset(tmp_path)
    items = [ds[i] for i in (4, 0, 7)]
    a = D.collate_pair(items)
    assert set(a) == set(fx['collate_keys'].tolist())
    for k in a:
        if torch.is_tensor(a[k]):
            want = fx[f'collate|{k}']
            assert a[k].dtype == torch.from_numpy(want).dtype and torch.equal(a[k], torch.from_numpy(want))
        else:
            want = [fx[f'collate|{k}|{b}'] for b in range(sum(key.startswith(f'collate|{k}|') for key in fx))]
            assert len(a[k]) == len(want) and all(
                (torch.equal(x, torch.from_numpy(y)) if torch.is_tensor(x) else x == y.item()) for x, y in zip(a[k], want))


def test_reads_the_reference_sample_pairs(tmp_path, fx):
    """The 3DMatch pairs shipped with the reference (data/indoor, demo.py) through the real benchmark pickle, both
    rebuilt from the fixtures: every row of test_3DMatch_info.pkl with the original Python types, and the clouds as
    float64 files from the fp32 input fixtures (the shipped files hold fp32 values; their SHA-256 pins that)."""
    root, info = tmp_path / 'indoor', tmp_path / 'test_3DMatch_info.pkl'
    with open(info, 'wb') as f:
        pickle.dump(dict(rot=list(fx['info_rot']), trans=list(fx['info_trans']), src=fx['info_src'].tolist(),
                         tgt=fx['info_tgt'].tolist(), overlap=[np.float64(v) for v in fx['info_overlap']]), f)
    n_clouds = 0
    for case in REAL_CASES:
        inp = np.load(os.path.join(GOLDEN, 'real', case + '_input.npz'))
        for side in ('src', 'tgt'):
            rel = str(inp[f'{side}_file'])
            if rel.startswith('indoor/'):
                cloud = inp[f'{side}_xyz'].astype(np.float64)
                assert np.array_equal(sha256_of(cloud), fx[f'cloud_sha256|{rel}']), rel
                os.makedirs(os.path.dirname(tmp_path / rel), exist_ok=True)
                torch.save(cloud, tmp_path / rel)
                n_clouds += 1
    assert n_clouds == sum(k.startswith('cloud_sha256|') for k in fx) == 6
    ds = D.ThreeDMatchPairs(str(root), str(info))
    assert len(ds) == 1623
    have = [i for i in range(len(ds)) if all(os.path.isfile(os.path.join(root, ds.infos[k][i])) for k in ('src', 'tgt'))]
    assert have, 'no complete pair among the shipped sample clouds'
    it = ds[have[0]]
    raw = torch.load(os.path.join(root, it['src_path']), weights_only=False)
    assert raw.dtype == np.float64 and torch.equal(it['src_xyz'], torch.from_numpy(raw).float())
    assert 5000 < it['src_xyz'].shape[0] < 60000 and it['pose'].shape == (3, 4)


def test_bucket_order_is_a_partition_grouped_by_capacity():
    rng = np.random.default_rng(1)
    sizes = rng.integers(20000, 60000, size=200).tolist()
    batches = D.bucket_order(sizes, batch_size=4, bucket=8192, window=64)
    flat = [i for b in batches for i in b]
    assert sorted(flat) == list(range(200))
    assert all(len(b) <= 4 for b in batches)
    assert max(flat[:64]) < 64 and min(flat[64:128]) >= 64                   # windows keep the dataset order
    cap = lambda i: -(-sizes[i] // 8192)
    assert all(cap(a) <= cap(b) for a, b in zip(flat[:63], flat[1:64]))       # grouped by bucket inside a window
    changes = sum(cap(a) != cap(b) for a, b in zip(flat, flat[1:]))
    naive = sum(cap(a) != cap(b) for a, b in zip(range(199), range(1, 200)))
    assert changes < naive / 3                                                # far fewer graph switches


def test_pair_stream_order_and_errors(tmp_path):
    ds, _ = _make_dataset(tmp_path, n_pairs=23)
    batches = D.bucket_order(ds.sizes(), batch_size=3, bucket=256, window=8)
    got = [b['idx'] for b in D.PairStream(ds, batches, workers=3, depth=2)]
    assert got == [list(b) for b in batches]
    os.remove(tmp_path / 'test' / 'scene' / 'cloud_bin_5.pth')
    with pytest.raises(Exception):
        list(D.PairStream(ds, batches, workers=2, depth=2))


def test_sequence_helpers_match_reference(fx):
    """regtr_b200.seq vs what utils/seq_manipulation.py returned on the same inputs, plus a padded round trip."""
    from regtr_b200 import seq as S
    seqs, six = ei.seq_inputs()
    padded, mask, lens = S.pad_sequence(seqs, require_padding_mask=True, require_lens=True)
    assert padded.shape == (11, 4, 5) and mask.shape == (4, 11) and lens == [7, 3, 11, 1]
    assert mask[1, 3:].all() and not mask[1, :3].any() and not mask[2].any()
    back = S.unpad_sequences(padded, lens)
    assert all(torch.equal(a, b) for a, b in zip(back, seqs))
    stacked = torch.cat(seqs)
    src, tgt = S.split_src_tgt(stacked, torch.tensor(lens))
    assert len(src) == 2 and torch.equal(tgt[1], seqs[3])
    T = lambda key: torch.from_numpy(fx[key])
    for i, kw in enumerate((dict(), dict(require_padding_mask=True, require_lens=True))):
        a = S.pad_sequence(seqs, **kw)
        assert torch.equal(a[0], T(f'pad{i}_padded'))
        assert (a[1] is None) == (f'pad{i}_mask' not in fx) and (a[2] is None) == (f'pad{i}_lens' not in fx)
        if a[1] is not None:
            assert torch.equal(a[1], T(f'pad{i}_mask')) and a[2] == fx[f'pad{i}_lens'].tolist()
    got = S.unpad_sequences(six, lens)
    assert len(got) == 4 and all(torch.equal(x, T(f'unpad_{b}')) for b, x in enumerate(got))
    a = S.split_src_tgt(stacked, lens)
    assert len(a[0]) == len(a[1]) == 2 and all(torch.equal(x, T(f'split_{b}')) for b, x in enumerate(a[0] + a[1]))


def test_compute_overlap_properties(tmp_path):
    rng = np.random.default_rng(4)
    tgt = rng.uniform(0, 1, size=(400, 3))
    src = np.concatenate([tgt[:250] + rng.normal(scale=0.002, size=(250, 3)), rng.uniform(2, 3, size=(80, 3))])
    sm, tm, corr = D.compute_overlap(src, tgt, 0.02)
    assert sm[:250].all() and not sm[250:].any()                 # the shifted copies overlap, the far blob does not
    assert tm[:250].all() and tm[250:].sum() < 40
    s_idx, t_idx = corr
    assert (np.linalg.norm(src[s_idx] - tgt[t_idx], axis=1) < 0.02).all()
    assert (s_idx[t_idx == s_idx] > 0).all() and len(s_idx) > 200     # mutual matches, index 0 excluded (reference quirk)
    # brute-force nearest neighbour agrees
    d = np.linalg.norm(src[:, None] - tgt[None], axis=-1)
    assert np.array_equal(sm, d.min(1) < 0.02)
    ds, infos = _make_dataset(tmp_path)
    ds.overlap_radius = 0.5
    it = ds[2]
    assert it['src_overlap'].dtype == torch.bool and it['src_overlap'].shape[0] == it['src_xyz'].shape[0]
    assert it['correspondences'].shape[0] == 2
    b = D.collate_pair([ds[0], ds[1]])
    assert isinstance(b['correspondences'], list) and len(b['src_overlap']) == 2
