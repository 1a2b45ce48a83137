"""Input pipeline (raindrop_b200/data.py) against the CPU restatement of the reference's host code
(oracle/data_oracle.py) -- and that restatement against the reference's own functions where they are present."""
import os

import numpy as np
import pytest
import torch

from helpers import normwise
from oracle import data_oracle as DO
from raindrop_b200 import data as RD


def _raw(n=23, T=17, F=6, D=4, seed=0):
    g = np.random.default_rng(seed)
    P = g.normal(50, 20, (n, T, F)) * (g.random((n, T, F)) < 0.35)
    P[P < 0] = 0
    lens = g.integers(2, T + 1, n)
    for i in range(n):
        P[i, lens[i]:] = 0
    minutes = np.cumsum(g.random((n, T)) * 60 + 1, 1) * (np.arange(T)[None, :] < lens[:, None])
    static = g.normal(1, 2, (n, D))
    y = (g.random(n) < 0.3).astype(np.int64)[:, None]
    return P, minutes, static, y


def test_on_disk_readers(tmp_path):
    """PTdict_list.npy as written by P12data/process_scripts/IrregularSampling.py:69-86, and the PAM array form."""
    P, minutes, static, y = _raw()
    lst = [{"id": i, "static": static[i, :2], "extended_static": static[i], "arr": P[i], "time": minutes[i][:, None],
            "length": int((minutes[i] > 0).sum())} for i in range(len(P))]
    np.save(tmp_path / "PTdict_list.npy", np.array(lst, dtype=object), allow_pickle=True)
    P2, m2, s2 = RD.load_ptdict_list(str(tmp_path / "PTdict_list.npy"))
    assert P2.dtype == np.float32 and np.array_equal(P2, P.astype(np.float32))
    assert np.array_equal(m2, minutes.astype(np.float32)) and np.array_equal(s2, static.astype(np.float32))
    np.save(tmp_path / "pam.npy", P)
    P3, m3, s3 = RD.load_array_dataset(str(tmp_path / "pam.npy"))
    assert s3 is None and np.array_equal(P3, P.astype(np.float32))
    assert np.allclose(m3[0], torch.linspace(0, P.shape[1], P.shape[1]).numpy())       # code/utils_rd.py:247
    np.save(tmp_path / "split.npy", np.array([np.arange(5), np.arange(5, 8), np.arange(8, 10)], dtype=object), allow_pickle=True)
    tr, va, te = RD.load_split(str(tmp_path / "split.npy"))
    assert list(tr) == [0, 1, 2, 3, 4] and list(va) == [5, 6, 7] and list(te) == [8, 9]


def test_epoch_sampler_matches_reference_procedure():
    """Same numpy RNG calls in the same order as code/Raindrop.py:292-309 -> the same batches."""
    y = (np.random.default_rng(3).random(1000) < 0.2).astype(np.int64)
    for strategy in (2, 3):
        np.random.seed(11)
        s = RD.EpochSampler(y, batch_size=128, strategy=strategy, device="cpu")
        mine = [s.epoch().numpy() for _ in range(3)]
        np.random.seed(11)
        state, ref = None, []
        for _ in range(3):
            b, state = DO.epoch_batches(y, 128, strategy, state)
            ref.append(b)
        assert all(np.array_equal(a, b) for a, b in zip(mine, ref))
        if strategy == 2:       # balanced: half negatives, half (upsampled) positives
            assert (y[mine[0][:, :64]] == 0).all() and (y[mine[0][:, 64:]] == 1).all()


def test_removal_indices_match_reference_choice():
    np.random.seed(5)
    idx = RD.removal_indices(7, 34, 0.3, "sample")
    np.random.seed(5)
    ref = np.stack([np.random.choice(34, round(0.3 * 34), replace=False) for _ in range(7)])
    assert idx.shape == (7, 10) and np.array_equal(idx, ref)
    assert list(RD.removal_indices(7, 34, 0.3, "set", density_scores=np.arange(34)[::-1])) == list(range(33, 23, -1))


def test_data_oracle_matches_reference(golden_dir):
    """Pins oracle/data_oracle.py to the reference's own utils_rd functions (bit-identical float64 results), stored by
    oracle/make_golden.py data_pipeline_case for these raw arrays."""
    z = np.load(os.path.join(golden_dir, "data_pipeline.npz"))
    P, minutes, static, y = _raw(seed=4)
    mf, stdf = DO.get_stats(P)
    if "getStats.mf" in z.files:
        assert np.array_equal(z["getStats.mf"], mf) and np.array_equal(z["getStats.stdf"], stdf)
    # numpy >= 1.24 rejects the reference's `np.max([stdf[f], eps])` (a (1,) array next to a scalar, code/utils_rd.py:160),
    # so the fixture may lack getStats; the restatement is the same arithmetic on the scalar.  Check it against a direct
    # computation as well.
    Pf = P.transpose((2, 0, 1)).reshape(P.shape[2], -1)
    for f in range(P.shape[2]):
        v = Pf[f][Pf[f] > 0]
        assert mf[f, 0] == np.mean(v) and stdf[f, 0] == max(np.std(v), 1e-7)
    assert np.array_equal(z["mask_normalize"], DO.mask_normalize(P.copy(), mf, stdf))
    ms, ss = z["getStats_static.ms"], z["getStats_static.ss"]
    assert ms.shape == ss.shape == (static.shape[1], 1)
    assert (ms == 0).all() and (ss == 1).all()                           # the always-false categorical test
    assert np.array_equal(z["mask_normalize_static"], DO.mask_normalize_static(static))
    a = [torch.from_numpy(z["tensorize_normalize.%d" % i]) for i in range(4)]
    b = DO.tensorize_normalize(P, minutes, static, y, mf, stdf)
    assert torch.equal(a[0].permute(1, 0, 2), b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(a[2].squeeze(2).permute(1, 0), b[2]) and torch.equal(a[3], b[3])


@pytest.mark.gpu
def test_device_normalisation_matches_reference_math():
    """rd_feature_stats / rd_mask_normalize: the mask is bit-exact, values agree with the float64 reference math to
    <= 1e-6 (the inputs are held in float32 on the device)."""
    P, minutes, static, y = _raw(n=301, T=60, F=34, D=6, seed=7)
    P32 = P.astype(np.float32)
    mf, stdf = DO.get_stats(P32.astype(np.float64))
    dev = torch.device("cuda")
    m_d, s_d = RD.feature_stats(torch.as_tensor(P32).to(dev))
    assert normwise(m_d, mf[:, 0]) < 1e-6 and normwise(s_d, stdf[:, 0]) < 1e-6
    ref = DO.tensorize_normalize(P32, minutes.astype(np.float32), static.astype(np.float32), y, mf, stdf)
    got = RD.tensorize_normalize(P32, minutes.astype(np.float32), static.astype(np.float32), y,
                                 torch.as_tensor(mf[:, 0]).float().to(dev), torch.as_tensor(stdf[:, 0]).float().to(dev))
    F_ = P.shape[2]
    assert torch.equal(got[0][:, :, F_:].cpu(), ref[0][:, :, F_:])                     # observation mask: bit-exact
    assert normwise(got[0][:, :, :F_], ref[0][:, :, :F_]) < 1e-6
    assert torch.equal(got[1].cpu(), ref[1]) and torch.equal(got[3].cpu(), ref[3])
    assert normwise(got[2], ref[2]) < 1e-7
    # with the device statistics end to end
    got2 = RD.tensorize_normalize(P32, minutes.astype(np.float32), None, y, m_d, s_d)
    assert got2[1] is None and normwise(got2[0][:, :, :F_], ref[0][:, :, :F_]) < 1e-5


@pytest.mark.gpu
def test_device_dataset_fill_and_feature_removal_are_bit_exact():
    from raindrop_b200.synth import make_batch, model_config
    cfg = model_config("P19", dropout=0.2)
    full = make_batch(cfg, 300, seed=9)
    ds = RD.DeviceDataset(full["src"], full["static"], full["times"], full["y"])
    B = 37
    buf = RD.BatchBuffers(cfg["max_len"], B, 2 * cfg["d_inp"], cfg["d_static"])
    idx = torch.randperm(300, generator=torch.Generator().manual_seed(1))[:B]
    np.random.seed(2)
    rem = RD.removal_indices(B, cfg["d_inp"], 0.3, "sample")
    ds.fill(buf, idx, removed=rem)
    ref = full["src"][:, idx].clone()
    for j in range(B):
        ref[:, j, rem[j]] = 0                                     # code/Raindrop.py:218-220 (value columns only)
    assert torch.equal(buf.src.cpu(), ref)
    assert torch.equal(buf.times.cpu(), full["times"][:, idx]) and torch.equal(buf.static.cpu(), full["static"][idx])
    assert torch.equal(buf.y.cpu(), full["y"][idx])
    assert torch.equal(buf.lengths.cpu(), torch.sum(full["times"][:, idx] > 0, dim=0))
    # 'set' level: one index list for everybody
    ds.fill(buf, idx, removed=np.array([0, 5, 33]))
    ref = full["src"][:, idx].clone(); ref[:, :, [0, 5, 33]] = 0
    assert torch.equal(buf.src.cpu(), ref)
    # odd width (PAM: 2 * 17 columns -> scalar copy path)
    cfgp = model_config("PAM", dropout=0.2)
    fp = make_batch(cfgp, 20, seed=3)
    dsp = RD.DeviceDataset(fp["src"], None, fp["times"], fp["y"])
    bp = RD.BatchBuffers(cfgp["max_len"], 7, 2 * cfgp["d_inp"], 0)
    ip = torch.tensor([3, 0, 19, 7, 7, 12, 1])
    dsp.fill(bp, ip)
    assert torch.equal(bp.src.cpu(), fp["src"][:, ip]) and torch.equal(bp.lengths.cpu(), torch.sum(fp["times"][:, ip] > 0, dim=0))
    # a dataset without statics (PAM)
    ds2 = RD.DeviceDataset(full["src"], None, full["times"], full["y"])
    buf2 = RD.BatchBuffers(cfg["max_len"], B, 2 * cfg["d_inp"], 0)
    ds2.fill(buf2, idx)
    assert torch.equal(buf2.src.cpu(), full["src"][:, idx])
