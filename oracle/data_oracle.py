"""TEST INFRASTRUCTURE -- CPU restatement (numpy, float64 like the reference) of the reference's host-side input
pipeline, the checker for raindrop_b200/data.py.  Only tests/ may import this file.

Each function follows the reference line by line:
  get_stats              code/utils_rd.py:149-161   (getStats)
  mask_normalize         code/utils_rd.py:164-175
  mask_normalize_static  code/utils_rd.py:203-218   (with getStats_static's always-false test, :195, giving ms=0, ss=1)
  tensorize_normalize    code/utils_rd.py:221-240 + the permutes of code/Raindrop.py:233-239
  remove_features        code/Raindrop.py:214-231
  epoch_batches          code/Raindrop.py:261-309  (strategy 2 and 3)
Pinned against the reference's own functions in tests/test_data_pipeline.py::test_data_oracle_matches_reference
(their outputs stored in tests/golden/data_pipeline.npz by oracle/make_golden.py).
"""
import numpy as np
import torch


def get_stats(P_tensor):
    N, T, F = P_tensor.shape
    Pf = P_tensor.transpose((2, 0, 1)).reshape(F, -1)
    mf, stdf = np.zeros((F, 1)), np.ones((F, 1))
    for f in range(F):
        vals = Pf[f, :]
        vals = vals[vals > 0]
        mf[f] = np.mean(vals)
        stdf[f] = np.max([np.std(vals), 1e-7])
    return mf, stdf


def mask_normalize(P_tensor, mf, stdf):
    N, T, F = P_tensor.shape
    Pf = P_tensor.transpose((2, 0, 1)).reshape(F, -1).astype(np.float64)
    M = 1 * (P_tensor > 0)
    M_3D = M.transpose((2, 0, 1)).reshape(F, -1)
    for f in range(F):
        Pf[f] = (Pf[f] - mf[f]) / (stdf[f] + 1e-18)
    Pf = Pf * M_3D
    Pnorm = Pf.reshape((F, N, T)).transpose((1, 2, 0))
    return np.concatenate([Pnorm, M], axis=2)


def mask_normalize_static(P_static):
    """ms = 0, ss = 1 always (getStats_static's `if bool_categorical == 0` compares a list with 0)."""
    Ps = np.array(P_static, dtype=np.float64) / (1.0 + 1e-18)
    Ps[Ps <= 0] = 0
    return Ps


def tensorize_normalize(P_raw, minutes, static, y, mf, stdf):
    """-> (P [T, n, 2F], Pstatic [n, D] | None, Ptime [T, n], y [n]) as float32 / int64 torch tensors."""
    P = torch.Tensor(mask_normalize(np.asarray(P_raw, dtype=np.float64), mf, stdf)).permute(1, 0, 2).contiguous()
    t = (torch.Tensor(np.asarray(minutes, dtype=np.float64)[:, :, None]) / 60.0).squeeze(2).permute(1, 0).contiguous()
    st = None if static is None else torch.Tensor(mask_normalize_static(static))
    yt = torch.Tensor(np.asarray(y).reshape(len(y), -1)[:, 0]).type(torch.LongTensor)
    return P, st, t, yt


def remove_features(P_ntf, missing_ratio, level="sample", density_scores=None):
    """In place on [n, T, 2F] like the reference (global numpy RNG)."""
    num_all = int(P_ntf.shape[2] / 2)
    k = round(missing_ratio * num_all)
    if level == "sample":
        for i in range(P_ntf.shape[0]):
            idx = np.random.choice(num_all, k, replace=False)
            P_ntf[i][:, idx] = 0
    else:
        idx = np.asarray(density_scores[:k]).astype(int)
        P_ntf[:, :, idx] = 0
    return P_ntf


def epoch_batches(y, batch_size, strategy, state):
    """One epoch of index batches.  `state` carries (idx_0, expanded_idx_1) across epochs like the reference's
    in-place shuffles."""
    y = np.asarray(y).reshape(len(y), -1)[:, 0]
    if state is None:
        idx_0, idx_1 = np.where(y == 0)[0], np.where(y == 1)[0]
        state = [idx_0, np.concatenate([idx_1, idx_1, idx_1], axis=0)]
    idx_0, exp1 = state
    half = int(batch_size / 2)
    if strategy == 2:
        n_batches = np.min([len(idx_0) // half, len(exp1) // half])
        np.random.shuffle(exp1)
        I1 = exp1
        np.random.shuffle(idx_0)
        I0 = idx_0
        out = [np.concatenate([I0[n * half:(n + 1) * half], I1[n * half:(n + 1) * half]], axis=0) for n in range(n_batches)]
    else:
        out = [np.random.choice(list(range(len(y))), size=int(batch_size), replace=False) for _ in range(30)]
    return np.stack(out), state
