"""The oracle against the committed golden vectors (tests/golden/*.npz), which were produced by
EXECUTING THE REFERENCE'S OWN CLASSES (oracle/make_golden.py).  CPU only."""
import glob
import json
import os

import numpy as np
import pytest
import torch

import mfar_oracle as O

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(glob.glob(os.path.join(GOLDEN, "*.npz")))


def load(path):
    z = np.load(path, allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    return z, meta


def test_golden_files_present():
    assert len(CASES) >= 5


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_dense_retrieve_batch_matches_reference(path):
    z, m = load(path)
    q = torch.from_numpy(z["q"])
    for f in range(m["Fd"]):
        v = torch.from_numpy(z["fields"][f])
        s, r = O.dense_retrieve_batch(q, v, m["k"], vector_batch_size=max(7, m["N"] // 3))
        np.testing.assert_allclose(s.numpy(), z["ref_retrieve_scores"][f], rtol=1e-6, atol=1e-6)
        # ids equal wherever the score is not tied with a neighbour
        ref_r = z["ref_retrieve_rows"][f]
        same = r.numpy() == ref_r
        if not same.all():
            sc = z["ref_retrieve_scores"][f]
            bad = np.argwhere(~same)
            for qi, j in bad:
                tied = (j > 0 and sc[qi, j] == sc[qi, j - 1]) or (j + 1 < sc.shape[1] and sc[qi, j] == sc[qi, j + 1])
                assert tied, f"field {f} q{qi} rank {j}: {r[qi, j]} vs {ref_r[qi, j]}"


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_score_batch_matches_reference(path):
    z, m = load(path)
    q = torch.from_numpy(z["q"])
    rows = z["cand_rows"].tolist()
    for f in range(m["Fd"]):
        got = O.dense_score_batch(q, torch.from_numpy(z["fields"][f]), rows)
        np.testing.assert_allclose(got.numpy(), z["ref_score_batch"][f], rtol=1e-6, atol=1e-6)
    if m["Fs"]:
        sp = torch.from_numpy(z["sparse"])
        for j in range(m["Fs"]):
            got = O.sparse_score_batch(sp[:, j, :], rows + [-1])
            np.testing.assert_array_equal(got.numpy(), z["ref_sparse_score_batch"][j])
            assert (got[:, -1] == 0).all()           # unknown key -> 0 (index.py:117)


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_exhaustive_scores_match_reference_mixture(path):
    """oracle.exhaustive_scores == reference LinearWeights over reference per-field scores of all docs."""
    z, m = load(path)
    q = torch.from_numpy(z["q"])
    W = torch.from_numpy(z["W"])
    w = O.mixture_weights(q if m["query_cond"] else None, W, m["query_cond"])
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    sp = torch.from_numpy(z["sparse"]) if m["Fs"] else None
    got = O.exhaustive_scores(q, fields, sp, w, torch.from_numpy(z["mask"]))
    ref = z["ref_mix_all"]
    np.testing.assert_allclose(got.numpy(), ref, rtol=2e-6, atol=2e-6 * np.abs(ref).max())


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_union_rescore_matches_reference_pipeline(path):
    z, m = load(path)
    q = torch.from_numpy(z["q"])
    W = torch.from_numpy(z["W"])
    fields = [torch.from_numpy(z["fields"][f]) for f in range(m["Fd"])]
    sp = torch.from_numpy(z["sparse"]) if m["Fs"] else None
    if bool(z["ref_union_raises"]):
        # duplicates of row 0 (zero-init quirk) left the union smaller than k: reference torch.topk raises
        with pytest.raises(Exception):
            O.union_rescore(q, fields, sp, q, W, m["query_cond"], torch.from_numpy(z["mask"]), m["k"],
                            vector_batch_size=max(7, m["N"] // 3))
        return
    vals, rows = O.union_rescore(q, fields, sp, q, W, m["query_cond"], torch.from_numpy(z["mask"]), m["k"],
                                 vector_batch_size=max(7, m["N"] // 3))
    for i in range(m["Q"]):
        np.testing.assert_allclose(vals[i].numpy(), z["ref_union_vals"][i], rtol=2e-6, atol=1e-6)
        ref_rows = z["ref_union_rows"][i]
        diff = np.asarray(rows[i]) != ref_rows
        if diff.any():                                # only exact ties may be ordered differently
            v = z["ref_union_vals"][i]
            for j in np.nonzero(diff)[0]:
                assert (j > 0 and v[j] == v[j - 1]) or (j + 1 < len(v) and v[j] == v[j + 1])


def test_zero_init_quirk_is_exercised():
    z, m = load(os.path.join(GOLDEN, "zero_init_quirk.npz"))
    sc, rows = z["ref_retrieve_scores"], z["ref_retrieve_rows"]
    assert (sc == 0.0).any() and (rows[sc == 0.0] == 0).all()      # (0.0, row 0) entries, index.py:192-193
    assert bool(z["ref_union_raises"])


def test_topk_sorted_tie_break_and_matches_torch():
    g = torch.Generator().manual_seed(3)
    s = torch.randn(4, 1000, generator=g)
    s[:, 10] = s[:, 20] = s[:, 5] = 9.0               # ties at the top: lower row first
    v, i = O.topk_sorted(s, 50)
    tv, _ = torch.topk(s, 50, dim=1)
    np.testing.assert_array_equal(v.numpy(), tv.numpy())
    assert i[:, :3].tolist() == [[5, 10, 20]] * 4
