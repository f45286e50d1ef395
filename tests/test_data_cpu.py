"""Packed feature shards + batch loader (SURVEY.md section 8 row f-2) against the reference's own loading / collate code
(main/dataset.py:644-696 feature loading, :534-540 TEF, utils/tensor_utils.py:6-53 pad_sequences_1d), on the CPU."""
import os

import numpy as np
import torch

from tests.helpers import GOLDEN
from univtg_b200 import data as D


def _fake_corpus(tmp_path, n_vid=7, n_q=19, seed=0):
    """Reference on-disk layout: two video feature dirs ({vid}.npz['features'], slightly different lengths) + one query dir."""
    rng = np.random.default_rng(seed)
    d1, d2, dq = tmp_path / "slowfast", tmp_path / "clip", tmp_path / "clip_text"
    for d in (d1, d2, dq):
        d.mkdir()
    lens = rng.integers(9, 41, n_vid)
    for i, n in enumerate(lens):
        np.savez(d1 / f"v{i}.npz", features=rng.standard_normal((n + (i % 2), 24)).astype(np.float32))
        np.savez(d2 / f"v{i}.npz", features=rng.standard_normal((n, 8)).astype(np.float16))
    anns = []
    for q in range(n_q):
        np.savez(dq / f"{q}.npz", last_hidden_state=rng.standard_normal((int(rng.integers(3, 12)), 16)).astype(np.float32),
                 pooler_output=np.zeros(16, np.float32))
        anns.append({"qid": q, "vid": f"v{int(rng.integers(0, n_vid))}"})
    return [str(d1), str(d2)], str(dq), anns


def test_shard_roundtrip_and_loader_batches(tmp_path):
    v_dirs, q_dir, anns = _fake_corpus(tmp_path)
    path = str(tmp_path / "train.uvshard")
    hdr = D.pack_from_npz_dirs(path, anns, v_dirs, q_dir)
    sh = D.Shard(path)
    assert len(sh) == len(anns) and sh.v_feat_dim == 24 + 8 + 2 and sh.t_feat_dim == 16 and hdr["n_samples"] == len(anns)
    # every stored matrix == prepare_*() rounded to fp16
    for k, ann in enumerate(anns):
        vi, qi = sh.samples[k]
        feats = [np.load(os.path.join(d, f"{ann['vid']}.npz"))["features"] for d in v_dirs]
        np.testing.assert_array_equal(np.asarray(sh.video(vi)), D.prepare_video(feats).astype(np.float16))
        q = np.load(os.path.join(q_dir, f"{ann['qid']}.npz"))["last_hidden_state"]
        np.testing.assert_array_equal(np.asarray(sh.query(qi)), D.prepare_query(q).astype(np.float16))
    # loader: padding to the batch maximum, float masks, every sample exactly once over the ranks
    seen = []
    for rank in range(2):
        loader = D.ShardLoader(sh, batch_size=4, shuffle=True, seed=3, rank=rank, world=2, slots=3, workers=2)
        for batch, idx in loader:
            B, Lv, Dv = batch["src_vid"].shape
            assert batch["src_vid"].dtype == torch.float16 and batch["src_vid_mask"].dtype == torch.float32
            lv, lt = sh.lengths(idx)
            assert Lv == lv.max() and batch["src_txt"].shape[1] == lt.max()
            for b, k in enumerate(idx):
                vi, qi = sh.samples[k]
                np.testing.assert_array_equal(batch["src_vid"][b, :lv[b]].numpy(), np.asarray(sh.video(vi)))
                assert float(batch["src_vid"][b, lv[b]:].abs().sum()) == 0.0
                assert batch["src_vid_mask"][b].tolist() == [1.0] * int(lv[b]) + [0.0] * int(Lv - lv[b])
                np.testing.assert_array_equal(batch["src_txt"][b, :lt[b]].numpy(), np.asarray(sh.query(qi)))
                assert batch["src_txt_mask"][b].sum() == lt[b]
            seen += list(idx)
    assert sorted(seen) == list(range(len(anns)))


def test_prepared_features_and_collate_match_the_reference_code(tmp_path):
    """prepare_video / prepare_query / the loader's padding against what the reference's functions made of the same corpus:
    main/dataset.py:674-690 + 534-540 with utils.basic_utils.l2_normalize_np_array, then utils.tensor_utils.pad_sequences_1d
    (tests/golden/reference_pins.npz, written by tests/golden/make_reference_pins.py)."""
    z = np.load(os.path.join(GOLDEN, "reference_pins.npz"))
    pad_v, mask_v = torch.from_numpy(z["collate/vid"]), torch.from_numpy(z["collate/vid_mask"])
    pad_q, mask_q = torch.from_numpy(z["collate/txt"]), torch.from_numpy(z["collate/txt_mask"])
    v_dirs, q_dir, anns = _fake_corpus(tmp_path, seed=5)
    for b, ann in enumerate(anns[:6]):
        v = pad_v[b, :int(mask_v[b].sum())]
        q = pad_q[b, :int(mask_q[b].sum())]
        feats = [np.load(os.path.join(d, f"{ann['vid']}.npz"))["features"] for d in v_dirs]
        np.testing.assert_allclose(D.prepare_video(feats), v.numpy(), rtol=1e-6, atol=1e-7)
        np.testing.assert_allclose(D.prepare_query(np.load(os.path.join(q_dir, f"{ann['qid']}.npz"))["last_hidden_state"]), q.numpy(),
                                   rtol=1e-6, atol=1e-7)
    path = str(tmp_path / "six.uvshard")
    D.pack_from_npz_dirs(path, anns[:6], v_dirs, q_dir)
    (batch, idx), = list(D.ShardLoader(path, batch_size=6))
    assert list(idx) == list(range(6))
    assert torch.equal(batch["src_vid_mask"], mask_v) and torch.equal(batch["src_txt_mask"], mask_q)
    torch.testing.assert_close(batch["src_vid"].float(), pad_v.half().float(), rtol=0, atol=0)
    torch.testing.assert_close(batch["src_txt"].float(), pad_q.half().float(), rtol=0, atol=0)


def test_page_extents_merge_neighbouring_arrays():
    """Direct mode page-locks the shard's feature arrays: they are neighbours in the file, so the video array's last page is
    usually the text array's first - one registration must cover both (found on the GPU box: the second cudaHostRegister failed)."""
    from univtg_b200.data import page_extents

    assert page_extents([(4096 * 3 + 100, 5000), (4096 * 3 + 5100, 300)]) == [[4096 * 3, 4096 * 5]]
    assert page_extents([(8192, 4096), (12288, 10)]) == [[8192, 16384]]  # touching extents merge too
    assert page_extents([(100, 10), (3 * 4096 + 1, 4096)]) == [[0, 4096], [3 * 4096, 5 * 4096]]
    assert page_extents([(100, 0), (5000, 1)]) == [[4096, 8192]]  # empty arrays are skipped
