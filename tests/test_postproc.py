"""Decode + temporal NMS (SURVEY.md section 8 rows a16 / f-1): oracle pinned to the reference, CUDA kernels bit-exact vs the oracle."""
import json
import os
import random

import pytest
import torch

from tests.helpers import GOLDEN


def _cases():
    with open(os.path.join(GOLDEN, "postproc_nms.json")) as f:
        return json.load(f)


def test_oracle_nms_matches_reference_fixtures():
    """tests/golden/postproc_nms.json was produced by the live reference utils.temporal_nms.temporal_nms."""
    from oracle import postproc_oracle as P

    cases = _cases()
    assert len(cases) == 64
    for c in cases:
        got = P.temporal_nms([list(r) for r in c["rows"]], c["nms_thd"], c["max_after_nms"])
        assert got == c["expected"], (c["nms_thd"], c["max_after_nms"], len(c["rows"]))


def random_nms_cases():
    """300 seeded (rows, nms_thd, max_after_nms) cases: empty lists, zero-length windows, zero scores."""
    rng = random.Random(3)
    cases = []
    for _ in range(300):
        n = rng.choice([0, 1, 2, 5, 10, 40])
        rows = []
        for _ in range(n):
            st = round(rng.uniform(0, 100), 4)
            rows.append([st, round(st + rng.choice([0.0, rng.uniform(0, 50)]), 4), round(rng.choice([0.0, rng.random()]), 4)])
        cases.append((rows, rng.choice([0.1, 0.5, 0.7, 0.9]), rng.choice([1, 3, 10, 100])))
    return cases


def test_oracle_nms_matches_live_reference_random():
    """Against what the reference's utils.temporal_nms.temporal_nms returned for random_nms_cases()
    (tests/golden/reference_pins.json, written by tests/golden/make_reference_pins.py)."""
    from oracle import postproc_oracle as P

    with open(os.path.join(GOLDEN, "reference_pins.json")) as f:
        expected = json.load(f)["temporal_nms_random"]
    cases = random_nms_cases()
    assert len(expected) == len(cases)
    for (rows, thd, ma), want in zip(cases, expected):
        assert P.temporal_nms([list(r) for r in rows], thd, ma) == want


def _random_batch(B, Lv, seed, ties=True):
    g = torch.Generator().manual_seed(seed)
    logits = torch.rand(B, Lv, 1, generator=g)
    if ties:  # repeated scores exercise the stable tie order
        logits = (logits * 16).round() / 16
    spans = torch.stack([-torch.rand(B, Lv, generator=g), torch.rand(B, Lv, generator=g)], dim=-1)
    lens = torch.randint(1, Lv + 1, (B,), generator=g)
    lens[0] = Lv
    mask = (torch.arange(Lv)[None, :] < lens[:, None]).float()
    centre = (torch.arange(Lv, dtype=torch.float32) + 0.5) / Lv
    ts = centre[None, :, None].expand(B, Lv, 2).contiguous()
    dur = (torch.rand(B, generator=g, dtype=torch.float64) * 140 + 10).tolist()
    sal = torch.randn(B, Lv, generator=g)
    return logits, spans, ts, mask, dur, sal


@pytest.mark.gpu
@pytest.mark.parametrize("B,Lv", [(1, 1), (3, 15), (32, 75), (8, 150), (2, 1200)])
def test_decode_kernel_bit_exact_vs_oracle(B, Lv):
    from oracle import postproc_oracle as P
    from univtg_b200 import postproc

    logits, spans, ts, mask, dur, _ = _random_batch(B, Lv, seed=100 + Lv)
    ref = P.decode_mr(logits, spans, ts, mask, dur, sort=True)
    out = postproc.decode_mr({"pred_logits": logits.cuda(), "pred_spans": spans.cuda()},
                             {"timestamp": ts.cuda(), "timestamp_mask": mask.cuda()}, dur, sort=True)
    got = out["windows_r4"].cpu().tolist()
    assert got == ref  # float(f"{e:.4f}") of every number, rows in Python's stable descending order
    # the fp32 rows are the unrounded values of the same ordering; order = source clip of each row
    order = out["order"].cpu().long()
    sc = logits[..., 0].clone()
    sc[mask == 0] = 0
    assert torch.equal(out["windows"][..., 2].cpu(), torch.gather(sc, 1, order))
    # unsorted variant keeps clip order
    out2 = postproc.decode_mr({"pred_logits": logits.cuda(), "pred_spans": spans.cuda()},
                              {"timestamp": ts.cuda(), "timestamp_mask": mask.cuda()}, dur, sort=False)
    assert out2["windows_r4"].cpu().tolist() == P.decode_mr(logits, spans, ts, mask, dur, sort=False)
    assert torch.equal(out2["order"].cpu(), torch.arange(Lv, dtype=torch.int32)[None].expand(B, Lv))


@pytest.mark.gpu
def test_round4_is_exact_on_adversarial_values():
    """Values whose fifth decimal sits next to a rounding boundary, exact ties included (x.xxxx5 representable cases)."""
    from oracle import postproc_oracle as P
    from univtg_b200 import postproc

    vals = [0.0, 1.0, 0.5, 0.00005, 0.00015, 0.12345, 0.123449999, 0.123450001, 2.5e-5, 7.5e-5, 1.00005, 149.99995, 150.0,
            0.03125, 0.09375, 3.0517578125e-05, 0.000152587890625, 1e-30, 0.99995, 0.999949, 123.45675, 99.99995]
    g = torch.Generator().manual_seed(5)
    vals += (torch.rand(2000, generator=g) * 150).tolist()
    vals += ((torch.randint(0, 1500000, (2000,), generator=g).float() + 0.5) / 10000).tolist()  # near-ties in fp32
    v = torch.tensor(vals, dtype=torch.float32)
    L = v.numel()
    logits = v[None, :, None].clone()  # the score column is rounded like the spans and is neither scaled nor clamped
    spans = torch.zeros(1, L, 2)
    ts = torch.zeros(1, L, 2)
    mask = torch.ones(1, L)
    for chunk in range(0, L, 4096):
        sl = slice(chunk, min(L, chunk + 4096))
        ref = P.decode_mr(logits[:, sl], spans[:, sl], ts[:, sl], mask[:, sl], [1.0], sort=False)
        out = postproc.decode_mr({"pred_logits": logits[:, sl].cuda(), "pred_spans": spans[:, sl].cuda()},
                                 {"timestamp": ts[:, sl].cuda(), "timestamp_mask": mask[:, sl].cuda()}, [1.0], sort=False)
        assert out["windows_r4"].cpu().tolist() == ref


@pytest.mark.gpu
@pytest.mark.parametrize("thd", [0.3, 0.7])
def test_nms_kernel_equals_oracle_on_decoded_rows(thd):
    from oracle import postproc_oracle as P
    from univtg_b200 import postproc

    logits, spans, ts, mask, dur, _ = _random_batch(16, 75, seed=9, ties=False)
    out = postproc.decode_mr({"pred_logits": logits.cuda(), "pred_spans": spans.cuda()},
                             {"timestamp": ts.cuda(), "timestamp_mask": mask.cuda()}, dur)
    rows = out["windows_r4"]
    for max_before, max_after in ((10, 10), (75, 5), (40, 100)):
        kept, counts = postproc.temporal_nms(rows, thd, max_before, max_after)
        ref = P.post_processing_mr_nms(rows.cpu().tolist(), thd, max_before, max_after)
        kept, counts = kept.cpu(), counts.cpu().tolist()
        for b in range(16):
            assert kept[b, :counts[b]].tolist() == ref[b]


@pytest.mark.gpu
def test_nms_kernel_equals_reference_fixtures():
    from univtg_b200 import postproc

    for c in _cases():
        rows = sorted([list(r) for r in c["rows"]], key=lambda r: r[2], reverse=True)  # the kernel takes sorted rows
        if not rows:
            continue
        w = torch.tensor([rows], dtype=torch.float64, device="cuda")
        kept, counts = postproc.temporal_nms(w, c["nms_thd"], len(rows), c["max_after_nms"])
        assert kept[0, :int(counts[0])].cpu().tolist() == c["expected"]


@pytest.mark.gpu
def test_compose_submission_matches_oracle_pipeline():
    from oracle import postproc_oracle as P
    from univtg_b200 import postproc

    B, Lv = 6, 75
    logits, spans, ts, mask, dur, sal = _random_batch(B, Lv, seed=21)
    meta = [{"qid": i, "query": f"q{i}", "vid": f"v{i}", "duration": dur[i]} for i in range(B)]
    outputs = {"pred_logits": logits.cuda(), "pred_spans": spans.cuda(), "saliency_scores": sal.cuda()}
    targets = {"timestamp": ts.cuda(), "timestamp_mask": mask.cuda()}
    inputs = {"src_vid_mask": mask.cuda()}
    for thd in (-1, 0.7):
        sub = postproc.compose_submission(meta, outputs, targets, inputs, nms_thd=thd)
        rows = P.decode_mr(logits, spans, ts, mask, dur)
        if thd != -1:
            rows = P.post_processing_mr_nms(rows, thd, 10, 10)
        sl = P.saliency_lists(sal, mask)
        for b in range(B):
            assert sub[b]["pred_relevant_windows"] == rows[b]
            assert sub[b]["pred_saliency_scores"] == sl[b]
            assert sub[b]["qid"] == b
