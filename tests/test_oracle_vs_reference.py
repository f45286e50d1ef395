"""Pin the oracle against the reference: tests/golden/reference_pins.{npz,json} hold what the unmodified reference computes for
each case below (written by tests/golden/make_reference_pins.py); inputs, weights and random draws are regenerated from seeds."""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from tests.helpers import GOLDEN
from univtg_b200 import synth

OUT_KEYS = ("pred_logits", "pred_spans", "saliency_scores", "vid_mem_proj", "txt_mem_proj")


def _pins():
    with open(os.path.join(GOLDEN, "reference_pins.json")) as f:
        return json.load(f)


def _ref_out(prefix, keys=OUT_KEYS):
    z = np.load(os.path.join(GOLDEN, "reference_pins.npz"))
    return {k: torch.from_numpy(z[f"{prefix}/{k}"]) for k in keys}


def _stored(out):
    """The oracle's outputs as the fixture stores them (vid_mem_proj at every vid_stride-th clip)."""
    stride = int(np.load(os.path.join(GOLDEN, "reference_pins.npz"))["meta/vid_stride"])
    return {k: (v[:, ::stride] if k == "vid_mem_proj" else v) for k, v in out.items()}


def _assert_losses(loss, ref_loss):
    assert sorted(loss) == sorted(ref_loss)
    for k, v in ref_loss.items():
        assert abs(float(loss[k]) - v) < 5e-6 * max(1.0, abs(v)), k


@pytest.mark.parametrize("cfg_name,ragged,batch", [("tiny", True, None), ("tiny", False, 5), ("cfg1", True, 3)])
def test_forward_and_losses(cfg_name, ragged, batch):
    from oracle import univtg_oracle as O

    cfg = synth.CONFIGS[cfg_name]
    sd = synth.make_state_dict(cfg, seed=123)
    inp = synth.make_inputs(cfg, seed=7, ragged=ragged, batch=batch)
    tgt = synth.make_targets(inp, seed=8)
    case = f"{cfg_name}_{int(ragged)}_{batch}"
    ref = _ref_out("forward/" + case)
    out = O.forward(sd, cfg, **inp)
    for k in OUT_KEYS:
        torch.testing.assert_close(_stored(out)[k], ref[k].double(), rtol=2e-5, atol=2e-5)
    _assert_losses(O.criterion(out, tgt), _pins()["forward_loss/" + case])


def test_bool_masks_of_the_highlight_path_give_the_same_outputs():
    """The HL collate hands the model bool masks (main/dataset.py:1104) where the MR collate hands float32 ones
    (utils/tensor_utils.py:36-53): the reference and the restatement must not care."""
    from oracle import univtg_oracle as O

    cfg = synth.CONFIGS["tiny"]
    sd = synth.make_state_dict(cfg, seed=11)
    inp = synth.make_inputs(cfg, seed=3, ragged=True, batch=4)
    as_bool = dict(inp, src_vid_mask=inp["src_vid_mask"].bool(), src_txt_mask=inp["src_txt_mask"].bool())
    ref_f, ref_b = _ref_out("bool_masks/float"), _ref_out("bool_masks/bool")
    out = _stored(O.forward(sd, cfg, **as_bool))
    for k in OUT_KEYS:
        torch.testing.assert_close(ref_b[k], ref_f[k], rtol=0, atol=0)
        torch.testing.assert_close(out[k], ref_f[k].double(), rtol=2e-5, atol=2e-5)


def test_droppath_scales_match_reference_train_mode():
    """Train mode with droppath: the reference draws floor(keep + U) per sample, per residual branch, in layer order;
    feeding the same draws to the oracle as scales reproduces its output."""
    from oracle import univtg_oracle as O

    cfg = synth.CONFIGS["tiny"]
    sd = synth.make_state_dict(cfg, seed=5)
    inp = synth.make_inputs(cfg, seed=9, ragged=True, batch=6)
    B = inp["src_vid"].shape[0]
    ref = _ref_out("droppath", ("pred_spans", "pred_logits"))  # reference in train mode, droppath 0.3, after manual_seed(77)
    torch.manual_seed(77)
    keep = 0.7
    scales = torch.stack([torch.floor(keep + torch.rand((B, 1, 1))).flatten() / keep for _ in range(2 * cfg["enc_layers"])])
    out = O.forward(sd, cfg, **inp, dp_scale=scales)
    torch.testing.assert_close(out["pred_spans"], ref["pred_spans"].double(), rtol=2e-5, atol=2e-5)
    torch.testing.assert_close(out["pred_logits"], ref["pred_logits"].double(), rtol=2e-5, atol=2e-5)


def test_state_dict_keys_and_shapes_match_reference():
    pins = _pins()
    for name in ("tiny", "cfg1"):
        ref = [(k, tuple(s)) for k, s in pins["state_dict/" + name]]
        assert ref == list(synth.state_dict_shapes(synth.CONFIGS[name]).items())


def test_input_dropout_masks_match_reference_train_mode():
    """Train mode with input dropout (nn.Dropout(0.5) inside every LinearLayer, model/univtg.py:394,401): the reference draws
    one Bernoulli mask per projector layer, video projector first (model/univtg.py:107-108).  Re-drawing the same masks with
    the same torch calls and handing them to the oracle (drop_masks=) reproduces the reference's train-mode output - this pins
    the mask semantics (multiplier 0 or 1/(1-p), applied after the LayerNorm, before the Linear) the CUDA path is tested against."""
    from oracle import univtg_oracle as O

    cfg = synth.CONFIGS["tiny"]
    sd = synth.make_state_dict(cfg, seed=5)
    inp = synth.make_inputs(cfg, seed=9, ragged=True, batch=6)
    tgt = synth.make_targets(inp, seed=10)
    B, Lv, Lt, d = inp["src_vid"].shape[0], inp["src_vid"].shape[1], inp["src_txt"].shape[1], cfg["hidden_dim"]
    ref = _ref_out("input_dropout", ("pred_logits", "pred_spans", "vid_mem_proj", "txt_mem_proj"))  # after manual_seed(31)
    torch.manual_seed(31)
    shapes = [(B, Lv, cfg["v_feat_dim"]), (B, Lv, d), (B, Lt, cfg["t_feat_dim"]), (B, Lt, d)]
    masks = [torch.nn.functional.dropout(torch.ones(s), 0.5, True) for s in shapes]
    out = O.forward(sd, cfg, **inp, drop_masks=masks)
    for k in ref:
        torch.testing.assert_close(_stored(out)[k], ref[k].double(), rtol=2e-5, atol=2e-5)
    _assert_losses(O.criterion(out, tgt), _pins()["input_dropout_loss"])


def test_hl_loss_list_matches_reference():
    """dset_type 'hl' / 'vs': losses = ['labels', 'saliency'] and the targets carry no timestamp / span_labels_nn
    (model/univtg.py:438-439, main/dataset.py:1118-1126)."""
    from oracle import univtg_oracle as O
    from univtg_b200 import build_model

    cfg = synth.CONFIGS["tiny"]
    sd = synth.make_state_dict(cfg, seed=5)
    pins = _pins()["hl"]
    assert pins["criterion_losses"] == ["labels", "saliency"]
    assert build_model(synth.reference_args(cfg, dset_type="hl"))[1].losses == pins["criterion_losses"]
    inp = synth.make_inputs(cfg, seed=9, ragged=True, batch=6)
    full = synth.make_targets(inp, seed=10)
    tgt = {"saliency_scores": full["saliency_scores"], "saliency_pos_labels": full["saliency_pos_labels"],
           "timestamp_mask": full["timestamp_mask"], "timestamp_window": 1 * (full["saliency_scores"] > 0)}
    assert sorted(pins["loss"]) == ["loss_f", "loss_s_inter", "loss_s_intra"]
    loss = O.criterion(O.forward(sd, cfg, **inp), tgt, losses=("labels", "saliency"))
    _assert_losses(loss, pins["loss"])


def decode_case():
    """Fixed model outputs replayed through the reference's evaluation loop: (outputs, timestamps, video mask, durations, Lt)."""
    g = torch.Generator().manual_seed(1234)
    B, Lv, Lt = 5, 23, 7
    lens = [23, 9, 17, 1, 12]
    vmask = torch.zeros(B, Lv)
    for b, n in enumerate(lens):
        vmask[b, :n] = 1
    pred_logits = torch.rand(B, Lv, 1, generator=g)
    pred_logits[0, 3] = pred_logits[0, 5]  # ties: sorted() is stable
    pred_logits[2, 0, 0] = 0.12345  # rounding-sensitive values
    pred_spans = torch.rand(B, Lv, 2, generator=g) * torch.tensor([-1.0, 1.0])
    sal = torch.randn(B, Lv, generator=g)
    ts = ((torch.arange(Lv, dtype=torch.float32) + 0.5) / Lv)[None, :, None].expand(B, Lv, 2).contiguous()
    durs = [150.0, 33.3, 126.0, 2.0, 150.0]
    return {"pred_logits": pred_logits, "pred_spans": pred_spans, "saliency_scores": sal}, ts, vmask, durs, Lt


@pytest.mark.parametrize("sort", [True, False])
def test_decode_restatement_matches_compute_mr_results(sort):
    """Pins oracle/postproc_oracle.decode_mr + saliency_lists to the reference's own evaluation loop: what compute_mr_results
    (main/inference_mr.py:86-193) returned with a stub model / loader that replay the outputs of decode_case()."""
    from oracle import postproc_oracle as PO

    outputs, ts, vmask, durs, _ = decode_case()
    res = _pins()[f"compute_mr_results/sort={sort}"]
    rows = PO.decode_mr(outputs["pred_logits"], outputs["pred_spans"], ts, vmask, durs, sort=sort)
    sal_lists = PO.saliency_lists(outputs["saliency_scores"], vmask)
    assert len(res) == vmask.shape[0]
    for b in range(len(res)):
        assert res[b]["pred_relevant_windows"] == rows[b], b
        assert res[b]["pred_saliency_scores"] == sal_lists[b], b


def test_reference_setup_model_builds_the_plugin(tmp_path):
    """Boundary (SURVEY 8b): main.config.setup_model does importlib.import_module('model.' + opt.model_id).build_model(opt)
    (main/config.py:341-342).  With the one-line shim of INTEGRATION.md on sys.path as model/univtg_b200.py that import builds
    (model, criterion); AdamW (all parameters with requires_grad, main/config.py:348-349) sees the same parameter names / order /
    shapes as setup_model gave the reference for --model_id univtg, and a checkpoint in the reference's layout (DDP prefixes every
    key with 'module.', train_vlp_ddp.py:157-164; setup_model strips it) loads strict=True."""
    ref = _pins()["setup_model"]
    shim = tmp_path / "model"
    shim.mkdir()
    (shim / "univtg_b200.py").write_text("from univtg_b200.plugin import build_model  # noqa: F401\n")
    sys.path.append(str(tmp_path))
    importlib.invalidate_caches()
    try:
        cfg = synth.CONFIGS["tiny"]
        opt = synth.reference_args(cfg, model_id="univtg_b200", gpu_id=0, lr=1e-4, wd=1e-4, lr_warmup=[10], lr_drop=400,
                                   lr_gamma=0.1, resume=None, resume_all=False)
        torch.manual_seed(0)
        m_new, c_new = importlib.import_module("model." + opt.model_id).build_model(opt)
        assert type(m_new).__module__ == "univtg_b200.plugin"
        params = [(n, list(p.shape)) for n, p in m_new.named_parameters() if p.requires_grad]
        assert params == [tuple(x) for x in ref["named_parameters"]]
        assert [s for _, s in params] == ref["optimizer_params"]
        assert c_new.weight_dict == ref["weight_dict"] and c_new.losses == ref["losses"]
        g = torch.Generator().manual_seed(3)
        ckpt = {"module." + k: torch.randn(s, generator=g) for k, s in ref["state_dict"]}
        m_new.load_state_dict({k.replace("module.", ""): v for k, v in ckpt.items()}, strict=True)
        for (k1, v1), (k2, v2) in zip(ckpt.items(), m_new.state_dict().items()):
            assert k1 == "module." + k2 and torch.equal(v1, v2)
    finally:
        sys.path.remove(str(tmp_path))
        sys.modules.pop("model.univtg_b200", None)
        sys.modules.pop("model", None)
