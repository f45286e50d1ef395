#!/usr/bin/env python
"""Writes tests/golden/reference_pins.npz and tests/golden/reference_pins.json: what the unmodified UniVTG reference computes
for the cases of tests/test_oracle_vs_reference.py, tests/test_data_cpu.py and tests/test_postproc.py, so those tests compare
against the reference without needing a copy of it.  Every input is regenerated from the same seeds by the tests.

Usage: python tests/golden/make_reference_pins.py <UniVTG checkout>   (CPU only, a few seconds)
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, REF)

from univtg_b200 import synth  # noqa: E402
from model.univtg import build_model  # noqa: E402  (the reference)

OUT_KEYS = ("pred_logits", "pred_spans", "saliency_scores", "vid_mem_proj", "txt_mem_proj")
FORWARD_CASES = [("tiny", True, None), ("tiny", False, 5), ("cfg1", True, 3)]
VID_STRIDE = 4  # vid_mem_proj is stored at every 4th clip: keeps the fixture small
arrays, pins = {"meta/vid_stride": np.int64(VID_STRIDE)}, {}


def forward_case_key(cfg_name, ragged, batch):
    return f"{cfg_name}_{int(ragged)}_{batch}"


def ref_model(cfg, sd, **over):
    model, crit = build_model(synth.reference_args(cfg, **over))
    model.load_state_dict(sd, strict=True)
    return model, crit


def put(prefix, out, keys=OUT_KEYS):
    for k in keys:
        v = out[k].detach().float()
        arrays[f"{prefix}/{k}"] = (v[:, ::VID_STRIDE] if k == "vid_mem_proj" else v).numpy()


def losses(d):
    return {k: float(v) for k, v in d.items()}


# test_oracle_vs_reference.py::test_forward_and_losses
for cfg_name, ragged, batch in FORWARD_CASES:
    cfg = synth.CONFIGS[cfg_name]
    sd = synth.make_state_dict(cfg, seed=123)
    model, crit = ref_model(cfg, sd)
    model.eval()
    inp = synth.make_inputs(cfg, seed=7, ragged=ragged, batch=batch)
    tgt = synth.make_targets(inp, seed=8)
    with torch.no_grad():
        ref = model(**inp)
        pins["forward_loss/" + forward_case_key(cfg_name, ragged, batch)] = losses(crit(ref, tgt))
    put("forward/" + forward_case_key(cfg_name, ragged, batch), ref)

# ::test_bool_masks_of_the_highlight_path_give_the_same_outputs
cfg = synth.CONFIGS["tiny"]
model, _ = ref_model(cfg, synth.make_state_dict(cfg, seed=11))
model.eval()
inp = synth.make_inputs(cfg, seed=3, ragged=True, batch=4)
with torch.no_grad():
    put("bool_masks/float", model(**inp))
    put("bool_masks/bool", model(**dict(inp, src_vid_mask=inp["src_vid_mask"].bool(), src_txt_mask=inp["src_txt_mask"].bool())))

# ::test_droppath_scales_match_reference_train_mode
model, _ = ref_model(cfg, synth.make_state_dict(cfg, seed=5), droppath=0.3, input_dropout=0.0)
model.train()
inp = synth.make_inputs(cfg, seed=9, ragged=True, batch=6)
torch.manual_seed(77)
put("droppath", model(**inp), ("pred_spans", "pred_logits"))

# ::test_state_dict_keys_and_shapes_match_reference
for name in ("tiny", "cfg1"):
    model, _ = ref_model(synth.CONFIGS[name], synth.make_state_dict(synth.CONFIGS[name]))
    pins["state_dict/" + name] = [[k, list(v.shape)] for k, v in model.state_dict().items()]

# ::test_input_dropout_masks_match_reference_train_mode
model, crit = ref_model(cfg, synth.make_state_dict(cfg, seed=5), droppath=0.0, input_dropout=0.5)
model.train()
inp = synth.make_inputs(cfg, seed=9, ragged=True, batch=6)
tgt = synth.make_targets(inp, seed=10)
torch.manual_seed(31)
ref = model(**inp)
pins["input_dropout_loss"] = losses(crit(ref, tgt))
put("input_dropout", ref, ("pred_logits", "pred_spans", "vid_mem_proj", "txt_mem_proj"))

# ::test_hl_loss_list_matches_reference
model, crit = ref_model(cfg, synth.make_state_dict(cfg, seed=5), dset_type="hl")
model.eval()
full = synth.make_targets(synth.make_inputs(cfg, seed=9, ragged=True, batch=6), seed=10)
tgt = {"saliency_scores": full["saliency_scores"], "saliency_pos_labels": full["saliency_pos_labels"],
       "timestamp_mask": full["timestamp_mask"], "timestamp_window": 1 * (full["saliency_scores"] > 0)}
with torch.no_grad():
    pins["hl"] = {"criterion_losses": list(crit.losses), "loss": losses(crit(model(**synth.make_inputs(cfg, seed=9, ragged=True, batch=6)), tgt))}

# ::test_decode_restatement_matches_compute_mr_results (main.dataset imports h5py / nncore, which the MR loop never calls)
sys.modules.setdefault("h5py", types.ModuleType("h5py"))
nn_, ds, par = types.ModuleType("nncore"), types.ModuleType("nncore.dataset"), types.ModuleType("nncore.parallel")
ds.DATASETS = types.SimpleNamespace(register=lambda *a, **k: (lambda c: c))
par.DataContainer = object
nn_.dataset, nn_.parallel = ds, par
sys.modules.update({"nncore": nn_, "nncore.dataset": ds, "nncore.parallel": par})
import main.inference_mr as M  # noqa: E402
from argparse import Namespace  # noqa: E402

from tests.test_oracle_vs_reference import decode_case  # noqa: E402

for sort in (True, False):
    outputs, ts, vmask, durs, Lt = decode_case()
    B, Lv = vmask.shape

    class FakeModel:
        def eval(self):
            return self

        def __call__(self, **kw):
            return {k: v.clone() for k, v in outputs.items()}

    meta = [{"qid": i, "query": "q", "vid": "v", "duration": durs[i]} for i in range(B)]
    batch = {"query_feat": (torch.zeros(B, Lt, 4), torch.ones(B, Lt)), "video_feat": (torch.zeros(B, Lv, 4), vmask),
             "timestamp": (ts, vmask), "timestamp_window": (torch.zeros(B, Lv),), "span_labels_nn": (torch.zeros(B, Lv, 2),)}
    opt = Namespace(device="cpu", pin_memory=False, span_loss_type="l1", model_id="univtg", eval_mode=None,
                    no_sort_results=not sort, debug=False, round_multiple=0, clip_length=2)
    res, _ = M.compute_mr_results(FakeModel(), [(meta, batch)], opt)
    pins[f"compute_mr_results/sort={sort}"] = [{"pred_relevant_windows": r["pred_relevant_windows"],
                                                "pred_saliency_scores": r["pred_saliency_scores"]} for r in res]

# ::test_reference_setup_model_builds_the_plugin: what main.config.setup_model builds for --model_id univtg
import main.config as C  # noqa: E402


class _CpuDevice(str):  # read both as torch.device(opt.device) and as int(opt.device) >= 0 (main/config.py:344)
    def __int__(self):
        return -1


opt = synth.reference_args(synth.CONFIGS["tiny"], model_id="univtg", device=_CpuDevice("cpu"), gpu_id=0, lr=1e-4, wd=1e-4,
                           lr_warmup=[10], lr_drop=400, lr_gamma=0.1, resume=None, resume_all=False)
m_ref, c_ref, o_ref, s_ref = C.setup_model(opt)
pins["setup_model"] = {"named_parameters": [[n, list(p.shape)] for n, p in m_ref.named_parameters() if p.requires_grad],
                       "optimizer_params": [list(p.shape) for p in o_ref.param_groups[0]["params"]],
                       "weight_dict": c_ref.weight_dict, "losses": list(c_ref.losses),
                       "state_dict": [[k, list(v.shape)] for k, v in m_ref.state_dict().items()]}

# test_postproc.py::test_oracle_nms_matches_live_reference_random
from utils.temporal_nms import temporal_nms  # noqa: E402
from tests.test_postproc import random_nms_cases  # noqa: E402

pins["temporal_nms_random"] = [temporal_nms([list(r) for r in rows], thd, ma) for rows, thd, ma in random_nms_cases()]

# test_data_cpu.py::test_prepared_features_and_collate_match_the_reference_code
import pathlib  # noqa: E402
import tempfile  # noqa: E402

from utils.basic_utils import l2_normalize_np_array  # noqa: E402
from utils.tensor_utils import pad_sequences_1d  # noqa: E402
from tests.test_data_cpu import _fake_corpus  # noqa: E402

with tempfile.TemporaryDirectory() as tmp:
    v_dirs, q_dir, anns = _fake_corpus(pathlib.Path(tmp), seed=5)
    ref_v, ref_q = [], []
    for ann in anns[:6]:
        # main/dataset.py:674-690 + 534-540, re-executed with the reference's helpers
        fl = [l2_normalize_np_array(np.load(os.path.join(d, f"{ann['vid']}.npz"))["features"].astype(np.float32)) for d in v_dirs]
        n = min(len(e) for e in fl)
        v = torch.from_numpy(np.concatenate([e[:n] for e in fl], axis=1))
        st = torch.arange(0, n, 1.0) / n
        ref_v.append(torch.cat([v, torch.stack([st, st + 1.0 / n], dim=1)], dim=1))
        ref_q.append(torch.from_numpy(l2_normalize_np_array(np.load(os.path.join(q_dir, f"{ann['qid']}.npz"))["last_hidden_state"].astype(np.float32))))
    for name, seqs in (("vid", ref_v), ("txt", ref_q)):
        pad, mask = pad_sequences_1d(seqs, dtype=torch.float32, fixed_length=None)
        arrays[f"collate/{name}"] = pad.numpy()
        arrays[f"collate/{name}_mask"] = mask.numpy()

np.savez_compressed(os.path.join(HERE, "reference_pins.npz"), **arrays)
with open(os.path.join(HERE, "reference_pins.json"), "w") as f:
    json.dump(pins, f, indent=0)
print("wrote reference_pins.npz (%d arrays) and reference_pins.json (%d entries)" % (len(arrays), len(pins)))
