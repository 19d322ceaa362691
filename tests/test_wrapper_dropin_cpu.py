"""Wrapper-level drop-in proof (VERDICT r1 missing #5): the reference's own AllenNLP model wrapper
`visualbert/models/model.py:191-306` (VisualBERTFixedImageEmbedding) drives TrainVisualBERTObjective after the one-line
import swap INTEGRATION.md §1 prescribes (`model.py:20`).

oracle/make_golden.py ran the unmodified wrapper on this package and recorded, in tests/golden/wrapper_<case>.npz, every
call it made into the objective: from_pretrained with the reference's keyword list, special_intialize, and the
13-keyword forward call with its tensors (image_mask rebuilt by the wrapper from the region count, model.py:262-268);
plus what the wrapper returned. This test replays those calls, for the nlvr / vqa / pretraining heads, and checks the
state_dict keys the training wrapper groups and restores by name (`model_wrapper.py:106-111, 201-221`), the loss
against the reference golden, the output keys the wrapper handed on and its accuracy metric. The CUDA encoder cannot
run without a GPU, so `bert.forward` is served by the oracle's encoder — the same arrangement as
tests/test_heads_cpu.py."""
import json
import os

import numpy as np
import pytest
import torch

import golden_util
import vb_oracle

MODEL_DIR = "<bert_model_dir>"   # oracle/make_golden.py: stands for the model directory the wrapper was handed


@pytest.mark.parametrize("case", ["small_nlvr", "small_vqa", "small_ragged_pretraining"])
def test_reference_allennlp_wrapper_runs_on_the_swapped_objective(case, tmp_path):
    from visualbert_b200 import BertConfig, TrainVisualBERTObjective
    cfg, sd, batch, c, gold = golden_util.load(case)
    rec = np.load(os.path.join(golden_util.GOLDEN_DIR, f"wrapper_{case}.npz"), allow_pickle=False)
    calls = json.loads(str(rec["calls"]))
    (tmp_path / "bert_config.json").write_text(BertConfig.from_dict(cfg).to_json_string())
    ctor = calls["from_pretrained"]
    m = TrainVisualBERTObjective.from_pretrained(*[str(tmp_path) if a == MODEL_DIR else a for a in ctor["args"]],
                                                 **ctor["kwargs"])
    m.bert.embeddings.special_intialize(*calls["special_intialize"]["args"], **calls["special_intialize"]["kwargs"])
    # names the training wrapper relies on (model_wrapper.py:106-111 grouping, 209-221 restore-by-name); it holds the
    # objective as `.bert`
    keys = set(m.state_dict().keys())
    assert "bert.encoder.layer.0.attention.self.query.weight" in keys and "bert.pooler.dense.weight" in keys
    assert any(k.endswith("LayerNorm.weight") for k in keys) and any("bias" in k for k in keys)
    res = m.load_state_dict(sd, strict=False)
    assert set(res.missing_keys) <= {"cls.predictions.decoder.weight"} and not res.unexpected_keys
    m.eval()
    # CPU stand-in for the CUDA encoder: the oracle's (sequence_output, pooled_output) for this batch
    kw = {k: v for k, v in batch.items() if k != "position_embeddings_visual"}
    with torch.no_grad():
        ref = vb_oracle.objective(sd, cfg, c["head"], **kw)
    m.bert.forward = lambda *a, **k: (ref["sequence_output"], ref["pooled_output"])
    fwd = {k[len("forward::"):]: torch.from_numpy(rec[k]) for k in rec.files if k.startswith("forward::")}
    fwd.update(calls["forward_values"])
    out = m(**fwd)
    assert abs(out["loss"].item() - float(gold["loss"])) <= 2e-5 * abs(float(gold["loss"]))
    assert set(out.keys()) | {"cnn_regularization_loss"} == set(calls["output_keys"])
    # the wrapper's metric (model.py:290-306): argmax accuracy of the logits for nlvr, the head's accuracy for vqa
    if c["head"] == "nlvr":
        accuracy = (out["logits"].argmax(-1) == fwd["label"]).float().mean().item()
    elif c["head"] == "vqa":
        accuracy = out["accuracy"].item()
    else:
        accuracy = 0.0
    assert abs(accuracy - calls["accuracy"]) <= 1e-6
