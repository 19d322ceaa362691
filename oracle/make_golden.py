"""Generate tests/golden/*.npz from the UNMODIFIED reference (uclanlp/visualbert) — TEST INFRASTRUCTURE.

Runs only in the build container, where the reference is mounted read-only at /root/reference:
    python oracle/make_golden.py
Imports visualbert/pytorch_pretrained_bert/modeling.py with the two shims of SURVEY.md §8c
(stub boto3/botocore; Tensor.cuda -> identity on CPU), loads seeded weights
(visualbert_b200.synthetic.init_state_dict) into the reference's TrainVisualBERTObjective, runs
forward (eval mode, fp32) + backward on seeded synthetic batches and stores outputs, losses and
gradient norms. Weights and inputs are NOT stored: tests regenerate them from the same seeds.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from visualbert_b200 import synthetic  # noqa: E402

REF = "/root/reference/visualbert"

CASES = {
    # BASELINE.json configs[0]: VisualBERT-base 2-layer, batch 4, 36 regions (2048-d) + 20 tokens
    "cfg1_pretraining": dict(model=dict(layers=2, hidden=768, heads=12, inter=3072, vocab=30522), Dv=2048,
                             head="pretraining", batch=dict(B=4, T=20, V=36)),
    "small_ragged_pretraining": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64,
                                     head="pretraining", batch=dict(B=3, T=12, V=7, ragged=True, nlvr_types=True)),
    "small_vqa": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="vqa",
                      batch=dict(B=3, T=12, V=7, ragged=True)),
    "small_nlvr": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="nlvr",
                       batch=dict(B=4, T=10, V=8, ragged=True, nlvr_types=True)),
    "small_multichoice": dict(model=dict(layers=1, hidden=128, heads=2, inter=512, vocab=512), Dv=64,
                              head="multichoice", batch=dict(B=2, T=9, V=5, ragged=True, choices=4)),
    # SURVEY.md §8f rank 4, the VCR-only branches of the reference
    "small_vcr_alignment": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="multichoice",
                                batch=dict(B=2, T=9, V=5, ragged=True, choices=4, alignment=3)),
    "small_bypass_nlvr": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="nlvr",
                              batch=dict(B=4, T=10, V=8, ragged=True, nlvr_types=True), flags=dict(bypass_transformer=True)),
    "small_attention_weights": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="nlvr",
                                    batch=dict(B=3, T=10, V=6, ragged=True), flags=dict(output_attention_weights=True)),
    # the two remaining task heads of TrainVisualBERTObjective (M.py:1527-1554, 1568-1598)
    "small_vqa_advanced": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="vqa_advanced",
                               batch=dict(B=3, T=12, V=7, ragged=True)),
    "small_flickr": dict(model=dict(layers=2, hidden=128, heads=2, inter=512, vocab=512), Dv=64, head="flickr",
                         batch=dict(B=3, T=12, V=7, ragged=True)),
    "base3_ragged_pretraining": dict(model=dict(layers=3, hidden=768, heads=12, inter=3072, vocab=2048), Dv=2048,
                                     head="pretraining", batch=dict(B=5, T=33, V=19, ragged=True)),
}


def import_reference():
    for name in ("boto3", "botocore", "botocore.exceptions"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["botocore.exceptions"].ClientError = Exception
    sys.path.insert(0, REF)
    torch.Tensor.cuda = lambda self, *a, **k: self  # M.py:1238,1247 hard-code .cuda()
    from pytorch_pretrained_bert import modeling
    return modeling


def build_case(name):
    c = CASES[name]
    m = c["model"]
    cfg = synthetic.bert_config_dict(m["layers"], m["hidden"], m["heads"], m["inter"], vocab=m["vocab"])
    sd = synthetic.init_state_dict(cfg, c["head"], c["Dv"], seed=0,
                                   bypass_transformer=c.get("flags", {}).get("bypass_transformer", False))
    b = dict(c["batch"])
    batch = synthetic.make_batch(Dv=c["Dv"], head=c["head"], seed=1234, vocab=m["vocab"], **b)
    return cfg, sd, batch, c


def subsample(t, n=4096):
    flat = t.detach().reshape(-1)
    step = max(1, flat.numel() // n)
    return flat[::step][:n].double().numpy()


def main():
    M = import_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    if "--only-wrapper" in sys.argv:
        return make_wrapper_golden(out_dir)
    make_bert_adam_golden(out_dir)
    if "--only-adam" in sys.argv:
        return
    only = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--case=")]
    for name in CASES:
        if only and name not in only:
            continue
        cfg, sd, batch, c = build_case(name)
        model = M.TrainVisualBERTObjective(M.BertConfig.from_dict(cfg), c["head"], visual_embedding_dim=c["Dv"],
                                           **c.get("flags", {}))
        missing = model.load_state_dict(sd, strict=False)
        assert set(missing.missing_keys) <= {"cls.predictions.decoder.weight"}, missing
        assert not missing.unexpected_keys, missing
        model.eval()
        out = model(**batch)
        if c.get("flags", {}).get("output_attention_weights"):
            # analysis mode: the reference returns ONLY {"attention_weights": [L x [B, A, S, S]], "loss": None} (M.py:1430-1444)
            assert out["loss"] is None and set(out) == {"attention_weights", "loss"}
            rec = {f"attn{i}_sub": subsample(w) for i, w in enumerate(out["attention_weights"])}
            rec["attn_shape"] = np.array(out["attention_weights"][0].shape)
            np.savez_compressed(os.path.join(out_dir, name + ".npz"), **rec)
            print(f"{name}: {len(out['attention_weights'])} attention maps {tuple(out['attention_weights'][0].shape)} -> {name}.npz")
            continue
        loss = out["loss"]
        loss.backward()
        rec = {"loss": np.float64(loss.item())}
        for k in ("masked_lm_loss", "next_sentence_loss"):
            if k in out:
                rec[k] = np.float64(out[k].item())
        for k in ("accuracy", "upperbound_accuracy", "entity_num"):
            if k in out and out[k] is not None:
                rec[k] = np.float64(float(out[k]))
        logits = out["logits"] if "logits" in out else loss.detach().reshape(1)  # the flickr head returns no logits
        rec["logits_sub"] = subsample(logits)
        rec["logits_stats"] = np.array([logits.double().mean().item(), logits.double().std().item(),
                                        logits.double().abs().max().item()])
        if "seq_relationship_score" in out:
            rec["nsp"] = out["seq_relationship_score"].detach().double().numpy()
        if c.get("flags", {}).get("bypass_transformer"):
            # the bypass model refuses output_all_encoded_layers (M.py:1300): capture the final hidden state with a hook
            keep = {}
            hook = model.bert.additional_layer.register_forward_hook(lambda m, i, o: keep.__setitem__("y", o))
            with torch.no_grad():
                model(**batch)
            hook.remove()
            rec[f"hidden{cfg['num_hidden_layers'] - 1}_sub"] = subsample(keep["y"])
            rec["pooled"] = model.bert.pooler(keep["y"]).detach().double().numpy()
        else:
            # hidden states (second forward with output_all_encoded_layers)
            with torch.no_grad():
                enc = model(**{**batch, "output_all_encoded_layers": True})
            for i, h in enumerate(enc["sequence_output"]):
                rec[f"hidden{i}_sub"] = subsample(h)
            rec["pooled"] = enc["pooled_output"].double().numpy()
        names, norms = [], []
        for k, p in model.named_parameters():
            if p.grad is not None:
                names.append(k)
                norms.append(p.grad.double().norm().item())
        rec["grad_names"] = np.array(names)
        rec["grad_norms"] = np.array(norms)
        for k in ("bert.encoder.layer.0.attention.self.query.weight", "bert.encoder.layer.0.output.dense.weight",
                  "bert.embeddings.projection.weight", "bert.embeddings.LayerNorm.weight",
                  "bert.encoder.layer.0.intermediate.dense.bias"):
            rec["grad_sub::" + k] = subsample(dict(model.named_parameters())[k].grad)
        np.savez_compressed(os.path.join(out_dir, name + ".npz"), **rec)
        print(f"{name}: loss={loss.item():.6f} logits{tuple(logits.shape)} -> {name}.npz")
    if not only:
        make_wrapper_golden(out_dir)


WRAPPER_CASES = ("small_nlvr", "small_vqa", "small_ragged_pretraining")
MODEL_DIR = "<bert_model_dir>"   # stands for the model directory the wrapper was handed


def _install_wrapper_standins(objective_cls):
    """allennlp.* names model.py:11-18 imports (AllenNLP 0.8 is not installable offline, SURVEY.md §8c); only Model (an
    nn.Module with a `register` decorator and a vocab) and the two metrics the wrapper instantiates need behaviour.
    pytorch_pretrained_bert.modeling serves `objective_cls`: the one-line import swap of INTEGRATION.md §1 (model.py:20).
    Returns the sys.modules entries it replaced."""

    class Model(torch.nn.Module):
        def __init__(self, vocab=None):
            super().__init__()
            self.vocab = vocab

        @classmethod
        def register(cls, name):
            return lambda klass: klass

    class CategoricalAccuracy:
        def __init__(self):
            self.correct, self.total = 0.0, 0.0

        def __call__(self, logits, labels):
            self.correct += (logits.argmax(-1).view(-1) == labels.view(-1)).float().sum().item()
            self.total += labels.numel()

        def get_metric(self, reset=False):
            v = self.correct / max(self.total, 1.0)
            if reset:
                self.correct = self.total = 0.0
            return v

    class Average:
        def __init__(self):
            self.s, self.n = 0.0, 0

        def __call__(self, v):
            self.s += float(v); self.n += 1

        def get_metric(self, reset=False):
            v = self.s / max(self.n, 1)
            if reset:
                self.s, self.n = 0.0, 0
            return v

    anything = type("Anything", (), {})
    mods = {
        "allennlp": {}, "allennlp.data": {}, "allennlp.data.vocabulary": dict(Vocabulary=anything),
        "allennlp.models": {}, "allennlp.models.model": dict(Model=Model),
        "allennlp.modules": dict(TextFieldEmbedder=anything, Seq2SeqEncoder=anything, FeedForward=anything,
                                 InputVariationalDropout=anything, TimeDistributed=anything),
        "allennlp.training": {}, "allennlp.training.metrics": dict(CategoricalAccuracy=CategoricalAccuracy, Average=Average),
        "allennlp.modules.matrix_attention": dict(BilinearMatrixAttention=anything),
        "allennlp.nn": dict(InitializerApplicator=anything),
        "allennlp.nn.util": dict(masked_softmax=None, weighted_sum=None, replace_masked_values=None),
        "pytorch_pretrained_bert": {},
        "pytorch_pretrained_bert.modeling": dict(TrainVisualBERTObjective=objective_cls, BertForMultipleChoice=anything),
        "pytorch_pretrained_bert.file_utils": dict(PYTORCH_PRETRAINED_BERT_CACHE="pretrained_cache"),
    }
    saved = {name: sys.modules.get(name) for name in mods}
    for name, attrs in mods.items():
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
    return saved


def make_wrapper_golden(out_dir):
    """The reference's AllenNLP wrapper `visualbert/models/model.py:191-306` (VisualBERTFixedImageEmbedding), executed
    unmodified on visualbert_b200.TrainVisualBERTObjective, with the oracle's (sequence_output, pooled_output) standing
    in for the CUDA encoder. Records every call the wrapper makes into the objective (from_pretrained arguments,
    special_intialize, the forward keywords with their tensors) and what the wrapper returns (output keys, loss,
    accuracy metric): tests/test_wrapper_dropin_cpu.py replays the calls and checks the results."""
    import json
    import tempfile

    import vb_oracle
    import visualbert_b200
    from visualbert_b200 import BertConfig
    from visualbert_b200.modeling import BertEmbeddingsWithVisualEmbedding

    calls = []

    class RecordingObjective(visualbert_b200.TrainVisualBERTObjective):
        @classmethod
        def from_pretrained(cls, *args, **kwargs):
            calls.append(dict(name="from_pretrained", args=args, kwargs=kwargs))
            return super().from_pretrained(*args, **kwargs)

        def forward(self, **kwargs):
            calls.append(dict(name="forward", kwargs=kwargs))
            return super().forward(**kwargs)

    special_init = BertEmbeddingsWithVisualEmbedding.special_intialize

    def recording_special_init(self, *args, **kwargs):
        calls.append(dict(name="special_intialize", args=args, kwargs=kwargs))
        return special_init(self, *args, **kwargs)

    saved = _install_wrapper_standins(RecordingObjective)
    BertEmbeddingsWithVisualEmbedding.special_intialize = recording_special_init
    try:
        path = os.path.join(REF, "models", "model.py")
        ns = {"__name__": "reference_models_model"}
        exec(compile(open(path).read(), path, "exec"), ns)
        for name in WRAPPER_CASES:
            cfg, sd, batch, c = build_case(name)
            calls.clear()
            with tempfile.TemporaryDirectory() as model_dir:
                with open(os.path.join(model_dir, "bert_config.json"), "w") as f:
                    f.write(BertConfig.from_dict(cfg).to_json_string())
                m = ns["VisualBERTFixedImageEmbedding"](vocab=None, bert_model_name=model_dir, training_head_type=c["head"],
                                                        visual_embedding_dim=c["Dv"], random_initialize=True,
                                                        special_visual_initialize=True)
                calls[0]["args"] = [MODEL_DIR if a == model_dir else a for a in calls[0]["args"]]
            res = m.bert.load_state_dict(sd, strict=False)
            assert set(res.missing_keys) <= {"cls.predictions.decoder.weight"} and not res.unexpected_keys, res
            m.eval()
            kw = {k: v for k, v in batch.items() if k != "position_embeddings_visual"}
            with torch.no_grad():
                ref = vb_oracle.objective(sd, cfg, c["head"], **kw)
            m.bert.bert.forward = lambda *a, **k: (ref["sequence_output"], ref["pooled_output"])
            image_dim = batch["image_mask"].sum(-1)   # the wrapper rebuilds image_mask from the region count (model.py:262-268)
            out = m(bert_input_ids=batch["input_ids"], bert_input_mask=batch["input_mask"],
                    bert_input_type_ids=batch["token_type_ids"], image_dim_variable=image_dim,
                    image_feat_variable=batch["visual_embeddings"], visual_embeddings_type=batch.get("visual_embeddings_type"),
                    label=batch.get("label"), masked_lm_labels=batch.get("masked_lm_labels"),
                    is_random_next=batch.get("is_random_next"))
            assert [x["name"] for x in calls] == ["from_pretrained", "special_intialize", "forward"], calls
            rec = {}
            fwd = calls[2]["kwargs"]
            for k, v in fwd.items():
                if torch.is_tensor(v):
                    rec["forward::" + k] = v.detach().numpy()
            meta = dict(
                from_pretrained=dict(args=calls[0]["args"], kwargs=calls[0]["kwargs"]),
                special_intialize=dict(args=calls[1]["args"], kwargs=calls[1]["kwargs"]),
                forward_values={k: v for k, v in fwd.items() if not torch.is_tensor(v)},
                output_keys=sorted(out.keys()), loss=out["loss"].item(), accuracy=m.get_metrics(reset=True)["accuracy"])
            rec["calls"] = np.array(json.dumps(meta, sort_keys=True))
            np.savez_compressed(os.path.join(out_dir, f"wrapper_{name}.npz"), **rec)
            print(f"wrapper_{name}: loss={meta['loss']:.6f} accuracy={meta['accuracy']:.4f} -> wrapper_{name}.npz")
    finally:
        BertEmbeddingsWithVisualEmbedding.special_intialize = special_init
        for name, mod in saved.items():
            if mod is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = mod


def make_bert_adam_golden(out_dir):
    """Reference BertAdam (opt.py:185-304), 4 steps on seeded tensors: two parameter groups (decay / no decay) like
    model_wrapper.py:106-111, warmup_linear schedule; gradients large enough that the per-parameter clip engages on
    some tensors and not on others. Stores parameters and both moments after every step."""
    from pytorch_pretrained_bert.optimization import BertAdam
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import adam_util
    init, grads = adam_util.scenario()
    shapes = adam_util.SHAPES
    params = [torch.nn.Parameter(t.clone()) for t in init]
    opt = BertAdam([{"params": params[:3], "weight_decay": 0.01}, {"params": params[3:], "weight_decay": 0.0}],
                   **adam_util.HYPER)
    rec = {"shapes": np.array([len(s) for s in shapes])}
    for step in range(4):
        for i, p in enumerate(params):
            p.grad = grads[step][i].clone()
        opt.step()
        for i, p in enumerate(params):
            rec[f"p{i}_s{step}"] = p.detach().numpy().copy()
            rec[f"m{i}_s{step}"] = opt.state[p]["next_m"].numpy().copy()
            rec[f"v{i}_s{step}"] = opt.state[p]["next_v"].numpy().copy()
    np.savez_compressed(os.path.join(out_dir, "bert_adam.npz"), **rec)
    print("bert_adam: 4 steps x", len(params), "tensors")


if __name__ == "__main__":
    main()
