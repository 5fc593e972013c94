"""Drop-in proof (SURVEY.md §8b, VERDICT r1 item 8): the REFERENCE's own Importer -> Trainer.build_model /
train_model -> Evaluator -> infer_* flow (scripts/pykg2vec_train.py:11-23) runs unchanged with the B200
classes patched into Importer.modelMap, and the checkpoint shipped with the reference loads through
Trainer.load_model into the mirror.

BASELINE.json configs[0] (`pykg2vec-train -mn TransE -ds umls`, CPU plumbing) is served by the UNMODIFIED
reference classes — the product has no CPU path by design (a CPU fallback would void every parity claim);
test_config1_cli_flow_reference_cpu runs exactly that flow here on the UMLS-shaped synthetic dataset, and
the -m gpu tests run the same flow through the B200 classes with `-device cuda`.

Needs oracle/_ref (the unmodified reference, installed there by build() from a checkout of it: oracle/ref_install.py)."""
import os
import sys

import numpy as np
import pytest
import torch

import dropin_util as du
from baseline import ref_loader

needs_ref = pytest.mark.skipif(not ref_loader.available(), reason="oracle/_ref not installed (build() installs it from a checkout of the reference)")
CFG1 = ["-mn", "TransE", "-l", "2", "-ts", "1", "-tn", "50", "-npg", "1"]   # defaults otherwise: d=50, B=128, adam, L1, margin 0.8


def _flow(tmp_path, monkeypatch, extra, importer_cls=None):
    ref_loader.load()
    ds = du.write_dataset(str(tmp_path / "data"))
    monkeypatch.chdir(tmp_path)   # the reference creates ../dataset relative to the CWD (datasets.py:84-86)
    return du.run_cli_flow(CFG1 + ["-ds", "syn", "-dsp", ds] + extra, importer_cls)


@needs_ref
def test_config1_cli_flow_reference_cpu(tmp_path, monkeypatch):
    """configs[0]: the reference CLI flow on CPU with its own classes (what `-device cpu` keeps using)."""
    tr = _flow(tmp_path, monkeypatch, ["-device", "cpu"])
    assert type(tr.model).__module__ == "pykg2vec.models.pairwise"
    assert len(tr.training_results) == 2 and np.isfinite(tr.training_results[-1][1])
    mc = tr.evaluator.metric_calculator
    assert len(mc.mr) >= 1 and all(np.isfinite(v) for v in mc.mr.values())


@needs_ref
@pytest.mark.gpu
@pytest.mark.parametrize("model,extra", [("TransE", []), ("DistMult", []), ("Complex", []),
                                         ("RotatE", ["-ngr", "4"]), ("TransH", []), ("Rescal", ["-k", "16"])])
def test_reference_trainer_drives_b200_classes(tmp_path, monkeypatch, model, extra):
    """the unmodified reference Trainer / Generator / Evaluator with the B200 model classes, -device cuda"""
    B200Importer = du.b200_importer_class()
    ref_loader.load()
    ds = du.write_dataset(str(tmp_path / "data"))
    monkeypatch.chdir(tmp_path)
    argv = ["-mn", model, "-l", "2", "-ts", "1", "-tn", "50", "-npg", "1", "-ds", "syn", "-dsp", ds, "-device", "cuda"] + extra
    tr = du.run_cli_flow(argv, B200Importer)
    assert type(tr.model).__module__.startswith("pykg2vec_b200.")
    assert next(tr.model.parameters()).is_cuda
    assert len(tr.training_results) == 2 and np.isfinite(tr.training_results[-1][1])
    # loss goes down on the training set between the two epochs (the kernels really train the tables)
    assert tr.training_results[1][1] < tr.training_results[0][1]
    mc = tr.evaluator.metric_calculator
    assert all(np.isfinite(v) for v in mc.mr.values())
    # Trainer.infer_* (trainer.py:330-386) through the reference's Evaluator.test_*_rank
    assert len(tr.infer_tails(1, 10, topk=5)) == 5
    assert len(tr.infer_heads(10, 20, topk=5)) == 5
    # the reference's ranks over the B200 forward == the batched rank kernel on the same weights
    from pykg2vec_b200.evaluator import Evaluator as B200Evaluator
    ev = B200Evaluator(tr.model, tr.config)
    ev.full_test(epoch=0)
    ref_mc = tr.evaluator.metric_calculator
    tr.model.eval()
    with torch.no_grad():
        tr.evaluator.full_test(0)
    got = np.stack([ev.metric_calculator.rank_tail, ev.metric_calculator.rank_head], axis=1)
    want = np.stack([ref_mc.rank_tail, ref_mc.rank_head], axis=1)
    # identical except where torch.topk's order under exact ties decides (count them: must be rare)
    assert (got != want).mean() < 0.02, (got != want).mean()


@needs_ref
@pytest.mark.gpu
def test_pretrained_checkpoint_loads_through_trainer_load_model(tmp_path, monkeypatch):
    """examples/pretrained/TransE/model.vec.pt + config.npy (FB15k, d=50, L1) through the reference's
    Trainer.load_model (trainer.py:399-419) with Importer resolving to the B200 TransE; scores equal the
    reference class's on the same checkpoint."""
    ref_loader.load()
    import pykg2vec.utils.trainer as ref_trainer
    from pykg2vec.models.pairwise import TransE as RefTransE
    B200Importer = du.b200_importer_class()
    monkeypatch.setattr(ref_trainer, "Importer", B200Importer)
    ckpt = os.path.join(ref_loader.REF_DIR, "examples", "pretrained", "TransE")
    tr = object.__new__(ref_trainer.Trainer)
    import types
    tr.config = types.SimpleNamespace(load_from_data=ckpt)
    tr.model = None
    tr.load_model(ckpt)
    m = tr.model
    assert type(m).__module__ == "pykg2vec_b200.pairwise" and m.ent_embeddings.weight.shape == (14951, 50)
    m = m.cuda()
    sd = torch.load(os.path.join(ckpt, "model.vec.pt"), map_location="cpu")
    ref = RefTransE(tot_entity=14951, tot_relation=1345, hidden_size=50, l1_flag=True)
    ref.load_state_dict(sd)
    rng = np.random.RandomState(0)
    h, r, t = (torch.from_numpy(rng.randint(n, size=4096)) for n in (14951, 1345, 14951))
    with torch.no_grad():
        want = ref(h, r, t).numpy()
        got = m(h.cuda(), r.cuda(), t.cuda()).cpu().numpy()
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-2 * np.abs(want).max())
    assert err.max() < 1e-4, err.max()


@pytest.mark.gpu
def test_pretrained_checkpoint_scores_match_reference_golden():
    """The same checkpoint without the reference installed (tests/golden/make_golden_dropin.py): the B200
    TransE built from the constructor arguments the reference's Trainer.load_model passed takes a state_dict
    in the checkpoint's layout and shape (the rows 1,024 seeded triples touch, the rest zero) and scores
    those triples as the reference class did."""
    import pykg2vec_b200
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pretrained_transe_fb15k_checkpoint.npz"))
    n_ent, n_rel, d = int(g["tot_entity"]), int(g["tot_relation"]), int(g["hidden_size"])
    m = pykg2vec_b200.import_model(str(g["model_name"]))(tot_entity=n_ent, tot_relation=n_rel, hidden_size=d,
                                                         l1_flag=bool(g["l1_flag"]))
    assert type(m).__module__ == "pykg2vec_b200.pairwise"
    ent, rel = torch.zeros(n_ent, d), torch.zeros(n_rel, d)
    ent[torch.from_numpy(g["ent_ids"])] = torch.from_numpy(g["ent_rows"])
    rel[torch.from_numpy(g["rel_ids"])] = torch.from_numpy(g["rel_rows"])
    m.load_state_dict({"ent_embeddings.weight": ent, "rel_embeddings.weight": rel})
    m = m.cuda().eval()
    h, r, t = (torch.from_numpy(g[k]).cuda() for k in ("h", "r", "t"))
    with torch.no_grad():
        got = m(h, r, t).cpu().numpy()
    want = g["scores"]
    err = np.abs(got - want) / np.maximum(np.abs(want), 1e-2 * np.abs(want).max())
    assert err.max() < 1e-4, err.max()
