#!/usr/bin/env python
"""Golden fixture of the pretrained-checkpoint drop-in check, by RUNNING THE REFERENCE ITSELF.

Needs a checkout of the reference (see make_golden.py):   python tests/golden/make_golden_dropin.py

The FB15k TransE checkpoint shipped with the reference (examples/pretrained/TransE: model.vec.pt +
config.npy, 14,951 x 50 entity and 1,345 x 50 relation rows, L1) is loaded through the reference's own
Trainer.load_model (pykg2vec/utils/trainer.py:399-419) and scores 1,024 seeded random triples.  The whole
checkpoint is 3.2 MB, so only the rows those triples touch are stored, with their row ids, next to the
constructor arguments load_model passed and the reference's scores.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402  (installs the import stubs and the reference on sys.path)
import pykg2vec.utils.trainer as ref_trainer  # noqa: E402

OUT = os.path.join(HERE, "pretrained_transe_fb15k_checkpoint.npz")


def main(n=1024, seed=0):
    ckpt = os.path.join(mg.REF, "examples", "pretrained", "TransE")
    tr = object.__new__(ref_trainer.Trainer)
    tr.config = types.SimpleNamespace(load_from_data=ckpt)
    tr.model = None
    tr.load_model(ckpt)
    cfg, m = tr.config, tr.model
    ent = m.ent_embeddings.weight.detach().numpy()
    rel = m.rel_embeddings.weight.detach().numpy()
    rng = np.random.RandomState(seed)
    h, r, t = (rng.randint(k, size=n).astype(np.int64) for k in (cfg.tot_entity, cfg.tot_relation, cfg.tot_entity))
    with torch.no_grad():
        scores = m(torch.from_numpy(h), torch.from_numpy(r), torch.from_numpy(t)).numpy().copy()
    ent_ids = np.unique(np.concatenate([h, t]))
    rel_ids = np.unique(r)
    np.savez_compressed(OUT, model_name=np.asarray(cfg.model_name), tot_entity=np.asarray(cfg.tot_entity),
                        tot_relation=np.asarray(cfg.tot_relation), hidden_size=np.asarray(cfg.hidden_size),
                        l1_flag=np.asarray(bool(cfg.l1_flag)), ent_ids=ent_ids, ent_rows=ent[ent_ids],
                        rel_ids=rel_ids, rel_rows=rel[rel_ids], h=h, r=r, t=t, scores=scores)
    print("wrote %s (%d bytes), %d entity rows, %d relation rows"
          % (OUT, os.path.getsize(OUT), len(ent_ids), len(rel_ids)))


if __name__ == "__main__":
    torch.set_num_threads(1)
    main()
