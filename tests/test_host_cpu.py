"""CPU tests (-m "not gpu") of the host logic and of the C-ABI library itself: it loads,
exports every symbol include/kge_b200.h declares, and the product refuses to run without
CUDA instead of falling back."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_loads_and_exports_every_declared_symbol():
    from pykg2vec_b200 import _lib, build
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "kge_b200.h")).read()
    declared = set(re.findall(r"\b(kge_[a-z0-9_]+)\s*\(", header))
    declared -= {"kge_model_t"}
    assert declared, "no declarations parsed"
    for sym in sorted(declared):
        assert hasattr(lib, sym), "libkge_b200.so does not export %s" % sym
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    L = _lib.lib()
    assert L.kge_abi_version() == _lib.ABI_VERSION
    assert b"sm_100a" in L.kge_version()
    # loading the library touches no CUDA state; checked in a fresh interpreter, because GPU tests run
    # earlier in this process launch kernels through the same loaded library
    import subprocess
    import sys
    code = "import sys; sys.path.insert(0, sys.argv[1]); from pykg2vec_b200 import _lib; print(_lib.lib().kge_launch_count())"
    res = subprocess.run([sys.executable, "-c", code, ROOT], capture_output=True, text=True, check=True)
    assert int(res.stdout.split()[-1]) == 0


def test_sass_shows_the_blackwell_instructions_the_design_claims():
    """DESIGN.md §4b / §4: the shipped library's SASS (cuobjdump, no GPU needed) holds the tcgen05 tensor-core
    path (UTCHMMA = tcgen05.mma kind::f16, LDTM = tcgen05.ld, UTCBAR = tcgen05.commit, TMEM allocation), TMA
    tensor loads incl. the cluster-multicast form, cp.async staging and the 128-bit exchange of the sparse
    optimizer — and no Hopper-style warpgroup MMA."""
    import shutil
    import subprocess
    from pykg2vec_b200 import build
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        import pytest
        pytest.skip("cuobjdump not installed")
    lib_path = build.build()
    objdir = os.path.join(os.path.dirname(lib_path), "obj")

    def sass_of(tu):   # per translation unit: the whole library takes cuobjdump minutes
        obj = os.path.join(objdir, tu + ".o")
        assert os.path.exists(obj), obj
        return subprocess.run([exe, "-sass", obj], capture_output=True, text=True, check=True).stdout

    tc, tiled, score, train = sass_of("kge_rank_tc"), sass_of("kge_rank_tiled"), sass_of("kge_score"), sass_of("kge_train")
    count = lambda text, pat: len(re.findall(pat, text))
    assert "sm_100a" in tc
    assert count(tc, r"\bUTCHMMA\b") >= 12       # three passes per k-step, SS and TS forms, two cluster variants
    assert count(tc, r"\bLDTM\b") >= 1 and count(tc, r"\bUTCBAR\b") >= 1 and count(tc, r"\bUTCATOMSWS\b") >= 1
    assert count(tc, r"\bUTMALDG\.2D\b") >= 8 and count(tc, r"UTMALDG\.2D\.MULTICAST") >= 1
    assert count(tiled, r"\bUTMALDG\.2D\b") >= 8   # the fp32 sweep's operand tiles arrive by TMA too
    assert count(score, r"\bLDGSTS\b") >= 8        # cp.async ring of the staged gather+score kernel
    assert count(train, r"ATOMG\.E\.EXCH\.128") >= 1   # atom.exch.b128 of the sparse optimizer
    assert count(tc, r"\bHGMMA\b") == 0 and count(tiled, r"\bHGMMA\b") == 0


def test_struct_layout_matches_header():
    from pykg2vec_b200 import _lib
    # int32 x4, float x2, int64 x2, 16 pointers
    assert ctypes.sizeof(_lib.KgeModel) == 4 * 4 + 2 * 4 + 2 * 8 + 16 * 8
    import oracle
    assert ctypes.sizeof(oracle.KgeModel) == ctypes.sizeof(_lib.KgeModel)
    assert _lib.MODEL_IDS == oracle.MODEL_IDS


def test_no_cpu_fallback():
    import pykg2vec_b200
    from pykg2vec_b200 import _lib
    m = pykg2vec_b200.import_model("distmult")(tot_entity=10, tot_relation=3, hidden_size=8, lmbda=0.1)
    ids = torch.tensor([1, 2])
    with pytest.raises(_lib.KgeError):
        m(ids, ids, ids)
    with pytest.raises(_lib.KgeError):
        m.get_reg(ids, ids, ids)
    with pytest.raises(_lib.KgeError):
        m.loss(torch.zeros(4), torch.ones(4))


def test_model_surface_matches_reference_contract():
    """constructor kwargs / error strings / state_dict keys (SURVEY.md §8b)."""
    import pykg2vec_b200
    from pykg2vec_b200.KGMeta import TrainingStrategy
    with pytest.raises(ValueError):
        pykg2vec_b200.import_model("nope")
    cls = pykg2vec_b200.import_model("TransE")
    with pytest.raises(Exception, match="hyperparameter l1_flag not found!"):
        cls(tot_entity=5, tot_relation=2, hidden_size=4)
    m = cls(tot_entity=5, tot_relation=2, hidden_size=4, l1_flag=True, extra_ignored=1)
    assert list(m.state_dict()) == ["ent_embeddings.weight", "rel_embeddings.weight"]
    assert m.model_name == "transe" and m.training_strategy == TrainingStrategy.PAIRWISE_BASED
    assert [p.name for p in m.parameter_list] == ["ent_embedding", "rel_embedding"]
    assert m.get_reg(None, None, None) == 0.0
    c = pykg2vec_b200.import_model("complex")(tot_entity=5, tot_relation=2, hidden_size=4, lmbda=0.1)
    assert list(c.state_dict()) == ["ent_embeddings_real.weight", "ent_embeddings_img.weight",
                                    "rel_embeddings_real.weight", "rel_embeddings_img.weight"]
    r = pykg2vec_b200.import_model("rotate")(tot_entity=5, tot_relation=2, hidden_size=4, margin=6.0)
    assert list(r.state_dict()) == ["ent_embeddings.weight", "ent_embeddings_imag.weight", "rel_embeddings.weight"]
    assert r.model_name == "rotate" and float(r.ent_embeddings.weight.abs().max()) <= (6.0 + 2.0) / 4
    with pytest.raises(NotImplementedError):
        c._reg(None, None, None, "l7")


def test_metric_calculator_settle_matches_reference_golden():
    import golden_util as gu
    from pykg2vec_b200.evaluator import MetricCalculator
    from pykg2vec_b200.synthetic import SyntheticConfig, SyntheticKnowledgeGraph
    g = gu.load("settle")
    mc = MetricCalculator(SyntheticConfig(SyntheticKnowledgeGraph(10, 2, 5, 2, 2), device="cpu"))
    mc.append_ranks(g["ranks"], epoch=0)
    mc.settle()
    assert mc.mr[0] == pytest.approx(float(g["mr"]), rel=1e-6)
    assert mc.fmrr[0] == pytest.approx(float(g["fmrr"]), rel=1e-6)
    for k in (1, 3, 5, 10):
        assert mc.hit[(0, k)] == pytest.approx(float(g["hit%d" % k]), rel=1e-6)
        assert mc.fhit[(0, k)] == pytest.approx(float(g["fhit%d" % k]), rel=1e-6)
    assert set(mc.get_curr_scores()) == {"mr", "fmr", "mrr", "fmrr"}


def test_metric_calculator_walk_equals_counts():
    """the reference-compatible sorted-list walk (append_result) equals the count formulation."""
    from pykg2vec_b200.evaluator import MetricCalculator, build_filter_csr
    from pykg2vec_b200.synthetic import SyntheticConfig, SyntheticKnowledgeGraph
    kg = SyntheticKnowledgeGraph(50, 3, 200, 10, 10, seed=2)
    mc = MetricCalculator(SyntheticConfig(kg, device="cpu"))
    rng = np.random.RandomState(0)
    h, r, t = [int(x) for x in kg.arrays["test"][0]]
    scores_t, scores_h = rng.standard_normal(50), rng.standard_normal(50)
    order_t, order_h = np.argsort(-scores_t), np.argsort(-scores_h)  # descending
    mc.append_result([order_t, order_h, h, r, t, 0])
    raw_t = int((scores_t < scores_t[t]).sum())
    filt_t = raw_t - sum(1 for e in mc.hr_t[(h, r)] if e != t and scores_t[e] < scores_t[t])
    raw_h = int((scores_h < scores_h[h]).sum())
    filt_h = raw_h - sum(1 for e in mc.tr_h[(t, r)] if e != h and scores_h[e] < scores_h[h])
    assert (mc.rank_tail[0], mc.f_rank_tail[0], mc.rank_head[0], mc.f_rank_head[0]) == (raw_t, filt_t, raw_h, filt_h)
    ptr, idx = build_filter_csr([(h, r), (999, 0)], mc.hr_t)
    assert ptr.tolist() == [0, len(mc.hr_t[(h, r)]), len(mc.hr_t[(h, r)])] and set(idx.tolist()) == mc.hr_t[(h, r)]


def test_relation_property_matches_reference_definition():
    """Bernoulli head-corruption probability = |distinct tails| / (|distinct heads| + |distinct tails|)
    per relation over the training triples (kgcontroller.py:466-492)."""
    from pykg2vec_b200.generator import relation_property
    train = np.array([[0, 0, 1], [0, 0, 2], [0, 0, 3], [4, 0, 3],   # r0: heads {0,4}, tails {1,2,3} -> 3/5
                      [1, 1, 1], [2, 1, 1]])                         # r1: heads {1,2}, tails {1}     -> 1/3
    p = relation_property(train, 3)
    assert p[0] == pytest.approx(3 / 5) and p[1] == pytest.approx(1 / 3) and p[2] == 0.0


def test_oracle_sampler_rules_on_cpu():
    """the oracle's negative sampler (the checker of kge_sample_negatives) obeys generator.py:42-158"""
    import oracle
    rng = np.random.RandomState(1)
    train = np.unique(np.stack([rng.randint(30, size=600), rng.randint(3, size=600), rng.randint(30, size=600)], 1), axis=0)
    pos = train[rng.randint(len(train), size=100)]
    nh, nr, nt = oracle.sample_negatives(train, pos[:, 0], pos[:, 1], pos[:, 2], 3, None, 30, seed=5, step=0)
    known = set(map(tuple, train.tolist()))
    assert not any((int(a), int(b), int(c)) in known for a, b, c in zip(nh, nr, nt))
    rep = np.repeat(pos, 3, axis=0)
    assert np.array_equal(nr, rep[:, 1]) and ((nh == rep[:, 0]) | (nt == rep[:, 2])).all()
    tail_corrupted = (nh == rep[:, 0]).mean()
    assert 0.3 < tail_corrupted < 0.7  # uniform sampling: p = 0.5
