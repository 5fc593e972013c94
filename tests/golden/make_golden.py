#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by RUNNING THE REFERENCE ITSELF.

Run in the build container only (needs /root/reference, which does not exist on the
GPU box):   python tests/golden/make_golden.py

The reference's own test-suite holds no known-answer vector for the scoring / rank
path (SURVEY.md §4), so these fixtures are what pins the oracle: they are outputs of
the unmodified reference classes (pykg2vec.models.pairwise/pointwise, Criterion,
Evaluator.test_*_rank, MetricCalculator.get_*_rank/settle) on seeded inputs, with
torch CPU fp32.  Three import stubs (hyperopt / seaborn / matplotlib) are needed to
import the package (SURVEY.md Appendix A); none of them is on the scored path.

One .npz per case: tables (C-ABI order of include/kge_b200.h), triple ids, reference
scores, autograd gradients of sum(scores * upstream), loss / regulariser values, and
for the eval cases the (trank, ftrank, hrank, fhrank) the reference's Python walk
returns together with the filter dictionaries it used.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"


def install_reference():
    sys.path.insert(0, REF)
    ho = types.ModuleType("hyperopt")
    ho.hp = types.SimpleNamespace()
    for n in ("fmin", "tpe", "Trials", "STATUS_OK", "space_eval"):
        setattr(ho, n, None)
    pyll = types.ModuleType("hyperopt.pyll")
    base = types.ModuleType("hyperopt.pyll.base")
    base.scope = types.SimpleNamespace()
    sb = types.ModuleType("seaborn")
    sb.set_style = lambda *a, **k: None
    mpl = types.ModuleType("matplotlib")
    plt = types.ModuleType("matplotlib.pyplot")
    mpl.colors = types.SimpleNamespace()
    mpl.pyplot = plt
    sys.modules.update({"hyperopt": ho, "hyperopt.pyll": pyll, "hyperopt.pyll.base": base,
                        "seaborn": sb, "matplotlib": mpl, "matplotlib.pyplot": plt})
    # utils/visualization.py:11-14, reached through pykg2vec.utils.trainer: stubbed when not installed
    import importlib.util
    if importlib.util.find_spec("networkx") is None:
        sys.modules["networkx"] = types.ModuleType("networkx")
    if importlib.util.find_spec("sklearn") is None:
        sk, manifold = types.ModuleType("sklearn"), types.ModuleType("sklearn.manifold")
        manifold.TSNE = None
        sk.manifold = manifold
        sys.modules.update({"sklearn": sk, "sklearn.manifold": manifold})


install_reference()
from pykg2vec.models import pairwise as ref_pairwise  # noqa: E402
from pykg2vec.models import pointwise as ref_pointwise  # noqa: E402
from pykg2vec.utils.criterion import Criterion  # noqa: E402
from pykg2vec.utils.evaluator import Evaluator, MetricCalculator  # noqa: E402

# name -> (reference class, ctor kwargs builder, state_dict keys in C-ABI table order)
SPECS = {
    "transe": (ref_pairwise.TransE, ["ent_embeddings", "rel_embeddings"]),
    "transh": (ref_pairwise.TransH, ["ent_embeddings", "rel_embeddings", "w"]),
    "transd": (ref_pairwise.TransD, ["ent_embeddings", "rel_embeddings", "ent_mappings", "rel_mappings"]),
    "transr": (ref_pairwise.TransR, ["ent_embeddings", "rel_embeddings", "rel_matrix"]),
    "rotate": (ref_pairwise.RotatE, ["ent_embeddings", "ent_embeddings_imag", "rel_embeddings"]),
    "distmult": (ref_pointwise.DistMult, ["ent_embeddings", "rel_embeddings"]),
    "cp": (ref_pointwise.CP, ["sub_embeddings", "rel_embeddings", "obj_embeddings"]),
    "complex": (ref_pointwise.Complex, ["ent_embeddings_real", "ent_embeddings_img",
                                        "rel_embeddings_real", "rel_embeddings_img"]),
    "rescal": (ref_pairwise.Rescal, ["ent_embeddings", "rel_matrices"]),
    "simple": (ref_pointwise.SimplE, ["ent_head_embeddings", "ent_tail_embeddings", "rel_embeddings",
                                      "rel_inv_embeddings"]),
    "simple_ignr": (ref_pointwise.SimplE_ignr, ["ent_head_embeddings", "ent_tail_embeddings",
                                                "rel_embeddings", "rel_inv_embeddings"]),
    "hole": (ref_pairwise.HoLE, ["ent_embeddings", "rel_embeddings"]),
    "slm": (ref_pairwise.SLM, ["ent_embeddings", "rel_embeddings", "mr1", "mr2"]),
    "ntn": (ref_pairwise.NTN, ["ent_embeddings", "rel_embeddings", "mr1", "mr2", "br", "mr"]),
    "sme": (ref_pairwise.SME, ["ent_embeddings", "rel_embeddings", "mu1", "mu2", "bu", "mv1", "mv2", "bv"]),
    "sme_bl": (ref_pairwise.SME_BL, ["ent_embeddings", "rel_embeddings", "mu1", "mu2", "bu", "mv1", "mv2", "bv"]),
    "kg2e": (ref_pairwise.KG2E, ["ent_embeddings_mu", "ent_embeddings_sigma", "rel_embeddings_mu",
                                 "rel_embeddings_sigma"]),
    "quate": (ref_pointwise.QuatE, ["ent_s_embedding", "ent_x_embedding", "ent_y_embedding", "ent_z_embedding",
                                    "rel_s_embedding", "rel_x_embedding", "rel_y_embedding", "rel_z_embedding"]),
    "octonione": (ref_pointwise.OctonionE, ["ent_embedding_%d" % i for i in range(1, 9)] +
                  ["rel_embedding_%d" % i for i in range(1, 9)]),
    "analogy": (ref_pointwise.ANALOGY, ["ent_embeddings", "rel_embeddings", "ent_embeddings_real",
                                        "ent_embeddings_img", "rel_embeddings_real", "rel_embeddings_img"]),
    "convkb": (ref_pointwise.ConvKB, ["ent_embeddings", "rel_embeddings"]),
}


def legacy_hole_forward(model, h, r, t):
    """HoLE.forward (pairwise.py:1119-1125) cannot run on torch >= 1.8 (torch.fft / torch.ifft are
    the removed legacy functions).  This reproduces what those lines computed under the pinned
    torch<1.7: fft of the zero-imaginary [b,d,2] views, torch.conj = no-op on a real tensor, `*`
    = elementwise product of the (re, im) pairs, ifft, real part.  Everything else (embed(), the
    tables, normalisation, sigmoid) is the reference's own code."""
    import torch.nn.functional as F
    h_e, r_e, t_e = model.embed(h, r, t)
    r_e = F.normalize(r_e, p=2, dim=-1)
    fh = torch.fft.fft(h_e.to(torch.complex64), dim=1)
    ft = torch.fft.fft(t_e.to(torch.complex64), dim=1)
    z = torch.complex(fh.real * ft.real, fh.imag * ft.imag)
    e = torch.fft.ifft(z, dim=1).real
    return -torch.sigmoid(torch.sum(r_e * e, 1))

CASES = [
    # name, model, N, R, kwargs, init ("ref" = reference initialiser, "normal" = N(0, 0.5))
    ("transe_l1_d50", "transe", 131, 7, dict(hidden_size=50, l1_flag=True), "ref"),
    ("transe_l2_d200", "transe", 131, 7, dict(hidden_size=200, l1_flag=False), "normal"),
    ("transe_l2_d33", "transe", 97, 5, dict(hidden_size=33, l1_flag=False), "normal"),
    ("transh_l2_d48", "transh", 101, 6, dict(hidden_size=48, l1_flag=False), "normal"),
    ("transh_l1_d50", "transh", 101, 6, dict(hidden_size=50, l1_flag=True), "ref"),
    ("transd_l1_d40", "transd", 101, 6, dict(ent_hidden_size=40, rel_hidden_size=40, l1_flag=True), "normal"),
    ("transd_l2_d200", "transd", 67, 4, dict(ent_hidden_size=200, rel_hidden_size=200, l1_flag=False), "ref"),
    ("transr_l2_24x16", "transr", 89, 5, dict(ent_hidden_size=24, rel_hidden_size=16, l1_flag=False), "normal"),
    ("transr_l1_50x50", "transr", 61, 4, dict(ent_hidden_size=50, rel_hidden_size=50, l1_flag=True), "ref"),
    ("rotate_d64", "rotate", 113, 9, dict(hidden_size=64, margin=6.0), "ref"),
    ("rotate_d200_wide", "rotate", 83, 9, dict(hidden_size=200, margin=24.0), "normal"),
    ("distmult_d200", "distmult", 131, 7, dict(hidden_size=200, lmbda=0.1), "ref"),
    ("distmult_d50", "distmult", 131, 7, dict(hidden_size=50, lmbda=0.1), "normal"),
    ("cp_d36", "cp", 73, 5, dict(hidden_size=36, lmbda=0.1), "normal"),
    ("complex_d200", "complex", 131, 7, dict(hidden_size=200, lmbda=0.1), "ref"),
    ("complex_d50", "complex", 131, 7, dict(hidden_size=50, lmbda=0.1), "normal"),
    ("rescal_d24", "rescal", 67, 4, dict(hidden_size=24, margin=1.0), "normal"),
    ("rescal_d50", "rescal", 53, 3, dict(hidden_size=50, margin=1.0), "ref"),
    ("simple_d48", "simple", 101, 6, dict(hidden_size=48, lmbda=0.1, tot_train_triples=1000, batch_size=100), "normal"),
    ("simple_ignr_d50", "simple_ignr", 101, 6, dict(hidden_size=50, lmbda=0.1, tot_train_triples=1000, batch_size=100), "normal"),
    ("slm_24x16", "slm", 71, 4, dict(ent_hidden_size=24, rel_hidden_size=16), "normal"),
    ("slm_50x30", "slm", 53, 3, dict(ent_hidden_size=50, rel_hidden_size=30), "ref"),
    ("ntn_16x12", "ntn", 47, 3, dict(ent_hidden_size=16, rel_hidden_size=12, lmbda=0.1), "normal"),
    ("ntn_20x20", "ntn", 41, 3, dict(ent_hidden_size=20, rel_hidden_size=20, lmbda=0.1), "ref"),
    ("sme_d24", "sme", 61, 4, dict(hidden_size=24), "normal"),
    ("sme_bl_d20", "sme_bl", 53, 3, dict(hidden_size=20), "normal"),
    ("kg2e_d40", "kg2e", 71, 4, dict(hidden_size=40, cmax=5.0, cmin=0.05), "ref"),
    ("kg2e_d50", "kg2e", 59, 3, dict(hidden_size=50, cmax=5.0, cmin=0.05), "ref"),
    ("quate_d20", "quate", 61, 4, dict(hidden_size=20, lmbda=0.1), "normal"),
    ("quate_d50", "quate", 53, 3, dict(hidden_size=50, lmbda=0.1), "ref"),
    ("octonione_d12", "octonione", 47, 3, dict(hidden_size=12, lmbda=0.1), "normal"),
    ("octonione_d50", "octonione", 41, 3, dict(hidden_size=50, lmbda=0.1), "ref"),
    ("analogy_d48", "analogy", 89, 5, dict(hidden_size=48, lmbda=0.1), "normal"),
    ("analogy_d100", "analogy", 71, 4, dict(hidden_size=100, lmbda=0.1), "ref"),
    ("hole_d30", "hole", 83, 5, dict(hidden_size=30, cmax=0.5, cmin=-0.5), "normal"),
    ("hole_d150", "hole", 61, 4, dict(hidden_size=150, cmax=0.5, cmin=-0.5), "ref"),
    # (new cases are appended so that the seeds of the existing ones never change)
    ("convkb_d24", "convkb", 71, 4, dict(hidden_size=24, num_filters=5, filter_sizes=[1, 2, 3], device="cpu"), "normal"),
    ("convkb_d100", "convkb", 53, 3, dict(hidden_size=100, num_filters=50, filter_sizes=[1, 2], device="cpu"), "ref"),
]
N_TRIPLES = 96
N_QUERIES = 6


def build_model(model, N, R, kw, init, seed):
    torch.manual_seed(seed)
    cls, keys = SPECS[model]
    m = cls(tot_entity=N, tot_relation=R, **kw)
    if init == "normal":
        with torch.no_grad():
            for k in keys:
                getattr(m, k).weight.normal_(0.0, 0.5)
    return m, keys


def random_filters(rng, N, R, queries, extra=40):
    """hr_t / tr_h dictionaries as KnowledgeGraph builds them (kgcontroller.py:410-428):
    every (h,r) -> set of tails and (t,r) -> set of heads over a set of known triples that
    contains the queries."""
    known = set((int(h), int(r), int(t)) for h, r, t in queries)
    for (h, r, t) in list(known):
        for _ in range(extra):
            if rng.rand() < 0.5:
                known.add((h, r, int(rng.randint(N))))
            else:
                known.add((int(rng.randint(N)), r, t))
    hr_t, tr_h = {}, {}
    for (h, r, t) in known:
        hr_t.setdefault((h, r), set()).add(t)
        tr_h.setdefault((t, r), set()).add(h)
    return hr_t, tr_h


def reference_ranks(model, N, queries, hr_t, tr_h):
    """Exactly the reference's evaluation path for each query (evaluator.py:313-326)."""
    ev = object.__new__(Evaluator)
    ev.model = model
    ev.config = types.SimpleNamespace(tot_entity=N, device="cpu")
    mc = object.__new__(MetricCalculator)
    mc.hr_t, mc.tr_h = hr_t, tr_h
    out = []
    with torch.no_grad():
        for (h, r, t) in queries:
            h_t, r_t, t_t = torch.LongTensor([h]), torch.LongTensor([r]), torch.LongTensor([t])
            hrank = ev.test_head_rank(r_t, t_t, N).detach().cpu().numpy()
            trank = ev.test_tail_rank(h_t, r_t, N).detach().cpu().numpy()
            tr, ftr = mc.get_tail_rank(trank, h, r, t)
            hk, fhk = mc.get_head_rank(hrank, h, r, t)
            out.append((tr, ftr, hk, fhk))
    return np.asarray(out, dtype=np.int32)


def csr(dct, keys):
    ptr, idx = [0], []
    for k in keys:
        idx.extend(sorted(dct.get(k, ())))
        ptr.append(len(idx))
    return np.asarray(ptr, dtype=np.int64), np.asarray(idx, dtype=np.int64)


def make_case(name, model, N, R, kw, init, seed):
    m, keys = build_model(model, N, R, kw, init, seed)
    if model == "hole":
        m.forward = lambda a, b, c: legacy_hole_forward(m, a, b, c)
    rng = np.random.RandomState(seed + 1000)
    h = rng.randint(N, size=N_TRIPLES).astype(np.int64)
    r = rng.randint(R, size=N_TRIPLES).astype(np.int64)
    t = rng.randint(N, size=N_TRIPLES).astype(np.int64)
    upstream = rng.standard_normal(N_TRIPLES).astype(np.float32)
    ht, rt, tt = torch.from_numpy(h), torch.from_numpy(r), torch.from_numpy(t)
    m.zero_grad()
    scores = m.forward(ht, rt, tt)  # (Rescal.forward row-normalises its tables in place first)
    (scores * torch.from_numpy(upstream)).sum().backward()
    out = {"model": model, "N": N, "R": R, "h": h, "r": r, "t": t, "upstream": upstream,
           "scores": scores.detach().numpy().copy()}
    for k, v in kw.items():
        out["kw_" + k] = np.asarray(v)
    if model == "hole":
        out["emulated_forward"] = np.asarray(True)
    for i, k in enumerate(keys):
        emb = getattr(m, k)
        out["table%d" % i] = emb.weight.detach().numpy().copy()
        out["grad%d" % i] = emb.weight.grad.detach().numpy().copy()
    out["table_keys"] = np.asarray(keys)
    if model == "convkb":
        # raw parameters of the reference (conv_list is a plain Python list: not in state_dict) and
        # their gradients, plus the C-ABI tables 2/3 = the collapsed affine form computed in fp64
        # from those parameters (oracle/ref_port.py convkb_collapse; see include/kge_b200.h)
        sys.path.insert(0, os.path.join(HERE, "..", ".."))
        from oracle import ref_port
        raw = [m.ent_embeddings.weight, m.rel_embeddings.weight]
        for conv in m.conv_list:
            raw += [conv.weight, conv.bias]
        raw += [m.fc1.weight, m.fc1.bias]
        for i, p_ in enumerate(raw):
            out["raw%d" % i] = p_.detach().numpy().copy()
            out["rawgrad%d" % i] = p_.grad.detach().numpy().copy()
        A, c0 = ref_port.convkb_collapse([c.weight.detach().double() for c in m.conv_list],
                                         [c.bias.detach().double() for c in m.conv_list],
                                         m.fc1.weight.detach().double(), m.fc1.bias.detach().double(),
                                         int(kw["hidden_size"]))
        out["table2"] = A.numpy().astype(np.float32)
        out["table3"] = c0.numpy().astype(np.float32)
        del out["kw_device"]
    # regularisers (pointwise models)
    if model in ("quate", "octonione"):
        with torch.no_grad():
            out["reg_f2"] = np.float32(m.get_reg(ht, rt, tt, reg_type="F2").item())
            out["reg_absn3"] = np.float32(m.get_reg(ht, rt, tt, reg_type="N3").item())
    if model in ("distmult", "complex", "cp", "analogy"):
        with torch.no_grad():
            out["reg_f2"] = np.float32(m.get_reg(ht, rt, tt, reg_type="F2").item())
            out["reg_n3"] = np.float32(m.get_reg(ht, rt, tt, reg_type="N3").item())
        if model == "complex":
            m3 = ref_pointwise.ComplexN3(tot_entity=N, tot_relation=R, **kw)
            m3.load_state_dict(m.state_dict())
            with torch.no_grad():
                out["reg_absn3"] = np.float32(m3.get_reg(ht, rt, tt).item())
    # evaluation through the reference's own Evaluator / MetricCalculator code
    q = [(int(h[i]), int(r[i]), int(t[i])) for i in range(N_QUERIES)]
    hr_t, tr_h = random_filters(rng, N, R, q)
    out["ranks"] = reference_ranks(m, N, q, hr_t, tr_h)
    out["filt_t_ptr"], out["filt_t_idx"] = csr(hr_t, [(a, b) for a, b, c in q])
    out["filt_h_ptr"], out["filt_h_idx"] = csr(tr_h, [(c, b) for a, b, c in q])
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote", name, "scores[:3]", out["scores"][:3], "ranks[0]", out["ranks"][0])


def make_losses(seed=7):
    rng = np.random.RandomState(seed)
    pos = (rng.standard_normal(64) * 2).astype(np.float32)
    neg = (rng.standard_normal(64) * 2).astype(np.float32)
    out = {"pos": pos, "neg": neg, "margin": np.float32(0.8)}
    p = torch.from_numpy(pos).requires_grad_()
    n = torch.from_numpy(neg).requires_grad_()
    loss = Criterion.pairwise_hinge(p, n, 0.8)
    loss.backward()
    out.update(hinge=np.float32(loss.item()), hinge_gpos=p.grad.numpy().copy(), hinge_gneg=n.grad.numpy().copy())
    # pointwise logistic: interleaved +1/-1 labels as generator.py:125-156; include large |x|
    preds = (rng.standard_normal(96) * 6).astype(np.float32)
    preds[:4] = [25.0, -25.0, 19.99, 20.01]
    target = np.where(np.arange(96) % 2 == 0, 1.0, -1.0).astype(np.float32)
    pr = torch.from_numpy(preds).requires_grad_()
    loss = Criterion.pointwise_logistic(pr, torch.from_numpy(target))
    loss.backward()
    out.update(preds=preds, target=target, logistic=np.float32(loss.item()), logistic_g=pr.grad.numpy().copy())
    # RotatE self-adversarial, neg_rate 8, alpha 1.0 and 0.1
    B, nr = 16, 8
    pos2 = (rng.standard_normal(B) * 3).astype(np.float32)
    neg2 = (rng.standard_normal(B * nr) * 3).astype(np.float32)
    out.update(sa_pos=pos2, sa_neg=neg2, sa_neg_rate=np.int32(nr))
    for tag, alpha in (("a1", 1.0), ("a01", 0.1)):
        p = torch.from_numpy(pos2).requires_grad_()
        n = torch.from_numpy(neg2).requires_grad_()
        loss = Criterion.pariwise_logistic(p, n, nr, alpha)
        loss.backward()
        out["sa_%s" % tag] = np.float32(loss.item())
        out["sa_%s_gpos" % tag] = p.grad.numpy().copy()
        out["sa_%s_gneg" % tag] = n.grad.numpy().copy()
    np.savez_compressed(os.path.join(HERE, "losses.npz"), **out)
    print("wrote losses", out["hinge"], out["logistic"], out["sa_a1"])


def make_settle(seed=11):
    """MetricCalculator.settle (evaluator.py:125-141) on a fixed rank list."""
    rng = np.random.RandomState(seed)
    ranks = rng.randint(0, 300, size=(40, 4)).astype(np.int32)
    ranks[:, 1] = np.minimum(ranks[:, 1], ranks[:, 0])
    ranks[:, 3] = np.minimum(ranks[:, 3], ranks[:, 2])
    mc = object.__new__(MetricCalculator)
    mc.config = types.SimpleNamespace(hits=[1, 3, 5, 10])
    mc.mr, mc.fmr, mc.mrr, mc.fmrr, mc.hit, mc.fhit = {}, {}, {}, {}, {}, {}
    mc.epoch = 0
    mc.rank_tail, mc.f_rank_tail = list(ranks[:, 0]), list(ranks[:, 1])
    mc.rank_head, mc.f_rank_head = list(ranks[:, 2]), list(ranks[:, 3])
    mc.settle()
    out = {"ranks": ranks, "mr": mc.mr[0], "fmr": mc.fmr[0], "mrr": mc.mrr[0], "fmrr": mc.fmrr[0]}
    for k in (1, 3, 5, 10):
        out["hit%d" % k] = mc.hit[(0, k)]
        out["fhit%d" % k] = mc.fhit[(0, k)]
    np.savez_compressed(os.path.join(HERE, "settle.npz"), **out)
    print("wrote settle", out["mr"], out["fmrr"])


def make_pretrained(n_ent=1024, n_rel=32, seed=3):
    """Real trained weights: the FB15k TransE checkpoint shipped with the reference
    (examples/pretrained/TransE/model.vec.pt, l1_flag=True, dim 50).  Only a slice of
    the tables is stored (first n_ent entity rows, first n_rel relation rows)."""
    sd = torch.load(os.path.join(REF, "examples/pretrained/TransE/model.vec.pt"), map_location="cpu")
    ent = sd["ent_embeddings.weight"][:n_ent].contiguous()
    rel = sd["rel_embeddings.weight"][:n_rel].contiguous()
    m = ref_pairwise.TransE(tot_entity=n_ent, tot_relation=n_rel, hidden_size=50, l1_flag=True)
    m.load_state_dict({"ent_embeddings.weight": ent, "rel_embeddings.weight": rel})
    rng = np.random.RandomState(seed)
    h = rng.randint(n_ent, size=128).astype(np.int64)
    r = rng.randint(n_rel, size=128).astype(np.int64)
    t = rng.randint(n_ent, size=128).astype(np.int64)
    with torch.no_grad():
        scores = m(torch.from_numpy(h), torch.from_numpy(r), torch.from_numpy(t)).numpy().copy()
    q = [(int(h[i]), int(r[i]), int(t[i])) for i in range(12)]
    hr_t, tr_h = random_filters(rng, n_ent, n_rel, q, extra=60)
    out = {"model": "transe", "N": n_ent, "R": n_rel, "kw_hidden_size": np.asarray(50),
           "kw_l1_flag": np.asarray(True), "table0": ent.numpy(), "table1": rel.numpy(),
           "h": h, "r": r, "t": t, "scores": scores,
           "ranks": reference_ranks(m, n_ent, q, hr_t, tr_h)}
    out["filt_t_ptr"], out["filt_t_idx"] = csr(hr_t, [(a, b) for a, b, c in q])
    out["filt_h_ptr"], out["filt_h_idx"] = csr(tr_h, [(c, b) for a, b, c in q])
    np.savez_compressed(os.path.join(HERE, "pretrained_transe_fb15k_slice.npz"), **out)
    print("wrote pretrained slice; ranks[0:3]", out["ranks"][:3].tolist())


if __name__ == "__main__":
    torch.set_num_threads(1)
    only = [a for a in sys.argv[1:] if not a.startswith("-")]   # optional: regenerate just these cases
    for i, (name, model, N, R, kw, init) in enumerate(CASES):
        if not only or name in only:
            make_case(name, model, N, R, kw, init, seed=100 + i)
    if not only:
        make_losses()
        make_settle()
        make_pretrained()
