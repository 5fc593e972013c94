"""Helpers shared by the tests: load a golden case (tests/golden/*.npz, produced by the
reference itself — see make_golden.py) as an oracle.Model."""
import glob
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NON_CASES = {"losses", "settle", "pretrained_transe_fb15k_checkpoint"}
PROJ_PREFIXES = ("conve_", "tucker_")
SHAPE_PREFIX = "shapes_"   # BASELINE-shape cases: ids / reference outputs only, tables regenerated from a seed


def case_names():
    names = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return [n for n in names if n not in NON_CASES and not n.startswith(PROJ_PREFIXES) and not n.startswith(SHAPE_PREFIX)]


def proj_case_names():
    """ConvE cases (tests/golden/make_golden_proj.py): full state_dict + tail operands, not table lists."""
    names = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))
    return [n for n in names if n.startswith("conve_")]


def proj_state(g):
    """state_dict (numpy) of the reference ConvE stored in a conve_* case"""
    return {k[3:]: g[k] for k in g if k.startswith("sd_") and not k.startswith("sd_after_")}


def load(name):
    return dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))


def tables_of(g):
    out, k = [], 0
    while "table%d" % k in g:
        out.append(g["table%d" % k])
        k += 1
    return out


def raw_tables_of(g):
    """ConvKB only: the reference's own parameters [ent, rel, conv_w0, conv_b0, ..., fc_w, fc_b]."""
    out, k = [], 0
    while "raw%d" % k in g:
        out.append(g["raw%d" % k])
        k += 1
    return out


def model_kwargs(g):
    """-> dict(name, dim, rel_dim, l1_flag, margin, embedding_range)"""
    name = str(g["model"])
    kw = {k[3:]: g[k] for k in g if k.startswith("kw_")}
    dim = int(kw.get("hidden_size", kw.get("ent_hidden_size", 0)))
    rel_dim = int(kw.get("rel_hidden_size", dim))
    margin = float(kw.get("margin", 0.0))
    if name in ("rescal", "sme", "sme_bl"):
        rel_dim = dim
    return dict(name=name, dim=dim, rel_dim=rel_dim, l1_flag=bool(kw.get("l1_flag", False)),
                margin=margin,
                embedding_range=((margin + 2.0) / dim) if name == "rotate" else None)


def oracle_model(g):
    import oracle
    kw = model_kwargs(g)
    return oracle.Model(kw["name"], tables_of(g), kw["dim"], rel_dim=kw["rel_dim"],
                        l1_flag=kw["l1_flag"], margin=kw["margin"],
                        embedding_range=kw["embedding_range"])


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-30)


# ---- BASELINE.json shapes: tables are regenerated from a seed on either side (numpy's
# RandomState stream is platform independent), only ids / reference scores / reference ranks are
# stored (tests/golden/shapes_*.npz, written by tests/golden/make_golden_shapes.py) ---------------
BASELINE_SHAPES = {
    # configs[1]: TransE on FB15k-237, d=200, L2 (-l1 False)
    "cfg2_transe_fb15k237": dict(model="transe", N=14541, R=237, d=200, l1=False, margin=0.0, seed=20237),
    # configs[2]: DistMult and ComplEx on WN18RR, d=200
    "cfg3_distmult_wn18rr": dict(model="distmult", N=40943, R=11, d=200, l1=False, margin=0.0, seed=20318),
    "cfg3_complex_wn18rr": dict(model="complex", N=40943, R=11, d=200, l1=False, margin=0.0, seed=20319),
    # configs[3]: RotatE on FB15k, d=1000, margin 24 (hyperparams/RotatE.yaml)
    "cfg4_rotate_fb15k": dict(model="rotate", N=14951, R=1345, d=1000, l1=False, margin=24.0, seed=20415),
    # configs[4]: ComplEx on YAGO3-10, d=500
    "cfg5_complex_yago310": dict(model="complex", N=123182, R=37, d=500, l1=False, margin=0.0, seed=20510),
}
_SHAPE_TABLES = {"transe": "er", "distmult": "er", "complex": "eerr", "rotate": "eer"}


def baseline_tables(spec):
    """Seeded tables in C-ABI order with the reference's initialisers: xavier_uniform
    U(+-sqrt(6/(rows+d))) (pairwise.py:46-47, pointwise.py:151-160,432-437), RotatE
    U(+-(margin+2)/d) (pairwise.py:748-755)."""
    rng = np.random.RandomState(spec["seed"])
    out = []
    for kind in _SHAPE_TABLES[spec["model"]]:
        rows = spec["N"] if kind == "e" else spec["R"]
        if spec["model"] == "rotate":
            a = (spec["margin"] + 2.0) / spec["d"]
        else:
            a = np.sqrt(6.0 / (rows + spec["d"]))
        out.append(rng.uniform(-a, a, size=(rows, spec["d"])).astype(np.float32))
    return out


def baseline_oracle_model(spec, tables=None):
    import oracle
    tables = baseline_tables(spec) if tables is None else tables
    return oracle.Model(spec["model"], tables, spec["d"], rel_dim=spec["d"], l1_flag=spec["l1"], margin=spec["margin"],
                        embedding_range=((spec["margin"] + 2.0) / spec["d"]) if spec["model"] == "rotate" else None)


def shape_case_path(name):
    return os.path.join(GOLDEN_DIR, "shapes_%s.npz" % name)


def fp64_candidate_scores(spec, tables, h, r, t, direction):
    """float64 scores of one query against EVERY entity as candidate tail (direction 0) or head (1),
    straight from the model definitions (pairwise.py:56-93,765-791; pointwise.py:444-446,163-188) —
    an arithmetic-order-free yardstick for near ties."""
    T = [x.astype(np.float64) for x in tables]
    m = spec["model"]
    if m == "transe":
        ent, rel = T
        nrm = lambda x: x / np.maximum(np.linalg.norm(x, axis=-1, keepdims=True), 1e-12)
        E = nrm(ent)
        if direction == 0:
            x = nrm(ent[h]) + nrm(rel[r]) - E
        else:
            x = E + nrm(rel[r]) - nrm(ent[t])
        return np.abs(x).sum(-1) if spec["l1"] else np.sqrt((x * x).sum(-1))
    if m == "distmult":
        ent, rel = T
        q = ent[h] * rel[r] if direction == 0 else rel[r] * ent[t]
        return -(ent @ q)
    if m == "complex":
        er, ei, rr, ri = T
        if direction == 0:   # sum (hr rr - hi ri) tr + (hi rr + hr ri) ti
            a, b = er[h] * rr[r] - ei[h] * ri[r], ei[h] * rr[r] + er[h] * ri[r]
        else:                # sum (tr rr + ti ri) hr + (ti rr - tr ri) hi
            a, b = er[t] * rr[r] + ei[t] * ri[r], ei[t] * rr[r] - er[t] * ri[r]
        return -(er @ a + ei @ b)
    if m == "rotate":
        er, ei, rel = T
        th = rel[r] / (((spec["margin"] + 2.0) / spec["d"]) / 3.14159265358979323846)
        c, s = np.cos(th), np.sin(th)
        if direction == 0:
            xr, xi = er[h] * c - ei[h] * s - er, er[h] * s + ei[h] * c - ei
        else:
            xr, xi = er * c - ei * s - er[t], er * s + ei * c - ei[t]
        return (xr * xr + xi * xi).sum(-1) - spec["margin"]
    raise KeyError(m)


def rank_interval(scores64, target, rel_tol=3e-6):
    """[lo, hi] of the raw 0-based rank any fp32 evaluation may report: candidates whose fp64 score is
    within rel_tol * scale of the target's are ambiguous (scale = the largest magnitude entering the
    last rounding: max |score|)."""
    s_t = scores64[target]
    delta = rel_tol * max(np.abs(scores64).max(), 1e-30)
    others = np.delete(scores64, target)
    return int((others < s_t - delta).sum()), int((others <= s_t + delta).sum())
