"""Pins the CPU oracle against the UNMODIFIED reference on seeded inputs beyond the other fixtures:
link-prediction ranks (raw and filtered, heads and tails), dense tail / head / relation scores bit
for bit, relation-prediction ranks, scoring_function -- for every model kind the oracle restates, at
plane widths that exercise the one-lane sum, the 8-lane sums and the cascade.

The reference's outputs were recorded by tests/golden/make_golden_live.py, which ran it on these
inputs, into tests/golden/live_reference.npz: rank vectors in full, dense scores as a digest of their
bits.  The inputs are rebuilt here from their seeds -- this package's model classes draw the
reference's weights bit for bit -- and digests of the tables and filter dictionaries the reference
held pin them."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import kge_oracle as oracle
from tests import helpers

GOLDEN = os.path.join(helpers.GOLDEN_DIR, "live_reference.npz")
N_ENT, N_REL, N_FACTS, N_TEST = 260, 6, 1800, 70
STATE_NAMES = {"ent_emb.weight": "ent", "rel_emb.weight": "rel", "rel_mat.weight": "rel_mat",
               "re_ent_emb.weight": "re_ent", "im_ent_emb.weight": "im_ent", "re_rel_emb.weight": "re_rel",
               "im_rel_emb.weight": "im_rel", "sc_ent_emb.weight": "sc_ent", "sc_rel_emb.weight": "sc_rel"}
LP_NAMES = ("rank_true_heads", "rank_true_tails", "filt_rank_true_heads", "filt_rank_true_tails")

CASES = [("transe_l1", 33), ("transe_l2", 50), ("transe_l2", 203), ("distmult", 7), ("distmult", 64),
         ("distmult", 520), ("rescal", 12), ("complex", 24), ("complex", 520), ("analogy", 14),
         ("analogy", 72), ("analogy", 1040), ("toruse_l1", 40), ("toruse_l2", 40)]


def case_facts(d):
    """All facts of case d; the first N_TEST are the test triples."""
    return helpers.random_graph(N_ENT, N_REL, N_FACTS, seed=d)


def draw_weights(model, kind):
    """The case's tables: `model` was just constructed after torch.manual_seed(1000 + d); rows are
    rescaled, entity rows 200:230 duplicate rows 0:30 (exact ties), and TorusE's tables hold the
    fractional parts its evaluator reads.  Returns the oracle parameters."""
    with torch.no_grad():
        for p in model.parameters():
            p.mul_(1.0 + 0.5 * torch.rand(p.shape[0], 1))
        for name, emb in model.named_children():
            if "ent" in name:
                emb.weight[200:230] = emb.weight[0:30]
    if kind.startswith("toruse"):
        model.normalize_parameters()
    return {STATE_NAMES[k]: v.detach().clone() for k, v in model.state_dict().items()}


def dict_arrays(d):
    """defaultdict(set) -> (sorted keys (n, 2), offsets (n + 1), sorted values)."""
    keys = sorted(d.keys())
    offs = np.zeros(len(keys) + 1, dtype=np.int64)
    vals = []
    for i, key in enumerate(keys):
        vals.extend(sorted(d[key]))
        offs[i + 1] = len(vals)
    return np.array(keys, dtype=np.int64).reshape(-1, 2), offs, np.array(vals, dtype=np.int64)


def digest(*arrays):
    """SHA-256 of the arrays' bytes.  Float tensors are hashed as float32 with -0 read as +0, so
    that equal digests mean what helpers.bits_equal(...).all() means: the same bits, up to the sign
    of zero."""
    h = hashlib.sha256()
    for a in arrays:
        if isinstance(a, torch.Tensor):
            a = (a.detach().float() + 0.0).contiguous().numpy()
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.fixture(scope="module")
def ref():
    z = np.load(GOLDEN, allow_pickle=False)
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("kind,d", CASES)
def test_oracle_equals_the_live_reference(kind, d, ref):
    pre = "%s_%d:" % (kind, d)
    g = {k[len(pre):]: v for k, v in ref.items() if k.startswith(pre)}

    def same(name, *arrays):
        return digest(*arrays) == str(g["sha256_" + name])

    h, t, r = case_facts(d)
    torch.manual_seed(1000 + d)
    P = draw_weights(helpers.KIND_TO_CLASS[kind](d, N_ENT, N_REL), kind)
    for name, w in P.items():
        assert same(name, w), "%s: not the table the reference held" % name
    dh, dt = oracle.build_filter_dicts(h, t, r)
    dr = oracle.build_rel_dict(h, t, r)
    assert same("dh", *dict_arrays(dh)) and same("dt", *dict_arrays(dt)) and same("dr", *dict_arrays(dr))
    hh, tt, rr = h[:N_TEST], t[:N_TEST], r[:N_TEST]

    got = oracle.link_prediction(kind, P, hh, tt, rr, dh, dt, 32)
    for mine, name in zip(got, LP_NAMES):
        assert np.array_equal(mine.numpy(), g[name]), (kind, d, name)

    assert same("scores_tail", oracle.scores_all(kind, P, hh[:8], tt[:8], rr[:8], "tail"))
    assert same("scores_head", oracle.scores_all(kind, P, hh[:8], tt[:8], rr[:8], "head"))
    if not kind.startswith("toruse"):                # scoring_function: the oracle restates the on-the-fly normalisation
        assert same("triple_scores", oracle.score_triples(kind, P, hh, tt, rr))

    if kind.startswith("toruse"):
        return                                       # the reference's TorusE relation case is broken (rel_emb_dim)
    for directed, tag in ((True, "dir"), (False, "undir")):
        a, b = oracle.relation_prediction(kind, P, hh, tt, rr, dr, 32, directed=directed)
        assert np.array_equal(a.numpy(), g["rank_true_rels_" + tag]), (kind, d, directed)
        assert np.array_equal(b.numpy(), g["filt_rank_true_rels_" + tag]), (kind, d, directed)
    assert same("scores_rel", oracle.relation_scores_all(kind, P, hh[:8], tt[:8]))
