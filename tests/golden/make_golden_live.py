"""tests/golden/live_reference.npz: outputs of the UNMODIFIED reference (torchkge v0.17.7) for the
cases of tests/test_oracle_live_reference.py, on the inputs that test rebuilds from its seeds.

    python tests/golden/make_golden_live.py <directory holding the reference's torchkge package>

For every case (kind, d) the keys "<kind>_<d>:<name>" hold the four rank vectors of its
LinkPredictionEvaluator and -- TorusE aside, whose relation case fails in the reference -- the ranks
of its RelationPredictionEvaluator, directed and undirected.  Keys "<kind>_<d>:sha256_<name>" hold
the digest (test_oracle_live_reference.digest) of every table the reference model held, of its
three filter dictionaries (dh, dt, dr), of the dense tail / head scores of the first 8 test triples
(inference_scoring_function), of scoring_function on the test triples and of the dense relation
scores of the first 8 pairs.  Weights are not stored: the script checks that this package's model
classes draw the same tables from the same seeds.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests import helpers  # noqa: E402
from tests import test_oracle_live_reference as live  # noqa: E402


def reference_model(m, kind, d):
    if kind in ("transe_l1", "transe_l2"):
        return m.TransEModel(d, live.N_ENT, live.N_REL, "L1" if kind == "transe_l1" else "L2")
    if kind == "distmult":
        return m.DistMultModel(d, live.N_ENT, live.N_REL)
    if kind == "rescal":
        return m.RESCALModel(d, live.N_ENT, live.N_REL)
    if kind == "complex":
        return m.ComplExModel(d, live.N_ENT, live.N_REL)
    if kind == "analogy":
        return m.AnalogyModel(d, live.N_ENT, live.N_REL)
    return m.TorusEModel(d, live.N_ENT, live.N_REL, "torus_L1" if kind == "toruse_l1" else "torus_L2")


def main(ref_dir):
    sys.path.insert(0, ref_dir)
    from torchkge import models
    from torchkge.data_structures import KnowledgeGraph
    from torchkge.evaluation import LinkPredictionEvaluator, RelationPredictionEvaluator
    out = {}
    ix = {i: i for i in range(live.N_ENT)}
    rx = {i: i for i in range(live.N_REL)}
    for kind, d in live.CASES:
        o = {}
        h, t, r = live.case_facts(d)
        n = live.N_TEST
        full = KnowledgeGraph(kg={"heads": h, "tails": t, "relations": r}, ent2ix=ix, rel2ix=rx)
        test = KnowledgeGraph(kg={"heads": h[:n], "tails": t[:n], "relations": r[:n]}, ent2ix=ix, rel2ix=rx,
                              dict_of_heads=full.dict_of_heads, dict_of_tails=full.dict_of_tails,
                              dict_of_rels=full.dict_of_rels)
        torch.manual_seed(1000 + d)
        model = reference_model(models, kind, d)
        P = live.draw_weights(model, kind)
        torch.manual_seed(1000 + d)
        mine = live.draw_weights(helpers.KIND_TO_CLASS[kind](d, live.N_ENT, live.N_REL), kind)
        assert list(mine) == list(P), (kind, d)
        sha = lambda name, *a: o.__setitem__("sha256_" + name, np.array(live.digest(*a)))  # noqa: E731
        for name, w in P.items():
            assert torch.equal(mine[name], w), (kind, d, name)
            sha(name, w)
        for tag, dct in (("dh", full.dict_of_heads), ("dt", full.dict_of_tails), ("dr", full.dict_of_rels)):
            sha(tag, *live.dict_arrays(dct))
        hh, tt, rr = test.head_idx, test.tail_idx, test.relations

        ev = LinkPredictionEvaluator(model, test)
        ev.evaluate(b_size=32, verbose=False)
        for name in live.LP_NAMES:
            o[name] = getattr(ev, name).numpy()
        with torch.no_grad():
            he, te, re_, cands = model.inference_prepare_candidates(hh[:8], tt[:8], rr[:8], entities=True)
            sha("scores_tail", model.inference_scoring_function(he, cands, re_))
            sha("scores_head", model.inference_scoring_function(cands, te, re_))
            if not kind.startswith("toruse"):
                sha("triple_scores", model.scoring_function(hh, tt, rr))
        if not kind.startswith("toruse"):
            for directed, tag in ((True, "dir"), (False, "undir")):
                rp = RelationPredictionEvaluator(model, test, directed=directed)
                rp.evaluate(b_size=32, verbose=False)
                o["rank_true_rels_" + tag] = rp.rank_true_rels.numpy()
                o["filt_rank_true_rels_" + tag] = rp.filt_rank_true_rels.numpy()
            with torch.no_grad():
                he, te, _, rcands = model.inference_prepare_candidates(hh[:8], tt[:8], rr[:8], entities=False)
                sha("scores_rel", model.inference_scoring_function(he, te, rcands))
        out.update({"%s_%d:%s" % (kind, d, k): v for k, v in o.items()})
        print(kind, d, "MRR filt heads %.4f" % (1.0 / o["filt_rank_true_heads"]).mean())
    path = os.path.join(HERE, "live_reference.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(os.path.abspath(sys.argv[1]))
