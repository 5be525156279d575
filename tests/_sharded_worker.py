"""Worker for tests/test_gpu_sharded.py under torch.distributed.run: one rank of a two-rank build, then the sharded
learners on its slice (ShardedRuleClassifications.from_distributed, TorchExchange), and on rank 0 the same calls on the
gathered matrix (gather() + load_result).  Each writes a JSON summary; the test compares them."""
import json
import os
import pickle
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def node(x):
    rule = None if x.rule is None else list(x.rule)
    return [rule, float(x.score).hex(), x.depth, x.n_pos, x.n_neg, x.present_child, x.absent_child, x.prediction,
            np.asarray(x.equivalent_rules).tolist(), x.equivalent_total]


def summary(rc, labels, seed):
    """The sharded or the whole-matrix results of one fixed set of calls, as JSON-able lists (floats as hex)."""
    from grm_b200 import cart, scm
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    from grm_b200.scm import SetCoveringMachine
    G = len(labels)
    n_train = G * 4 // 5
    pos = [g for g in range(n_train) if labels[g]]
    neg = [g for g in range(n_train) if not labels[g]]
    tpos = [g for g in range(n_train, G) if labels[g]]
    tneg = [g for g in range(n_train, G) if not labels[g]]
    test = tpos + tneg
    machines = [SetCoveringMachine(mt, p, 5) for mt in ("conjunction", "disjunction") for p in (0.5, 1.0, 4.0)]
    scm.fit_many(rc, [(m, pos, neg) for m in machines], rule_blacklist=[3, rc.shape[1] // 2 + 1])
    trees = [DecisionTreeClassifier(max_depth=5, max_equivalent_rules=cap) for cap in (None, 0, 3)]
    cart.fit_many(rc, [(t, pos, neg) for t in trees])
    a = cross_validate_scm(rc, pos, neg, ["conjunction", "disjunction"], [0.3, 1.0, 3.0], 4, 3, random_seed=seed,
                           test_pos=tpos, test_neg=tneg).to_dict()
    b = cross_validate_cart(rc, pos, neg, [None, {0: 0.5, 1: 2.0}], [1, 2, 4], [2, 8], 3, random_seed=seed,
                            test_pos=tpos, test_neg=tneg, max_equivalent_rules=4).to_dict()
    a.pop("seconds"), b.pop("seconds")
    return {
        "U": rc.shape[1] // 2,
        "scm": [[[it.rule, float(it.utility).hex(), it.positive_errors, it.negative_covers,
                  np.asarray(it.equivalent_rules).tolist()] for it in m.iterations] + [[list(r) for r in m.model]]
                for m in machines],
        "trees": [[node(x) for x in t.nodes] for t in trees],
        "cv_scm": json.dumps(a, sort_keys=True), "cv_cart": json.dumps(b, sort_keys=True),
        "predict": [m.predict(rc, test).tolist() for m in machines + trees],
        "columns": rc.get_columns([0, rc.shape[1] - 1]).tolist(),
    }


def main():
    out_dir, k = sys.argv[1], int(sys.argv[2])
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import DistributedBuilder, init_process_group_from_env
    from grm_b200.learning import KmerRuleClassifications, ShardedRuleClassifications
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_dev = torch.cuda.device_count()
    backend = "nccl" if n_dev >= world else "gloo"      # one GPU: the ranks share it and talk over the host
    device = local_rank % n_dev
    torch.cuda.set_device(device)
    dist = init_process_group_from_env(backend)
    with open(os.path.join(out_dir, "genomes.pkl"), "rb") as f:
        genomes, labels = pickle.load(f)
    G = len(genomes)
    db = DistributedBuilder(k=k, keep_singletons=True, n_genomes=G, rank=rank, world=world, device=device)
    try:
        db.reset()
        for i, g in enumerate(db.local_rows):
            db.add_genome_bytes(i, genomes[g])
        db.build()
        rc = ShardedRuleClassifications.from_distributed(db, G)
        res = summary(rc, labels, seed=7)
        res["backend"], res["slice"] = backend, rc.col_counts
        with open(os.path.join(out_dir, f"sharded_{rank}.json"), "w") as f:
            json.dump(res, f)
        whole = db.gather()
        if rank == 0:
            with KmerMatrixBuilder(k=k, device=device) as b:
                b.load_result(whole[0], whole[1], G)
                with open(os.path.join(out_dir, "whole.json"), "w") as f:
                    json.dump(summary(KmerRuleClassifications(b, G), labels, seed=7), f)
        dist.barrier()
    finally:
        db.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
