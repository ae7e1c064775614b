"""A stand-in for the state ``BasicDataLoader._build_fact_mat`` reads (gnn/dataset_load.py:473-527): per-question
(head, rel, tail) local-id arrays, the global->local maps (only their length is used) and three scalars."""
import numpy as np


class FakeLoader:
    data_eff = False

    def __init__(self, seed, num_questions, max_local_entity, num_kb_relation, use_self_loop=True,
                 facts_lo=0, facts_hi=40):
        rs = np.random.RandomState(seed)
        self.max_local_entity = max_local_entity
        self.num_kb_relation = num_kb_relation
        self.use_self_loop = use_self_loop
        self.kb_adj_mats, self.global2local_entity_maps = [], []
        for _ in range(num_questions):
            n_ent = int(rs.randint(1, max_local_entity + 1))
            n_fact = int(rs.randint(facts_lo, facts_hi + 1))
            h = rs.randint(0, n_ent, n_fact).astype(int)
            t = rs.randint(0, n_ent, n_fact).astype(int)
            r = rs.randint(0, max(num_kb_relation - 1, 1), n_fact).astype(int)
            if n_fact > 3:                       # repeated (head, rel) pairs and a hub head
                h[1], r[1] = h[0], r[0]
                h[2] = h[0]
            self.kb_adj_mats.append((h, r, t))
            self.global2local_entity_maps.append({1000 + k: k for k in range(n_ent)})


CASES = {   # name -> (loader kwargs, sample_ids, fact_dropout, numpy seed)
    "small": (dict(seed=1, num_questions=6, max_local_entity=12, num_kb_relation=9), [0, 1, 2, 3, 4, 5], 0.0, 11),
    "dropout_subset": (dict(seed=2, num_questions=8, max_local_entity=20, num_kb_relation=7), [7, 2, 2, 5], 0.3, 12),
    "no_self_loop": (dict(seed=3, num_questions=4, max_local_entity=9, num_kb_relation=5, use_self_loop=False),
                     [3, 0, 1], 0.0, 13),
    "empty_questions": (dict(seed=4, num_questions=5, max_local_entity=6, num_kb_relation=4, facts_hi=1),
                        [0, 1, 2, 3, 4], 0.5, 14),
}

# Larger loader states (thousands of facts per batch), big enough for a meaningful timing comparison.
LARGE_CASES = {
    "large_a": (dict(seed=100, num_questions=12, max_local_entity=300, num_kb_relation=50, facts_lo=100, facts_hi=900),
                list(np.random.RandomState(0).permutation(12)), 0.0, 7),
    "large_b": (dict(seed=101, num_questions=20, max_local_entity=500, num_kb_relation=200, facts_lo=0, facts_hi=1500),
                list(np.random.RandomState(1).permutation(20)), 0.25, 8),
}
