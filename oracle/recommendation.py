"""Oracle restatement of the recommendation_evaluation protocol (test infrastructure).

NOT pinned by goldens: the reference file (DRecPy/Evaluation/Processes/recommendation_evaluation.py:18-192) is restated
from its cited behaviour and from ranking_evaluation's conventions (oracle.ranking, which is pinned).  Steps 1-3 of a
user are oracle.ranking.user_candidates with n_neg=None and no generated negatives; the metrics are oracle.ranking's.
"""
import random

from .ranking import METRICS, user_candidates


def recommendation_evaluation_oracle(recommend_fn, test_users, test_items, test_vals, thr, n_test_users=None, k=10,
                                     n_pos_interactions=None, novelty=False, ignore_low_predictions_threshold=None,
                                     seed=0, metrics=('Precision', 'Recall', 'HitRatio', 'NDCG'), record=None):
    """recommend_fn(user, n, novelty, interaction_threshold) -> recommended raw item ids, best first; raises
    AssertionError for a user the model does not know.  Arrays are the test set in row order.

    Restates the protocol (not pinned by goldens): users in order of first appearance, the first n_test_users; user
    idx draws from random.Random(seed + idx); positives = test rows >= thr (all, or rng.sample of
    n_pos_interactions, too few -> skipped); the evaluated set C = sampled positives + every test row below thr
    (user_candidates with n_neg=None, no generated negatives); relevancy = first test row's value for items of C, 0 for
    recommended items outside C; a metric that raises skips that (metric, k) for the user; round(sum / count, 4)."""
    ks = k if isinstance(k, list) else [k]
    sums = {(m, k_): [0, 0] for m in metrics for k_ in ks}
    order, rows = [], {}
    for u, it, v in zip(test_users, test_items, test_vals):
        if u not in rows:
            rows[u] = []
            order.append(u)
        rows[u].append((it, v))
    n_test_users = len(order) if n_test_users is None else min(n_test_users, len(order))
    for idx, user in enumerate(order[:n_test_users]):
        rng = random.Random(seed + idx)
        res = user_candidates(rng, rows[user], set(), 0, thr, n_pos_interactions, None, False)
        if res is None:
            continue
        all_items, positives, rel_c = res
        try:
            recommendations = list(recommend_fn(user, max(ks), novelty, ignore_low_predictions_threshold))
        except AssertionError:
            continue
        relevancies = {it: 0 for it in recommendations}
        relevancies.update(rel_c)
        if record is not None:
            record.append((user, list(all_items), list(recommendations)))
        for m in metrics:
            kind, fn = METRICS[m]
            for k_ in ks:
                try:
                    if kind == 'rr':
                        val = fn(recommendations, k=k_, relevant_recommendations=positives)
                    else:
                        val = fn(recommendations, k=k_, relevancies=relevancies)
                    sums[(m, k_)][0] += val
                    sums[(m, k_)][1] += 1
                except Exception:
                    pass
    return {f'{m}@{k_}': (round(sums[(m, k_)][0] / sums[(m, k_)][1], 4) if sums[(m, k_)][1] > 0 else 0)
            for m, k_ in sums}
