"""Oracle restatement of the predictive_evaluation protocol (test infrastructure).

NOT pinned by goldens: the reference files (DRecPy/Evaluation/Processes/predictive_evaluation.py:7-65 and
Evaluation/Metrics/regression.py) are restated from their cited behaviour.  The regression metrics are sklearn's
mean_squared_error / mean_absolute_error for one output, and RMSE is the square root of MSE.
"""
import math

import numpy as np


def mse(y_true, y_pred):
    d = np.asarray(y_true, np.float64) - np.asarray(y_pred, np.float64)
    return float(np.mean(d ** 2))


def rmse(y_true, y_pred):
    return math.sqrt(mse(y_true, y_pred))


def mae(y_true, y_pred):
    return float(np.mean(np.abs(np.asarray(y_true, np.float64) - np.asarray(y_pred, np.float64))))


METRICS = {'RMSE': rmse, 'MSE': mse, 'MAE': mae}


def predictive_evaluation_oracle(predict_fn, test_users, test_items, test_vals, count_none_predictions=False,
                                 n_test_predictions=None, metrics=('RMSE', 'MSE')):
    """predict_fn(user, item) -> a prediction or None.  Arrays are the test set in row order.

    Rows in order; a None prediction is skipped, or counted as 0 when count_none_predictions; no row is predicted after
    n_test_predictions counted rows; {name: round(metric(y_true, y_pred), 4)}.  Returns (results, y_true, y_pred)."""
    y_true, y_pred = [], []
    for u, it, v in zip(test_users, test_items, test_vals):
        if n_test_predictions is not None and len(y_pred) >= n_test_predictions:
            break
        p = predict_fn(u, it)
        if p is None:
            if not count_none_predictions:
                continue
            p = 0.0
        y_true.append(float(v))
        y_pred.append(float(p))
    yt, yp = np.array(y_true, np.float64), np.array(y_pred, np.float64)
    return {m: round(METRICS[m](yt, yp), 4) for m in metrics}, yt, yp
