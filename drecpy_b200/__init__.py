"""drecpy_b200: the B200-native hot path of DRecPy's embedding-based deep recommenders (CDAE, DMF, Caser).

Host code is Python and keeps DRecPy's public surface; all arithmetic runs in hand-written sm_100a CUDA behind
the C-ABI library libdrb.so (include/drb.h), bound with ctypes.  PyTorch only owns device buffers.
"""
from .dataset import InteractionData, synthetic_interactions, synthetic_item_shard
from .sampler import PointSampler
from .recommender import DeepRecommenderABC
from .cdae import CDAE
from .dmf import DMF
from .caser import Caser
from .evaluation import (ranking_evaluation, recommendation_evaluation, predictive_evaluation, HitRatio, NDCG, DCG,
                         Precision, Recall, RMSE, MSE, MAE)
from .splits import leave_k_out
from .early_stopping import MaxValidationValueRule
from .loss_tracker import LossTracker

InteractionDataset = InteractionData

__all__ = ['InteractionData', 'InteractionDataset', 'synthetic_interactions', 'synthetic_item_shard', 'PointSampler', 'DeepRecommenderABC', 'leave_k_out',
           'CDAE', 'DMF', 'Caser', 'ranking_evaluation', 'recommendation_evaluation', 'predictive_evaluation', 'HitRatio', 'NDCG', 'DCG',
           'Precision', 'Recall', 'RMSE', 'MSE', 'MAE',
           'MaxValidationValueRule', 'LossTracker']
