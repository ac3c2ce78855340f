"""B200-native NGCF embedding-propagation hot path behind the reference's NGCF / BPR API."""
from .NGCF import NGCF
from .bprloss import BPR
from .experiment import Experiment, eval_groups
from .graph import GraphedStep
from .optim import Adam
from .sampler import TourDataset, sample_negatives
from .scoring import Interactions, full_rank_eval, rank_metrics, score_topk

__all__ = ["NGCF", "BPR", "GraphedStep", "Adam", "score_topk", "Experiment", "eval_groups", "TourDataset",
           "sample_negatives", "Interactions", "full_rank_eval", "rank_metrics"]
