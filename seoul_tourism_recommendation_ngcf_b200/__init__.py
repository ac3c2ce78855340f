"""B200-native NGCF embedding-propagation hot path behind the reference's NGCF / BPR API."""
from .NGCF import NGCF
from .bprloss import BPR
from .experiment import Experiment, eval_groups
from .graph import GraphedStep
from .lightgcn import LightGCN, XSimGCL
from .optim import Adam
from .sampler import HardNegatives, TourDataset, sample_negatives
from .scoring import Interactions, full_rank_eval, rank_metrics, score_topk
from .softmax_loss import SoftmaxLoss

__all__ = ["NGCF", "LightGCN", "XSimGCL", "BPR", "GraphedStep", "Adam", "score_topk", "Experiment", "eval_groups",
           "TourDataset", "sample_negatives", "Interactions", "full_rank_eval", "rank_metrics", "HardNegatives",
           "SoftmaxLoss"]
