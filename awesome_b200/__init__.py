"""awesome_b200 -- B200-native shape-prior fitting path of jp-schneider/awesome.

Drop-in names for the reference's YAML configs (``prior_model_type`` / ``optimizer_type``):
``awesome_b200.ConvexNextNet``, ``awesome_b200.ConvexNet``, ``awesome_b200.PathConnectedNet``,
``awesome_b200.real_nvp_path_connected_net``, ``awesome_b200.FusedAdam``, ``awesome_b200.FusedAdamax``.
All arithmetic runs in ``csrc/libawb.so`` (hand-written sm_100a CUDA); there is no CPU fallback.
"""
from .core import GridSpecHost, Prior, iou_counts, target_counts  # noqa: F401
from .fit import (FlowIdentityFitter, LossConfig, OptimConfig, PriorFitter, SlicedFitter, rank_slices,  # noqa: F401
                  slice_plan)
from .optim import FusedAdam, FusedAdamax  # noqa: F401
from .pretrain import (FitSchedule, FrameResult, collect_unaries, evaluate_frames, fit_frames, fit_frames_grouped,  # noqa: F401
                       fit_sequence, load_pretrain_checkpoint, mask_iou, noisy_unaries, save_pretrain_checkpoint)
from .prior_cache import DevicePriorCache, PriorManager  # noqa: F401
from .sharded_fit import fit_sequence_sharded, plan_segments, segments_of_rank  # noqa: F401
from . import synth  # noqa: F401
from .joint import GradBucket, JointTrainer  # noqa: F401
from . import image, measures  # noqa: F401
from .model import (BatchSizeMultiPriorModule, ConvexDiffeomorphismNet, ConvexNet, ConvexNextNet, MeanStd, MinMax,  # noqa: F401
                    MultipleObjectsAwarePathConnectedNet, NoisyPathConnectedNet, NormNet, NumberBasedMultiPriorModule, PathConnectedNet,
                    PixelizeNet, StarFitter, StarShapedNet, get_norm, init_realnvp, real_nvp_path_connected_net)

from .reference_bridge import integrate_with_reference  # noqa: F401,E402

integrate_with_reference()          # no-op unless the reference package is already imported in this process

__version__ = "0.2.0"
