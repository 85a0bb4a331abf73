"""dct_b200 -- B200 (sm_100a) kernels for the consistency hot path of Deep Co-Training
(K-view JSD, adversarial KL / VAT normalisation, Dice / confusion counting) behind the
reference's own loss / meter / generator interfaces.

Import as ``dct_b200`` (the repo-root alias module) or via importlib under the directory name.
"""
from . import _lib, _runtime  # noqa: F401
from . import loss, metrics, generators, utils, distributed, ensemble  # noqa: F401
from ._lib import DctError, build, library_path  # noqa: F401
from ._runtime import get_check_mode, raise_if_flagged, set_check_mode  # noqa: F401
from .ensemble import Ensembleway, Kappa2Annotator, KappaMetrics, KappaMetrics2, hard_vote, soft_vote, vote_class  # noqa: F401
from .generators import FSGMGenerator, VATGenerator, fgsm_perturb, l2_normalize  # noqa: F401
from .install import install, uninstall  # noqa: F401
from .loss import (JSD, JSD_2D, CrossEntropyLoss2d, Entropy, Entropy_2D, FusedJSDConsistency, KL_div, KL_Divergence_2D,  # noqa: F401
                   KL_Divergence_2D_Logit, get_loss_fn, jsd_consistency_from_logits, jsd_map_from_logits,
                   kl_consistency_from_logits, kl_div_with_logit, softmax_dim1, supervised_from_logits)
from .metrics import (ConfusionMatrix, DiceMeter, DiceMeter2, HausdorffMeter, IoU, SurfaceDistanceMeter,  # noqa: F401
                      dice_counts, dice_from_counts, hausdorff, surface_distances)

__version__ = "0.1.0"
