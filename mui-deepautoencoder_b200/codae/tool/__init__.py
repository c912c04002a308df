"""codae.tool -- masks, criteria, ranking, logging helpers (the reference's import surface) plus the B200 additions:
FusedStep (the fused training-step schedule), ComplementarityScorer / SwapScorer / CompatibilityScorer (stage IV) and the .cemb
binary embedding file."""
# reference surface
from .data_tool import (Corrupter, Normalizer, collate_embedding, get_mask_transformation, load_dataset_of_embeddings,
                        simple_collate)
from .metering import CombinedCriterion, RankingLoss, get_rmse
from .logger import PlotDrawer, display_info, export_parameters_to_json, get_date, set_logging
from .dictionnary import Dict
from .parser import parse
# additions
from .fused_step import FusedStep
from .inference import CompatibilityScorer, ComplementarityScorer, SwapScorer, compatibility_auc
from .embedding_file import convert_json_to_cemb, load_cemb_dataset, read_cemb, write_cemb
