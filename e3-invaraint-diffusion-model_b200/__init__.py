"""e3-invaraint-diffusion-model_b200 -- B200 (sm_100a) implementation of the sequence-model hot path of
LabJunBMI/E3-invaraint-diffusion-model: denoiser forward + discrete BLOSUM reverse-diffusion step,
behind the reference's own model.py / sample.py / utils.py interface.

The directory name contains '-', so import it with
    importlib.import_module("e3-invaraint-diffusion-model_b200")
or through the root-level alias module `seqdiff_b200`.
"""
from . import _cabi, dataset, design, distributed, model, sample, structure_model, train, utils  # noqa: F401
from .dataset import LigandBindingSiteDataset, collate_complexes  # noqa: F401
from ._cabi import SeqdiffError, lib  # noqa: F401
from .design import design_dataset  # noqa: F401
from .distributed import denoise_sharded, design_sharded, p_sample_loop_sharded, shard_batch, shard_bounds  # noqa: F401
from .model import AA_VOCAB, BertConfig, ConditionalBertForDiffusionBase, PeptideDiff  # noqa: F401
from .sample import decode_tensors, denoise, denoise_tensors, score, score_tensors, denoise_with_generated_angles, load_generated_angles, sample_dataset, generate_discrete_noise, sample_p_zs_given_zt_discrete  # noqa: F401
from .utils import BlosumTransition, DiscreteUniformTransition, PredefinedNoiseScheduleDiscrete  # noqa: F401

__all__ = ["model", "sample", "utils", "structure_model", "design", "train", "lib", "SeqdiffError", "BertConfig", "ConditionalBertForDiffusionBase", "PeptideDiff",
           "denoise", "denoise_tensors", "score", "score_tensors", "generate_discrete_noise", "sample_p_zs_given_zt_discrete", "BlosumTransition",
           "DiscreteUniformTransition", "PredefinedNoiseScheduleDiscrete", "AA_VOCAB"]
