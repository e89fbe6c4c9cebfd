"""cpc_b200 -- B200-native (sm_100a) implementation of the CPC-audio training hot path.

Public surface mirrors the reference's modules (SURVEY.md 8b):
    frontend : CQT, InverseCQT, PhaseDifference, PhaseAccumulation, PreprocessingModule
    encoders : AudioEncoder, ScalogramEncoder, ScalogramEncoderBlock, ScalogramResidualEncoder
    model    : AudioPredictiveCodingModel, ActivationRegister, ActivationWriter
    ar_models: AudioGRUModel, ConvolutionalArModel, AttentionModel        (stock PyTorch, caller-side)
    trainer  : ContrastiveEstimationTrainer, linear/softplus/difference_score_function
    sampler  : FileBatchSampler, SyntheticAudioDataset
    audio_dataset: AudioDataset, AudioTestingDataset (WAV folders as one item stream)
    device_loader: DeviceBatchLoader (AudioDataset batches decoded and assembled on the GPU from raw PCM bytes)
    ddp      : one-process-per-GPU gradient averaging
    optim    : Adam (torch.optim.Adam semantics, one kernel per step)
    snapshots: state_dict of the reference's whole-model snapshot pickles, without importing reference code
    ops      : conv1d / conv2d / infonce / cqt_frontend autograd functions over the C-ABI
"""
from . import _lib, ops                                                        # noqa: F401
from .frontend import CQT, InverseCQT, PhaseAccumulation, PhaseDifference, PreprocessingModule  # noqa: F401
from .model import (ActivationRegister, ActivationWriter, AudioPredictiveCodingModel,  # noqa: F401
                    cuda0_writing_condition, load_to_cpu, num_parameters)
from .encoders import (AudioEncoder, Conv1d, Conv2d, Conv2dSeparable, ScalogramEncoder,  # noqa: F401
                       ScalogramEncoderBlock, ScalogramResidualEncoder, cqt_default_dict,
                       encoder_default_dict, scalogram_encoder_default_dict)
from .ar_models import AttentionModel, AudioGRUModel, ConvolutionalArBlock, ConvolutionalArModel  # noqa: F401
from .trainer import (ContrastiveEstimationTrainer, DeterministicSampler, GraphedTrainStep, difference_score_function,  # noqa: F401
                      linear_score_function, softplus_score_function)
from .sampler import FileBatchSampler, SyntheticAudioDataset                  # noqa: F401
from .audio_dataset import AudioDataset, AudioTestingDataset, list_all_audio_files  # noqa: F401
from . import configs, ddp, optim, snapshots                                                    # noqa: F401

__version__ = "0.1.0"
