"""hifigan_b200 — B200-native (sm_100a) HiFi-GAN vocoder hot path behind the reference's module API."""
from . import _lib  # noqa: F401
from .configs import load_config  # noqa: F401
from .env import AttrDict, build_env  # noqa: F401
from .meldataset import MAX_WAV_VALUE, CorpusSampler, MelDataset, SegmentSampler, mel_spectrogram  # noqa: F401
from .models import (LRELU_SLOPE, DiscriminatorP, DiscriminatorS, Generator,  # noqa: F401
                     MultiPeriodDiscriminator, MultiScaleDiscriminator, ResBlock1, ResBlock2,
                     discriminator_loss, feature_loss, generator_loss)
from .utils import (apply_weight_norm, get_padding, init_weights, load_checkpoint,  # noqa: F401
                    save_checkpoint, scan_checkpoint)

__version__ = "0.1.0"
