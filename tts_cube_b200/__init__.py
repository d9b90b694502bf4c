"""tts_cube_b200 - B200-native (sm_100a) vocoder hot path for TTS-Cube.

Host side mirrors the reference's interfaces for this path:
  ``CubeGenerator``            drop-in for ``hifigan.models.Generator`` (hifigan/models.py:72-125)
  ``ParallelWaveNetVocoder``   ClariNet IAF student + UpsampleNet2 (weights shipped by the reference)
  ``WaveRNNVocoder`` / ``CubenetVocoder``  autoregressive WaveRNN path (cube/networks/modules.py:392-503, vocoder.py)
  ``MULAWOutput`` ...          output heads of ``cube/networks/loss.py``
  ``mel_spectrogram`` / ``MelVocoder``  log-mel front-ends (hifigan/meldataset.py:50-74, cube/io_utils/vocoder.py:54-62)
  ``synthesize``               batch entry (mel list -> audio), sharded over ranks under torchrun
  ``HifiganStream``            incremental HiFi-GAN sessions (``CubeGenerator.open_stream`` / ``step_streams``)
  ``languasito_inference_batch``  batch > 1 driver of the reference ``Languasito2``'s own modules (PyTorch glue, frontend.py)
All vocoder compute happens in libcube_vocoder.so (C ABI in include/cube_vocoder.h).
"""
from ._lib import CubeVocError, build_info, LIB_PATH  # noqa: F401
from .generator import CubeGenerator, install_into_cubegan  # noqa: F401
from .clarinet import ParallelWaveNetVocoder  # noqa: F401
from .heads import MULAWOutput, RAWOutput, MOLOutput, GaussianOutput  # noqa: F401
from .wavernn import WaveRNNVocoder, CubenetVocoder, UpsampleNet  # noqa: F401
from .api import synthesize, lpt_shard, cubegan_inference_batch  # noqa: F401
from .streaming import HifiganStream, step_streams  # noqa: F401
from .mel import MelSpectrogram, MelVocoder, mel_spectrogram, slaney_mel_basis  # noqa: F401
from .frontend import languasito_inference_batch, durations_to_frame_index, expand_rows  # noqa: F401

__version__ = "0.1.0"
