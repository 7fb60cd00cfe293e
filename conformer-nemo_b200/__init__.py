"""B200-native Conformer encoder forward (drop-in for nemo.collections.asr.modules.ConformerEncoder.forward).

The directory is named ``conformer-nemo_b200`` (not an identifier); import it through the repo-root shim
``conformer_nemo_b200`` which points ``__path__`` here.
"""
from .encoder import ConformerEncoder  # noqa: F401
from .config import instantiate_encoder, load_encoder_config  # noqa: F401
from .sharding import plan_shards, forward_sharded  # noqa: F401
from .ctc_head import ConvASRDecoder, ctc_collapse_device, ctc_greedy_decode  # noqa: F401
from .preprocessor import AudioToMelSpectrogramPreprocessor  # noqa: F401
from .rnnt import RNNTDecoder, RNNTJoint, GreedyBatchedRNNTInfer, GreedyRNNTInfer, Hypothesis  # noqa: F401
from .rnnt import BeamRNNTInfer, NBestHypotheses  # noqa: F401
from .collation import (BucketingIterator, CollationService, ManifestEntry, read_manifest, speech_collate)  # noqa: F401
from .buffered import FrameBatchASR, buffered_ctc_transcribe  # noqa: F401
from .buffered import BatchedFrameASRRNNT, buffered_rnnt_transcribe  # noqa: F401
