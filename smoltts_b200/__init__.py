"""smoltts_b200 -- B200-native DualAR / RQ-Transformer decode step for SmolTTS checkpoints.

Importing the package is cheap and CPU-safe (config, synthetic inputs, the build script);
``RQTransformer`` and the generate API need a CUDA device and the in-tree CUDA library and raise
otherwise -- there is no CPU or eager-PyTorch fallback.
"""
from .config import MODEL_SIZES, RQTransformerModelArgs, named_config  # noqa: F401
from .generate import (  # noqa: F401
    GenerationSettings,
    SingleBatchGenerator,
    VQToken,
    generate_batch,
    generate_blocking,
)
from .model import (  # noqa: F401
    DecodeBatch,
    FastCache,
    RQTransformer,
    SlowCache,
    TokenConfig,
    make_prompt_cache,
)

from .serving import ContinuousBatcher, PromptEncoder, byte_level_tokenizer  # noqa: F401,E402
from .shard import ShardedGenerator, generate_sharded  # noqa: F401,E402
from .mimi import MimiCache, MimiConfig, MimiModel, load_mimi  # noqa: F401,E402
from .resample import Resampler, design_filter  # noqa: F401,E402
from .tts import SmolTTS  # noqa: F401,E402

__version__ = "0.1.0"
