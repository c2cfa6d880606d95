"""parakeet.cpp_b200 -- B200-native Parakeet hot path behind the reference's API.

    PCM -> log-mel -> FastConformer encoder -> CTC / TDT / RNNT greedy decode

as hand-written sm_100a CUDA (csrc/) behind the C-ABI of include/parakeet_b200.h.
This Python package is only the ctypes binding + harness helpers; the C++
drop-in shim with the reference's class signatures is include/parakeet/transcribe.hpp.

(The directory name contains a dot, as the project brief names it; import it with
`__graft_entry__.load_package()` which registers it as module `parakeet_cpp_b200`.)
"""
from .engine import (Decoder, Engine, ModelConfig, TranscribeOptions, TranscribeResult, Transcriber,  # noqa: F401
                     TimestampedToken, WordTimestamp, lib_path, load_library, make_110m_config,
                     make_tdt_600m_config, make_tiny_config, make_eou_120m_config, make_tiny_stream_config,
                     make_rnnt_600m_config, make_tiny_rnnt_config)
