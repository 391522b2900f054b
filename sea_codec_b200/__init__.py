"""sea_codec_b200 -- B200-native (sm_100a) implementation of the SEA audio codec's encode/decode hot path.

The product is libsea_b200.so (C-ABI in include/sea_b200.h, kernels in csrc/); this package is the Python host-side
mirror of the reference crate's API on top of it.  See DESIGN.md and INTEGRATION.md.
"""
from .api import (Context, Corpus, EncoderSettings, MultiContext, SeaDecodeInfo, SeaDecoder, SeaEncoder, SeaError, SeaFileHeader, default_context,
                  lib, parse_header, sea_decode, sea_encode)

__all__ = ["Context", "Corpus", "EncoderSettings", "MultiContext", "SeaDecodeInfo", "SeaDecoder", "SeaEncoder", "SeaError", "SeaFileHeader",
           "default_context", "lib", "parse_header", "sea_decode", "sea_encode"]
