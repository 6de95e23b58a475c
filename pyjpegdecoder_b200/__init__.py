"""pyjpegdecoder_b200 -- B200-native JPEG decode path behind PyJpegDecoder's entry point.

    from pyjpegdecoder_b200 import JpegDecoder
    img = JpegDecoder("photo.jpg").image_array          # uint8 (width, height, 3), like the reference
    x = decode_to_tensor(paths, size=(224, 224))         # (N, 3, 224, 224) float32 batch on the device

Host code (marker/segment parsing) is Python; entropy decode, IDCT, upsampling and colour conversion
are hand-written sm_100a CUDA kernels in libb200jpeg.so behind a C ABI (include/b200jpeg.h).
No CPU fallback: without the CUDA library or a GPU the decoder raises NativeLibraryError.
"""
from .errors import CorruptedJpeg, JpegError, NativeLibraryError, NotJpeg, UnsupportedJpeg
from .parser import parse_jpeg

__all__ = ["JpegDecoder", "decode_batch", "decode_stream", "decode_to_tensor", "decode_files_multi_gpu", "parse_jpeg", "JpegError", "NotJpeg",
           "CorruptedJpeg", "UnsupportedJpeg", "NativeLibraryError"]


def __getattr__(name):
    # torch is imported lazily so that the parser can be used without it
    if name in ("JpegDecoder", "decode_batch"):
        from . import decoder
        return getattr(decoder, name)
    if name == "decode_stream":
        from .loader import decode_stream
        return decode_stream
    if name == "decode_to_tensor":
        from .tensor_out import decode_to_tensor
        return decode_to_tensor
    if name == "decode_files_multi_gpu":
        from .multigpu import decode_files_multi_gpu
        return decode_files_multi_gpu
    raise AttributeError(name)
