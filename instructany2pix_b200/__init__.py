"""B200-native (sm_100a) implementation of the InstructAny2Pix denoising hot path.

Drop-in modules behind the reference's own interfaces (see DESIGN.md / INTEGRATION.md):
``B200UNet`` (diffusers ``UNet2DConditionModel`` call surface + attention-processor plugin API),
``B200DDIMScheduler`` / ``B200DDPMScheduler``, ``B200Prior`` (``generate_diffusion``), plus the fused sampler, and the SDXL
prompt encoders ``B200CLIPTextModel`` / ``B200CLIPTextModelWithProjection`` with ``encode_prompt``.
All arithmetic on the hot path runs in hand-written CUDA kernels from ``libia2p_sm100a.so`` (C ABI:
``include/ia2p.h``); there is no PyTorch / CPU fallback.
"""
from ._lib import IA2PError, LIB_PATH  # noqa: F401

__all__ = ["IA2PError", "LIB_PATH", "B200CLIPTextModel", "B200CLIPTextModelWithProjection", "encode_prompt"]

_LAZY = {"B200CLIPTextModel": "text_encoder", "B200CLIPTextModelWithProjection": "text_encoder", "encode_prompt": "text_encoder"}


def __getattr__(name):
    """the torch-based modules load on first use, so importing the package stays cheap"""
    if name in _LAZY:
        import importlib
        return getattr(importlib.import_module(f".{_LAZY[name]}", __name__), name)
    raise AttributeError(name)
