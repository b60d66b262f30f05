"""HP-SWT: mirrors ``main.transforms`` of the reference (``main/transforms/__init__.py:1``) for the SWT hot path."""
from .custom_transforms import BaseWaveletTransform, DWTTransform, RawStackTransform, SWTTransform, dwt2, resize_u8, swt2
from .ragged import RaggedImages, collate_ragged, resize_center_crop

__all__ = ["BaseWaveletTransform", "SWTTransform", "RawStackTransform", "DWTTransform", "swt2", "dwt2", "resize_u8",
           "RaggedImages", "collate_ragged", "resize_center_crop"]
