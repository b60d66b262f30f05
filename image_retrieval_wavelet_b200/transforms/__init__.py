"""HP-SWT: mirrors ``main.transforms`` of the reference (``main/transforms/__init__.py:1``) for the SWT hot path."""
from .custom_transforms import BaseWaveletTransform, DWTTransform, RawStackTransform, SWTTransform, dwt2, resize_u8, swt2
from .jpeg import EncodedImages, collate_jpeg, collate_jpeg_train, decode_jpeg
from .ragged import RaggedImages, collate_ragged, collate_ragged_train, random_resized_crop_params, resize_center_crop, resize_random_crop_flip

__all__ = ["BaseWaveletTransform", "SWTTransform", "RawStackTransform", "DWTTransform", "swt2", "dwt2", "resize_u8",
           "RaggedImages", "collate_ragged", "resize_center_crop", "random_resized_crop_params", "collate_ragged_train",
           "resize_random_crop_flip", "EncodedImages", "collate_jpeg", "collate_jpeg_train", "decode_jpeg"]
