"""ctypes binding of libledb200.so (declared in include/ledb200.h).

The product path has NO CPU fallback: if the shared library is missing or a call fails,
`LedB200Error` is raised with the library's own message.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libledb200.so')

F32, BF16, U8, I64, I32 = 0, 1, 2, 3, 4
IMG_NCHW_F32, IMG_NCHW_U8, IMG_NHWC_U8 = 0, 1, 2

# every symbol include/ledb200.h declares (tests check the .so exports all of them)
SYMBOLS = [
    'ledb200_version', 'ledb200_last_error', 'ledb200_create', 'ledb200_destroy',
    'ledb200_set_param', 'ledb200_num_params', 'ledb200_param_name', 'ledb200_finalize',
    'ledb200_forward_infer', 'ledb200_backbone_forward', 'ledb200_head_forward', 'ledb200_head_infer',
    'ledb200_debug_fetch', 'ledb200_profile_ops', 'ledb200_op_info', 'ledb200_op_name', 'ledb200_plan_launches',
    'ledb200_head_fuse_argmax', 'ledb200_confusion_accumulate', 'ledb200_ohem_workspace_bytes',
    'ledb200_ohem_ce', 'ledb200_ohem_up_fwd', 'ledb200_ohem_up_bwd', 'ledb200_conv2d',
    'ledb200_train_packed_weight_floats', 'ledb200_train_pack_weight', 'ledb200_train_conv_fwd',
    'ledb200_train_conv_dgrad', 'ledb200_train_conv_wgrad', 'ledb200_train_bn_fwd', 'ledb200_train_bn_bwd',
    'ledb200_train_bn_reduce', 'ledb200_train_bn_fwd_apply', 'ledb200_train_bn_bwd_apply',
    'ledb200_train_bn_workspace_bytes', 'ledb200_train_wgrad_workspace_bytes',
    'ledb200_train_resize_fwd', 'ledb200_train_resize_bwd', 'ledb200_train_add_relu', 'ledb200_train_relu_bwd',
    'ledb200_train_avgpool_fwd', 'ledb200_train_avgpool_bwd', 'ledb200_train_copy_channels',
    'ledb200_train_layout', 'ledb200_train_sgd_step',
    'ledb200_train_conv_tc_ok', 'ledb200_train_packed_weight_tc_floats', 'ledb200_train_pack_weight_tc',
    'ledb200_train_conv_fwd_tc', 'ledb200_train_conv_dgrad_tc', 'ledb200_train_set_tf32_rounding', 'ledb200_train_set_tf32_passes', 'ledb200_train_set_wgrad_passes',
    'ledb200_peer_allreduce_buffer_bytes', 'ledb200_peer_allreduce_f64',
    'ledb200_train_stem_fwd', 'ledb200_train_stem_wgrad',
    'ledb200_train_wgrad_tc_workspace_bytes', 'ledb200_train_conv_wgrad_tc',
    'ledb200_sesp_param_floats', 'ledb200_sesp_forward',
    'ledb200_mfaf_param_floats', 'ledb200_mfaf_workspace_bytes', 'ledb200_mfaf_forward',
    'ledb200_getb_param_floats', 'ledb200_getb_create', 'ledb200_getb_destroy', 'ledb200_getb_forward',
    'ledb200_postprocess', 'ledb200_slide_accumulate', 'ledb200_slide_finalize', 'ledb200_slide_merge', 'ledb200_stack_pad',
    'ledb200_tta_merge', 'ledb200_crop_select', 'ledb200_train_augment', 'ledb200_view_resize',
    'ledb200_png_bound', 'ledb200_png_workspace_bytes', 'ledb200_png_encode',
    'ledb200_png_lut_bound', 'ledb200_png_encode_lut',
    'ledb200_png_rgb_bound', 'ledb200_png_rgb_workspace_bytes', 'ledb200_png_encode_rgb',
    'ledb200_seg_locate_workspace_bytes', 'ledb200_seg_label_locations', 'ledb200_seg_overlay',
    'ledb200_png_decode_workspace_bytes', 'ledb200_png_decode', 'ledb200_png_decode_host',
    'ledb200_png_decode_mode_workspace_bytes',
    'ledb200_cityscapes_out_ints', 'ledb200_cityscapes_workspace_bytes', 'ledb200_cityscapes_accumulate',
    'ledb200_jpeg_decode_workspace_bytes', 'ledb200_jpeg_decode', 'ledb200_jpeg_decode_host',
    'ledb200_seam_param_floats', 'ledb200_seam_workspace_bytes', 'ledb200_seam_forward',
    'ledb200_conv_layer_create', 'ledb200_conv_layer_forward', 'ledb200_conv_layer_destroy',
    'ledb200_avgpool2d', 'ledb200_resize_bilinear', 'ledb200_add_relu', 'ledb200_conv_layer_forward_image',
    'ledb200_dappm_create', 'ledb200_dappm_eligible', 'ledb200_dappm_forward', 'ledb200_dappm_destroy',
]


class LedB200Error(RuntimeError):
    pass


class Cfg(C.Structure):
    _fields_ = [('in_channels', C.c_int32), ('channels', C.c_int32), ('ppm_channels', C.c_int32),
                ('head_channels', C.c_int32), ('num_classes', C.c_int32),
                ('align_corners', C.c_int32), ('dtype', C.c_int32), ('device', C.c_int32),
                ('variant', C.c_int32), ('conv_backend', C.c_int32), ('mean', C.c_float * 3),
                ('std', C.c_float * 3), ('bgr_to_rgb', C.c_int32), ('reserved', C.c_int32 * 7)]


class TtaView(C.Structure):
    """ledb200_tta_view: image n of the view at logits + n * image_stride (fp32 elements); padding / flip to undo."""
    _fields_ = [('logits', C.c_void_p), ('image_stride', C.c_int64), ('H', C.c_int32), ('W', C.c_int32),
                ('pad_lrtb', C.c_int32 * 4), ('flip', C.c_int32)]


class AugSample(C.Structure):
    """ledb200_aug_sample: one sample's source buffers, resized size, candidate boxes, flip and photometric draws."""
    _fields_ = [('img', C.c_void_p), ('label', C.c_void_p), ('h', C.c_int32), ('w', C.c_int32),
                ('rh', C.c_int32), ('rw', C.c_int32), ('num_candidates', C.c_int32),
                ('offsets', (C.c_int32 * 2) * 11), ('flip', C.c_int32), ('contrast_mode', C.c_int32),
                ('brightness', C.c_int32), ('contrast', C.c_int32), ('saturation', C.c_int32), ('hue', C.c_int32),
                ('beta', C.c_float), ('contrast_alpha', C.c_float), ('saturation_alpha', C.c_float),
                ('hue_delta', C.c_int32)]


class ViewDesc(C.Structure):
    """ledb200_view_desc: one decoded uint8 [3,h,w] source, its resized size and the unflipped / flipped outputs."""
    _fields_ = [('src', C.c_void_p), ('out', C.c_void_p), ('out_flip', C.c_void_p), ('h', C.c_int32), ('w', C.c_int32),
                ('rh', C.c_int32), ('rw', C.c_int32)]


class PngFile(C.Structure):
    """ledb200_png_file: one PNG file (its bytes and size), its output and the IHDR's h, w and colour type."""
    _fields_ = [('data', C.c_void_p), ('size', C.c_int64), ('out', C.c_void_p), ('h', C.c_int32), ('w', C.c_int32),
                ('color_type', C.c_int32)]


class SegStamp(C.Structure):
    """ledb200_seg_stamp: one label stamp's image, panel, box in panel coordinates and byte offset of its pixels."""
    _fields_ = [('image', C.c_int32), ('panel', C.c_int32), ('x0', C.c_int32), ('y0', C.c_int32), ('w', C.c_int32),
                ('h', C.c_int32), ('offset', C.c_int64)]


PNG_COLOR, PNG_LABEL, PNG_GREY16 = 0, 1, 16
# ledb200_png_decode's per-file status codes (include/ledb200.h LEDB200_PNG_*)
PNG_STATUS = {
    1: 'signature or IHDR does not match the descriptor',
    2: 'malformed chunk layout (a chunk past the end of the file, a bad chunk name or order, an unknown critical '
       'chunk, or no IDAT / IEND)',
    3: 'CRC-32 mismatch in a critical chunk',
    4: 'palette image without a valid PLTE chunk',
    5: 'unsupported: the file has an eXIf chunk (EXIF orientation is not applied)',
    6: 'invalid zlib header, or data after the end of the zlib stream',
    7: 'invalid deflate data',
    8: 'the compressed data ends early',
    9: 'wrong number of decompressed bytes for the image size',
    10: 'Adler-32 mismatch of the decompressed data',
    11: 'invalid scanline filter type',
}


# ledb200_cityscapes_accumulate's per-image status bits (include/ledb200.h)
CITYSCAPES_STATUS = {
    1: 'a ground-truth labelId above 33 (unknown label)',
    2: 'a predicted labelId outside 0 .. 33 (unknown label)',
    4: 'an instance id whose class is not an instance class of the evaluation (cityscapesscripts raises KeyError)',
    8: 'an int64 prediction outside 0 .. 255',
}


class JpegFile(C.Structure):
    """ledb200_jpeg_file: one baseline JPEG file (its bytes and size), its output and the frame's h, w, components."""
    _fields_ = [('data', C.c_void_p), ('size', C.c_int64), ('out', C.c_void_p), ('h', C.c_int32), ('w', C.c_int32),
                ('components', C.c_int32)]


# ledb200_jpeg_decode's per-file status codes (include/ledb200.h LEDB200_JPEG_*)
JPEG_STATUS = {
    1: 'no SOI, or the frame header does not match the descriptor',
    2: 'malformed marker structure (a segment past the end of the file or of the wrong length, a marker out of '
       'place, or the scan not followed by EOI)',
    3: 'unsupported: not a baseline 8-bit interleaved YCbCr / grey file, or an Exif orientation other than 1',
    4: 'invalid or missing quantisation / Huffman table',
    5: 'invalid Huffman code in the entropy-coded data',
    6: 'the entropy-coded data ends early',
    7: 'restart marker out of sequence or missing',
    8: 'coefficient index past 63',
}


_lib = None


def get():
    """Load the library once; fail loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise LedB200Error(
            f'{LIB_PATH} is missing: build it with `python led-net_b200/build.py` '
            '(or __graft_entry__.build()).  There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    lib.ledb200_version.restype = C.c_int
    lib.ledb200_last_error.restype = C.c_char_p
    lib.ledb200_create.argtypes = [C.POINTER(Cfg), C.POINTER(vp)]
    lib.ledb200_destroy.argtypes = [vp]
    lib.ledb200_set_param.argtypes = [vp, C.c_char_p, vp, C.POINTER(i64), i32, i32]
    lib.ledb200_num_params.argtypes = [vp]
    lib.ledb200_param_name.argtypes = [vp, i32]
    lib.ledb200_param_name.restype = C.c_char_p
    lib.ledb200_finalize.argtypes = [vp]
    lib.ledb200_forward_infer.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32, vp, vp]
    lib.ledb200_backbone_forward.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.ledb200_head_forward.argtypes = [vp, vp, vp, vp] + [i32] * 7 + [vp, vp, vp, vp]
    lib.ledb200_head_infer.argtypes = [vp, vp, vp, vp] + [i32] * 7 + [vp, i32, vp, vp]
    lib.ledb200_debug_fetch.argtypes = [vp, C.c_char_p, vp, i64, C.POINTER(i32), vp]
    lib.ledb200_profile_ops.argtypes = [vp, i32, vp, i32, vp]
    lib.ledb200_op_name.argtypes = [vp, i32]
    lib.ledb200_op_info.argtypes = [vp, i32, C.POINTER(C.c_double)]
    lib.ledb200_op_name.restype = C.c_char_p
    lib.ledb200_plan_launches.argtypes = [vp]
    lib.ledb200_head_fuse_argmax.argtypes = [vp, vp, vp, i32] + [i32] * 8 + [vp, i32, vp, vp]
    lib.ledb200_confusion_accumulate.argtypes = [vp, vp, i32, i32, i64, i32, i32, vp, vp]
    lib.ledb200_ohem_workspace_bytes.argtypes = [i64]
    lib.ledb200_ohem_workspace_bytes.restype = i64
    lib.ledb200_ohem_ce.argtypes = [vp, vp, i32, i32, i32, i32, i32, f32, i64, f32, vp, vp, vp, vp, vp]
    lib.ledb200_ohem_up_fwd.argtypes = [vp, vp] + [i32] * 7 + [f32, i64, f32, vp, vp, vp, vp]
    lib.ledb200_ohem_up_bwd.argtypes = [vp, vp] + [i32] * 7 + [f32, vp, vp, vp, vp, vp]
    lib.ledb200_conv2d.argtypes = [vp, vp, vp, i32] + [i32] * 8 + [vp, vp, vp, vp, i32, i32, i32, i32, vp]
    lib.ledb200_train_packed_weight_floats.argtypes = [i32] * 4
    lib.ledb200_train_packed_weight_floats.restype = i64
    lib.ledb200_train_pack_weight.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    lib.ledb200_train_conv_fwd.argtypes = [vp, vp, vp, vp] + [i32] * 7 + [vp]
    lib.ledb200_train_conv_dgrad.argtypes = [vp, vp, vp] + [i32] * 7 + [vp]
    lib.ledb200_train_conv_wgrad.argtypes = [vp, vp, vp, vp] + [i32] * 7 + [vp, vp]
    lib.ledb200_train_set_tf32_rounding.argtypes = [i32]
    lib.ledb200_train_set_tf32_passes.argtypes = [i32]
    lib.ledb200_train_set_wgrad_passes.argtypes = [i32]
    lib.ledb200_train_stem_fwd.argtypes = [vp, vp, vp, vp] + [i32] * 6 + [vp]
    lib.ledb200_train_stem_wgrad.argtypes = [vp, vp, vp] + [i32] * 6 + [vp, vp]
    lib.ledb200_peer_allreduce_buffer_bytes.argtypes = [i32]
    lib.ledb200_peer_allreduce_buffer_bytes.restype = i64
    lib.ledb200_peer_allreduce_f64.argtypes = [vp, i32, i32, i32, vp, C.c_uint32, i32, vp, vp]
    lib.ledb200_train_wgrad_tc_workspace_bytes.argtypes = [i32] * 7
    lib.ledb200_train_wgrad_tc_workspace_bytes.restype = i64
    lib.ledb200_train_conv_wgrad_tc.argtypes = [vp, vp, vp] + [i32] * 7 + [vp, vp]
    lib.ledb200_train_conv_tc_ok.argtypes = [i32] * 8
    lib.ledb200_train_conv_tc_ok.restype = i32
    lib.ledb200_train_packed_weight_tc_floats.argtypes = [i32] * 4
    lib.ledb200_train_packed_weight_tc_floats.restype = i64
    lib.ledb200_train_pack_weight_tc.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    lib.ledb200_train_conv_fwd_tc.argtypes = [vp, vp, vp, vp] + [i32] * 7 + [vp]
    lib.ledb200_train_conv_dgrad_tc.argtypes = [vp, vp, vp] + [i32] * 7 + [vp]
    lib.ledb200_train_bn_fwd.argtypes = [vp] * 9 + [f32, f32, i32, i64, i32, vp, vp]
    lib.ledb200_train_bn_bwd.argtypes = [vp] * 10 + [i32, i64, i32, vp, vp]
    lib.ledb200_train_bn_workspace_bytes.argtypes = [i32]
    lib.ledb200_train_bn_workspace_bytes.restype = i64
    lib.ledb200_train_wgrad_workspace_bytes.argtypes = [i32, i32, i32]
    lib.ledb200_train_wgrad_workspace_bytes.restype = i64
    lib.ledb200_train_bn_reduce.argtypes = [vp] * 5 + [i32, i32, i64, i32, vp, vp]
    lib.ledb200_train_bn_fwd_apply.argtypes = [vp] * 9 + [f32, f32, i32, i64, C.c_double, i32, vp, vp]
    lib.ledb200_train_bn_bwd_apply.argtypes = [vp] * 10 + [i32, i64, C.c_double, i32, vp, vp]
    lib.ledb200_train_resize_fwd.argtypes = [vp, vp] + [i32] * 6 + [vp]
    lib.ledb200_train_resize_bwd.argtypes = [vp, vp] + [i32] * 6 + [vp]
    lib.ledb200_train_add_relu.argtypes = [vp, vp, vp, i32, i64, vp]
    lib.ledb200_train_relu_bwd.argtypes = [vp, vp, vp, i64, vp]
    lib.ledb200_train_avgpool_fwd.argtypes = [vp, vp] + [i32] * 9 + [vp]
    lib.ledb200_train_avgpool_bwd.argtypes = [vp, vp] + [i32] * 9 + [vp]
    lib.ledb200_train_copy_channels.argtypes = [vp, i32, i32, vp, i32, i32, i64, i32, vp]
    lib.ledb200_train_layout.argtypes = [vp, vp] + [i32] * 5 + [vp]
    lib.ledb200_train_sgd_step.argtypes = [vp, vp, vp, i64, f32, f32, f32, i32, f32, vp]
    lib.ledb200_sesp_param_floats.argtypes = [i32, i32]
    lib.ledb200_sesp_param_floats.restype = i64
    lib.ledb200_sesp_forward.argtypes = [vp, vp] + [i32] * 6 + [vp, i32, vp, vp]
    lib.ledb200_mfaf_param_floats.argtypes = [i32, i32]
    lib.ledb200_mfaf_param_floats.restype = i64
    lib.ledb200_mfaf_workspace_bytes.argtypes = [i32, i32]
    lib.ledb200_mfaf_workspace_bytes.restype = i64
    lib.ledb200_mfaf_forward.argtypes = [vp, vp, vp] + [i32] * 6 + [vp, vp, vp]
    lib.ledb200_getb_param_floats.argtypes = [i32, i32, i32]
    lib.ledb200_getb_param_floats.restype = i64
    lib.ledb200_getb_create.argtypes = [i32, i32, i32, i32, i32, vp, C.POINTER(vp)]
    lib.ledb200_getb_destroy.argtypes = [vp]
    lib.ledb200_getb_forward.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.ledb200_postprocess.argtypes = [vp, i32, i32, i32, vp, i32, i32, i32, i32, f32, vp, i32, vp, vp]
    lib.ledb200_slide_accumulate.argtypes = [vp, vp, vp] + [i32] * 8 + [vp]
    lib.ledb200_slide_finalize.argtypes = [vp, vp] + [i32] * 4 + [vp, i32, vp]
    lib.ledb200_slide_merge.argtypes = [vp, i32, vp, vp] + [i32] * 6 + [vp, vp, i32, vp]
    lib.ledb200_stack_pad.argtypes = [vp, i32, i32, i32, i32, vp, vp, f32, vp, i32, i32, vp, i32, vp, i32, vp]
    lib.ledb200_tta_merge.argtypes = [C.POINTER(TtaView)] + [i32] * 7 + [f32, vp, i32, vp, vp]
    lib.ledb200_crop_select.argtypes = [C.POINTER(AugSample)] + [i32] * 4 + [C.c_double, i32, vp, vp]
    lib.ledb200_train_augment.argtypes = [C.POINTER(AugSample)] + [i32] * 4 + [vp, i32, vp, vp, f32, vp, i32, i32, vp,
                                                                               i32, vp]
    lib.ledb200_view_resize.argtypes = [C.POINTER(ViewDesc)] + [i32] * 4 + [vp, vp, f32, vp]
    lib.ledb200_png_bound.argtypes = [i32, i32]
    lib.ledb200_png_bound.restype = i64
    lib.ledb200_png_workspace_bytes.argtypes = [i32, i32, i32]
    lib.ledb200_png_workspace_bytes.restype = i64
    lib.ledb200_png_encode.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.ledb200_png_lut_bound.argtypes = [i32, i32, i32]
    lib.ledb200_png_lut_bound.restype = i64
    lib.ledb200_png_encode_lut.argtypes = [vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp]
    lib.ledb200_png_rgb_bound.argtypes = [i32, i32]
    lib.ledb200_png_rgb_bound.restype = i64
    lib.ledb200_png_rgb_workspace_bytes.argtypes = [i32, i32, i32]
    lib.ledb200_png_rgb_workspace_bytes.restype = i64
    lib.ledb200_png_encode_rgb.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp]
    lib.ledb200_seg_locate_workspace_bytes.argtypes = [i32, i32, i32]
    lib.ledb200_seg_locate_workspace_bytes.restype = i64
    lib.ledb200_seg_label_locations.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.ledb200_seg_overlay.argtypes = [vp, vp, i32, vp, i32] + [i32] * 4 + [vp, vp, vp, i32, vp, i64, vp, vp]
    lib.ledb200_png_decode_mode_workspace_bytes.argtypes = [C.POINTER(PngFile), i32, i32]
    lib.ledb200_png_decode_mode_workspace_bytes.restype = i64
    lib.ledb200_cityscapes_out_ints.argtypes = [i32]
    lib.ledb200_cityscapes_out_ints.restype = i64
    lib.ledb200_cityscapes_workspace_bytes.argtypes = [i32]
    lib.ledb200_cityscapes_workspace_bytes.restype = i64
    lib.ledb200_cityscapes_accumulate.argtypes = [vp, i32, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.ledb200_png_decode_workspace_bytes.argtypes = [C.POINTER(PngFile), i32]
    lib.ledb200_png_decode_workspace_bytes.restype = i64
    lib.ledb200_png_decode.argtypes = [C.POINTER(PngFile), i32, i32, vp, vp, vp, vp]
    lib.ledb200_png_decode_host.argtypes = [C.POINTER(PngFile), i32, i32, vp, vp]
    lib.ledb200_jpeg_decode_workspace_bytes.argtypes = [C.POINTER(JpegFile), i32]
    lib.ledb200_jpeg_decode_workspace_bytes.restype = i64
    lib.ledb200_jpeg_decode.argtypes = [C.POINTER(JpegFile), i32, vp, vp, vp]
    lib.ledb200_jpeg_decode_host.argtypes = [C.POINTER(JpegFile), i32, vp]
    lib.ledb200_conv_layer_create.argtypes = [vp, vp, vp, vp] + [i32] * 5 + [C.POINTER(vp)]
    lib.ledb200_conv_layer_forward.argtypes = [vp, vp, vp, vp] + [i32] * 9 + [vp]
    lib.ledb200_conv_layer_destroy.argtypes = [vp]
    lib.ledb200_conv_layer_forward_image.argtypes = [vp, vp, i32, vp] + [i32] * 6 + [vp]
    lib.ledb200_dappm_create.argtypes = [i32, i32, i32, vp, vp, vp, vp, C.POINTER(vp)]
    lib.ledb200_dappm_eligible.argtypes = [i32] * 7
    lib.ledb200_dappm_forward.argtypes = [vp, vp, vp] + [i32] * 4 + [vp]
    lib.ledb200_dappm_destroy.argtypes = [vp]
    lib.ledb200_avgpool2d.argtypes = [vp, vp] + [i32] * 10 + [vp]
    lib.ledb200_resize_bilinear.argtypes = [vp, vp] + [i32] * 9 + [vp]
    lib.ledb200_add_relu.argtypes = [vp, vp, vp, i32, i64] + [i32] * 5 + [vp]
    lib.ledb200_seam_param_floats.argtypes = [i32]
    lib.ledb200_seam_param_floats.restype = i64
    lib.ledb200_seam_workspace_bytes.argtypes = [i32, i32, i32]
    lib.ledb200_seam_workspace_bytes.restype = i64
    lib.ledb200_seam_forward.argtypes = [vp, vp, vp] + [i32] * 5 + [f32, vp, vp, vp]
    for name in SYMBOLS:
        fn = getattr(lib, name)
        if fn.restype is C.c_int and name not in ('ledb200_version',):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc, what=''):
    if rc < 0:
        msg = get().ledb200_last_error()
        raise LedB200Error(f'{what} failed ({rc}): {msg.decode() if msg else "?"}')
    return rc


def stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def torch_dtype_code(t):
    import torch
    return {torch.float32: F32, torch.bfloat16: BF16, torch.uint8: U8, torch.int64: I64,
            torch.int32: I32}[t.dtype]
