"""ctypes binding of libsymgpu.so (the in-tree build; never a site-packages copy)."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class NativeLibraryMissing(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "libsymgpu.so")


# numpy mirror of `symgpu_mp3_gc` (include/symgpu.h), 64 bytes
MP3_GC_DTYPE = np.dtype([
    ("rzero", "<u2"), ("global_gain", "u1"), ("block_type", "u1"), ("flags", "u1"),
    ("sample_rate_idx", "u1"), ("subblock_gain", "u1", (3,)), ("scalefacs", "u1", (39,)),
    ("reserved", "u1", (16,)),
])
assert MP3_GC_DTYPE.itemsize == 64
# `symgpu_mp3_run`, 16 bytes
MP3_RUN_DTYPE = np.dtype([
    ("stream", "<u4"), ("first_frame", "<u4"), ("n_frames", "<u4"),
    ("granules_per_frame", "u1"), ("channels", "u1"), ("reserved", "<u2"),
])
assert MP3_RUN_DTYPE.itemsize == 16

# `symgpu_mpa12_run`, 16 bytes (Layer I / II)
MPA12_RUN_DTYPE = np.dtype([("stream", "<u4"), ("first_frame", "<u4"), ("n_frames", "<u4"), ("channels", "u1"),
                            ("reserved", "u1", (3,))])
assert MPA12_RUN_DTYPE.itemsize == 16

# FLAC (include/symgpu.h): `symgpu_flac_subframe` 144 bytes, `symgpu_flac_frame` 16 bytes
FLAC_SUBFRAME_DTYPE = np.dtype([("offset", "<u8"), ("n", "<u4"), ("type", "u1"), ("order", "u1"), ("shift", "u1"),
                                ("wasted", "u1"), ("coeffs", "<i4", (32,))])
FLAC_FRAME_DTYPE = np.dtype([("first_subframe", "<u4"), ("channels", "u1"), ("assignment", "u1"), ("bits_per_sample", "u1"),
                             ("reserved", "u1"), ("reserved2", "<u4", (2,))])
assert FLAC_SUBFRAME_DTYPE.itemsize == 144 and FLAC_FRAME_DTYPE.itemsize == 16
FLAC_CONSTANT, FLAC_VERBATIM, FLAC_FIXED, FLAC_LPC = 0, 1, 2, 3
FLAC_INDEPENDENT, FLAC_LEFT_SIDE, FLAC_MID_SIDE, FLAC_RIGHT_SIDE = 0, 1, 2, 3

# AAC / Vorbis structs (include/symgpu.h)
AAC_UNIT_DTYPE = np.dtype([("window_sequence", "u1"), ("window_shape", "u1"), ("prev_window_shape", "u1"),
                           ("n_tns", "u1"), ("tns_first", "<u4"), ("reserved", "<u4", (2,))])
AAC_TNS_DTYPE = np.dtype([("start", "<u2"), ("end", "<u2"), ("order", "u1"), ("direction", "u1"), ("reserved", "<u2"),
                          ("lpc", "<f4", (20,))])
AAC_RUN_DTYPE = np.dtype([("stream", "<u4"), ("first_frame", "<u4"), ("n_frames", "<u4"), ("channels", "u1"),
                          ("reserved", "u1", (3,))])
VORBIS_FLOOR1_DTYPE = np.dtype([("multiplier", "u1"), ("n_posts", "u1"), ("x_list", "<u2", (65,)), ("low", "u1", (65,)),
                                ("high", "u1", (65,)), ("sort_order", "u1", (65,)), ("reserved", "u1", (5,))])
VORBIS_STREAM_DTYPE = np.dtype([("bs0_exp", "u1"), ("bs1_exp", "u1"), ("channels", "u1"), ("coupled", "u1")])
VORBIS_UNIT_DTYPE = np.dtype([("block_flag", "u1"), ("prev_block_flag", "u1"), ("do_not_decode", "u1", (2,)),
                              ("floor", "<u2", (2,)), ("reserved", "u1", (8,))])
VORBIS_RUN_DTYPE = np.dtype([("stream", "<u4"), ("first_packet", "<u4"), ("n_packets", "<u4"), ("reserved", "<u4")])
assert AAC_UNIT_DTYPE.itemsize == 16 and AAC_TNS_DTYPE.itemsize == 88 and AAC_RUN_DTYPE.itemsize == 16
VORBIS_STREAM_MC_DTYPE = np.dtype([("bs0_exp", "u1"), ("bs1_exp", "u1"), ("channels", "u1"), ("n_couplings", "u1"),
                                   ("magnitude_ch", "u1", (16,)), ("angle_ch", "u1", (16,))])
VORBIS_UNIT_MC_DTYPE = np.dtype([("block_flag", "u1"), ("prev_block_flag", "u1"), ("do_not_decode", "u1", (8,)), ("floor", "<u2", (8,)),
                                 ("reserved", "u1", (6,))])
assert VORBIS_STREAM_MC_DTYPE.itemsize == 36 and VORBIS_UNIT_MC_DTYPE.itemsize == 32
assert VORBIS_FLOOR1_DTYPE.itemsize == 332 and VORBIS_STREAM_DTYPE.itemsize == 4
assert VORBIS_UNIT_DTYPE.itemsize == 16 and VORBIS_RUN_DTYPE.itemsize == 16
# `symgpu_pcm_span`, 32 bytes; sample formats of the output stage
PCM_SPAN_DTYPE = np.dtype([("src", "<u8"), ("plane_stride", "<u4"), ("frames", "<u4"), ("trim_start", "<u4"),
                           ("trim_end", "<u4"), ("dst_frame", "<u8")])
assert PCM_SPAN_DTYPE.itemsize == 32
AAC_ASC_DTYPE = np.dtype([("sample_rate", "<u4"), ("ext_sample_rate", "<u4"), ("samples", "<u2"), ("object_type", "u1"), ("channels", "u1"),
                          ("sbr_present", "u1"), ("ps_present", "u1"), ("has_ext", "u1"), ("ext_channels", "u1"), ("reserved", "u1", (8,))])
assert AAC_ASC_DTYPE.itemsize == 24
FMT_F32, FMT_S16, FMT_S24, FMT_S32, FMT_U8 = 0, 1, 2, 3, 4
FMT_NUMPY = {FMT_F32: np.float32, FMT_S16: np.int16, FMT_S24: np.int32, FMT_S32: np.int32, FMT_U8: np.uint8}
# packetisers (include/symgpu.h "Packetisers")
MPA_TRACK_DTYPE = np.dtype([("first_header", "<u4"), ("sample_rate", "<u4"), ("version", "u1"), ("layer", "u1"), ("channels", "u1"),
                            ("tag", "u1"), ("has_delay", "u1"), ("has_num_frames", "u1"), ("reserved", "u1", (2,)), ("delay", "<u4"),
                            ("padding", "<u4"), ("reserved2", "<u4", (2,)), ("num_frames", "<u8"), ("first_packet_pos", "<u8")])
MPA_PACKET_DTYPE = np.dtype([("offset", "<u8"), ("size", "<u4"), ("header", "<u4"), ("pts", "<i8"), ("dur", "<u4"), ("trim_start", "<u4"),
                             ("trim_end", "<u8"), ("main_data_begin", "<i4"), ("reserved", "<u4")])
ADTS_PACKET_DTYPE = np.dtype([("offset", "<u8"), ("size", "<u4"), ("sample_rate", "<u4"), ("pts", "<i8"), ("channels", "u1"),
                              ("profile", "u1"), ("reserved", "u1", (6,))])
PIECE_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("reserved", "<u4")])
OGG_PACKET_DTYPE = np.dtype([("serial", "<u4"), ("page_sequence", "<u4"), ("page_absgp", "<u8"), ("len", "<u8"), ("first_piece", "<u4"),
                             ("n_pieces", "<u4"), ("last_on_page", "u1"), ("reserved", "u1", (7,))])
VORBIS_IDENT_DTYPE = np.dtype([("sample_rate", "<u4"), ("channels", "u1"), ("bs0_exp", "u1"), ("bs1_exp", "u1"), ("reserved", "u1")])
assert MPA_TRACK_DTYPE.itemsize == 48 and MPA_PACKET_DTYPE.itemsize == 48 and ADTS_PACKET_DTYPE.itemsize == 32
MP3_FRAME_INFO_DTYPE = np.dtype([("sample_rate", "<u4"), ("channels", "u1"), ("granules", "u1"), ("sample_rate_idx", "u1"), ("version", "u1"),
                                 ("underflow_bytes", "<u4"), ("main_data_bytes", "<u4")])
assert MP3_FRAME_INFO_DTYPE.itemsize == 16
FLAC_FRAME_INFO_DTYPE = np.dtype([("sequence", "<u8"), ("block_size", "<u4"), ("sample_rate", "<u4"), ("by_sample", "u1"), ("reserved", "u1", (7,))])
assert FLAC_FRAME_INFO_DTYPE.itemsize == 24
FLAC_STREAM_INFO_DTYPE = np.dtype([("n_samples", "<u8"), ("first_frame_pos", "<u8"), ("sample_rate", "<u4"), ("frame_min", "<u4"), ("frame_max", "<u4"),
                                   ("block_min", "<u2"), ("block_max", "<u2"), ("channels", "u1"), ("bits_per_sample", "u1"), ("has_md5", "u1"),
                                   ("reserved", "u1"), ("md5", "u1", (16,)), ("reserved2", "u1", (4,))])
FLAC_PACKET_DTYPE = np.dtype([("offset", "<u8"), ("ts", "<u8"), ("size", "<u4"), ("dur", "<u4")])
assert FLAC_STREAM_INFO_DTYPE.itemsize == 56 and FLAC_PACKET_DTYPE.itemsize == 24
MP3_FILE_DTYPE = np.dtype([("data", "<u8"), ("n", "<u8"), ("packets", "<u8"), ("n_packets", "<u8"), ("stream", "<u4"), ("reserved", "<u4")])
assert MP3_FILE_DTYPE.itemsize == 40
VORBIS_SETUP_INFO_DTYPE = np.dtype([("n_codebooks", "<u4"), ("n_floors", "<u4"), ("n_residues", "<u4"), ("n_mappings", "<u4"), ("n_modes", "<u4"),
                                    ("reserved", "<u4"), ("long_block_mask", "<u8"), ("mode_mapping", "u1", (64,)), ("floor_type", "u1", (64,))])
assert VORBIS_SETUP_INFO_DTYPE.itemsize == 160
assert PIECE_DTYPE.itemsize == 16 and OGG_PACKET_DTYPE.itemsize == 40 and VORBIS_IDENT_DTYPE.itemsize == 8
AAC_ONLY_LONG, AAC_LONG_START, AAC_EIGHT_SHORT, AAC_LONG_STOP = 0, 1, 2, 3

MP3_LONG, MP3_START, MP3_SHORT, MP3_END = 0, 1, 2, 3
F_MIXED, F_SCALEFAC_SCALE, F_PREFLAG, F_SFC_LSB = 1, 2, 4, 8
F_MID_SIDE, F_INTENSITY, F_MPEG1, F_MUTE = 16, 32, 64, 128


def lib():
    """Loads the library; raises NativeLibraryMissing (never falls back to anything)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise NativeLibraryMissing(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C symphonia_b200/csrc`). There is no CPU fallback.")
    L = ctypes.CDLL(path)
    vp, u32, sz = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_size_t
    L.symgpu_abi_version.restype = ctypes.c_int
    L.symgpu_strerror.restype = ctypes.c_char_p
    L.symgpu_strerror.argtypes = [ctypes.c_int]
    L.symgpu_last_cuda_error.restype = ctypes.c_char_p
    L.symgpu_last_cuda_error.argtypes = [vp]
    L.symgpu_ctx_create.restype = ctypes.c_int
    L.symgpu_ctx_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    L.symgpu_ctx_destroy.restype = None
    L.symgpu_ctx_destroy.argtypes = [vp]
    L.symgpu_tables_host_blob.restype = sz
    L.symgpu_tables_host_blob.argtypes = [vp, sz]
    L.symgpu_codec_tables_host_blob.restype = sz
    L.symgpu_codec_tables_host_blob.argtypes = [vp, sz]
    L.symgpu_tables_upload.restype = ctypes.c_int
    L.symgpu_tables_upload.argtypes = [vp, vp, sz]
    L.symgpu_sync.restype = ctypes.c_int
    L.symgpu_sync.argtypes = [vp]
    L.symgpu_cuda_stream.restype = vp
    L.symgpu_cuda_stream.argtypes = [vp]
    L.symgpu_launch_count.restype = ctypes.c_uint64
    L.symgpu_launch_count.argtypes = [vp]
    L.symgpu_mp3_pow43.restype = sz
    L.symgpu_mp3_pow43.argtypes = [vp, sz]
    L.symgpu_mp3_streams_alloc.restype = ctypes.c_int
    L.symgpu_mp3_streams_alloc.argtypes = [vp, u32]
    L.symgpu_mp3_stream_reset.restype = ctypes.c_int
    L.symgpu_mp3_stream_reset.argtypes = [vp, u32]
    for name in ("symgpu_mp3_synth_host", "symgpu_mp3_synth_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, vp, u32, u32, vp]
    L.symgpu_aac_streams_alloc.restype = ctypes.c_int
    L.symgpu_aac_streams_alloc.argtypes = [vp, u32]
    L.symgpu_aac_stream_reset.restype = ctypes.c_int
    L.symgpu_aac_stream_reset.argtypes = [vp, u32]
    for name in ("symgpu_aac_synth_host", "symgpu_aac_synth_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, u32, vp, vp, u32, u32, vp]
    L.symgpu_vorbis_streams_set.restype = ctypes.c_int
    L.symgpu_vorbis_streams_set.argtypes = [vp, vp, u32]
    L.symgpu_vorbis_floors_set.restype = ctypes.c_int
    L.symgpu_vorbis_floors_set.argtypes = [vp, vp, u32]
    L.symgpu_vorbis_stream_reset.restype = ctypes.c_int
    L.symgpu_vorbis_stream_reset.argtypes = [vp, u32]
    for name in ("symgpu_vorbis_synth_host", "symgpu_vorbis_synth_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, vp, vp, u32, u32, u32, vp]
    L.symgpu_vorbis_mc_streams_set.restype = ctypes.c_int
    L.symgpu_vorbis_mc_streams_set.argtypes = [vp, vp, u32]
    for name in ("symgpu_vorbis_mc_synth_host", "symgpu_vorbis_mc_synth_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, vp, vp, u32, u32, u32, u32, vp]
    L.symgpu_sample_bytes.restype = sz
    L.symgpu_sample_bytes.argtypes = [ctypes.c_int]
    L.symgpu_pcm_pack_dev.restype = ctypes.c_int
    L.symgpu_pcm_pack_dev.argtypes = [vp, vp, vp, u32, u32, u32, u32, ctypes.c_int, vp]
    L.symgpu_pcm_pack_host.restype = ctypes.c_int
    L.symgpu_pcm_pack_host.argtypes = [vp, vp, sz, vp, u32, u32, u32, u32, ctypes.c_int, vp, sz]
    L.symgpu_mp3_synth_host_packed.restype = ctypes.c_int
    L.symgpu_mp3_synth_host_packed.argtypes = [vp, vp, vp, vp, u32, u32, ctypes.c_int, vp]
    for name in ("symgpu_mpa12_synth_host", "symgpu_mpa12_synth_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, vp, u32, u32, u32, vp]
    for name in ("symgpu_flac_restore_host", "symgpu_flac_restore_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, u32, vp, u32, vp, sz]
    for name in ("symgpu_flac_decode_host", "symgpu_flac_decode_dev"):
        fn = getattr(L, name)
        fn.restype = ctypes.c_int
        fn.argtypes = [vp, vp, u32, vp, u32, vp, sz, vp, ctypes.c_int, vp, sz]
    L.symgpu_mp3_units_check.restype = ctypes.c_int
    L.symgpu_mp3_units_check.argtypes = [vp, vp, u32, u32]
    L.symgpu_aac_units_check.restype = ctypes.c_int
    L.symgpu_aac_units_check.argtypes = [vp, vp, u32, u32]
    L.symgpu_mp3_synth_host_quantized.restype = ctypes.c_int
    L.symgpu_mp3_synth_host_quantized.argtypes = [vp, vp, vp, vp, u32, u32, ctypes.c_int, vp]
    psz = ctypes.POINTER(sz)
    L.symgpu_mpa_index.restype = ctypes.c_int
    L.symgpu_mpa_index.argtypes = [vp, sz, ctypes.c_int, vp, vp, sz, psz]
    L.symgpu_adts_index.restype = ctypes.c_int
    L.symgpu_adts_index.argtypes = [vp, sz, vp, sz, psz, ctypes.POINTER(ctypes.c_int)]
    L.symgpu_ogg_index.restype = ctypes.c_int
    L.symgpu_ogg_index.argtypes = [vp, sz, vp, sz, psz, vp, sz, psz]
    L.symgpu_vorbis_ident_parse.restype = ctypes.c_int
    L.symgpu_vorbis_ident_parse.argtypes = [vp, sz, vp]
    L.symgpu_vorbis_setup_modes.restype = ctypes.c_int
    L.symgpu_vorbis_setup_modes.argtypes = [vp, sz, vp, ctypes.POINTER(u32), ctypes.POINTER(ctypes.c_uint64)]
    L.symgpu_vorbis_setup_parse.restype = ctypes.c_int
    L.symgpu_vorbis_setup_parse.argtypes = [vp, sz, vp, vp, vp]
    L.symgpu_vorbis_packet_durations.restype = ctypes.c_int
    L.symgpu_vorbis_packet_durations.argtypes = [vp, u32, ctypes.c_uint64, vp, vp, sz, vp, vp, vp]
    L.symgpu_mp3_fe_create.restype = ctypes.c_int
    L.symgpu_mp3_fe_create.argtypes = [ctypes.POINTER(vp)]
    L.symgpu_mp3_fe_destroy.restype = None
    L.symgpu_mp3_fe_destroy.argtypes = [vp]
    L.symgpu_mp3_fe_reset.restype = None
    L.symgpu_mp3_fe_reset.argtypes = [vp]
    L.symgpu_mp3_fe_decode.restype = ctypes.c_int
    L.symgpu_mp3_fe_decode.argtypes = [vp, vp, sz, vp, vp, vp]
    L.symgpu_mp3_fe_decode_packets.restype = ctypes.c_int
    L.symgpu_mp3_fe_decode_packets.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp, psz, vp]
    L.symgpu_mp3_entropy_plan.restype = ctypes.c_int
    L.symgpu_mp3_entropy_plan.argtypes = [vp, sz, vp, sz, vp, vp, sz, psz, vp, vp, psz, vp]
    L.symgpu_mp3_entropy_run_cpu.restype = ctypes.c_int
    L.symgpu_mp3_entropy_run_cpu.argtypes = [vp, sz, vp, sz, vp, vp, vp]
    L.symgpu_mp3_entropy_run_cpu_mt.restype = ctypes.c_int
    L.symgpu_mp3_entropy_run_cpu_mt.argtypes = [vp, sz, vp, sz, vp, vp, vp, u32]
    L.symgpu_mp3_entropy_decode_cpu.restype = ctypes.c_int
    L.symgpu_mp3_entropy_decode_cpu.argtypes = [vp, sz, vp, sz, vp, vp, vp, psz, vp, ctypes.POINTER(u32)]
    L.symgpu_mp3_entropy_dev.restype = ctypes.c_int
    L.symgpu_mp3_entropy_dev.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp]
    L.symgpu_mp3_decode_files_host.restype = ctypes.c_int
    L.symgpu_mp3_decode_files_host.argtypes = [vp, vp, u32, vp, sz, vp, vp, ctypes.POINTER(u32)]
    L.symgpu_mpa12_fe_decode.restype = ctypes.c_int
    L.symgpu_mpa12_fe_decode.argtypes = [vp, sz, ctypes.c_int, vp, vp]
    L.symgpu_mpa12_fe_decode_packets.restype = ctypes.c_int
    L.symgpu_mpa12_fe_decode_packets.argtypes = [vp, sz, vp, sz, ctypes.c_int, vp, vp, psz, vp]
    L.symgpu_mpa12_constants.restype = sz
    L.symgpu_mpa12_constants.argtypes = [vp, sz]
    L.symgpu_flac_fe_decode_packets.restype = ctypes.c_int
    L.symgpu_flac_fe_decode_packets.argtypes = [vp, sz, vp, sz, u32, u32, u32, vp, vp, vp, vp, sz, vp, sz, psz, psz, psz]
    L.symgpu_flac_index.restype = ctypes.c_int
    L.symgpu_flac_index.argtypes = [vp, sz, vp, vp, sz, psz]
    L.symgpu_vorbis_fe_create.restype = ctypes.c_int
    L.symgpu_vorbis_fe_create.argtypes = [vp, sz, vp, sz, ctypes.POINTER(vp)]
    L.symgpu_vorbis_fe_destroy.restype = None
    L.symgpu_vorbis_fe_destroy.argtypes = [vp]
    L.symgpu_vorbis_fe_reset.restype = None
    L.symgpu_vorbis_fe_reset.argtypes = [vp]
    L.symgpu_vorbis_fe_config.restype = ctypes.c_int
    L.symgpu_vorbis_fe_config.argtypes = [vp, vp, vp, ctypes.POINTER(u32)]
    L.symgpu_vorbis_fe_decode.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode.argtypes = [vp, vp, sz, u32, u32, vp, vp, vp]
    L.symgpu_ogg_gather.restype = ctypes.c_int
    L.symgpu_ogg_gather.argtypes = [vp, sz, vp, sz, vp, sz, vp, sz, vp, ctypes.POINTER(sz)]
    L.symgpu_ogg_page_end_trims.restype = ctypes.c_int
    L.symgpu_ogg_page_end_trims.argtypes = [vp, vp, vp, vp, sz, vp]
    L.symgpu_aac_fe_create.restype = ctypes.c_int
    L.symgpu_aac_fe_create.argtypes = [u32, u32, ctypes.POINTER(vp)]
    L.symgpu_aac_asc_parse.restype = ctypes.c_int
    L.symgpu_aac_asc_parse.argtypes = [vp, sz, vp]
    L.symgpu_aac_fe_create_asc.restype = ctypes.c_int
    L.symgpu_aac_fe_create_asc.argtypes = [vp, sz, ctypes.POINTER(vp), vp]
    L.symgpu_aac_fe_destroy.restype = None
    L.symgpu_aac_fe_destroy.argtypes = [vp]
    L.symgpu_aac_fe_reset.restype = None
    L.symgpu_aac_fe_reset.argtypes = [vp]
    L.symgpu_aac_fe_decode.restype = ctypes.c_int
    L.symgpu_aac_fe_decode.argtypes = [vp, vp, sz, u32, vp, vp, ctypes.POINTER(u32), vp]
    L.symgpu_aac_fe_decode_packets.restype = ctypes.c_int
    L.symgpu_aac_fe_decode_packets.argtypes = [vp, vp, sz, vp, sz, u32, vp, vp, sz, vp, vp, ctypes.POINTER(sz), ctypes.POINTER(sz)]
    L.symgpu_vorbis_fe_decode_packets.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode_packets.argtypes = [vp, vp, sz, vp, sz, u32, u32, vp, vp, vp, vp, ctypes.POINTER(sz)]
    L.symgpu_aac_fe_decode_packets_jobs.restype = ctypes.c_int
    L.symgpu_aac_fe_decode_packets_jobs.argtypes = [u32, u32, vp, sz, vp, sz, u32, vp, vp, sz, vp, ctypes.POINTER(sz), u32]
    L.symgpu_vorbis_fe_decode_packets_jobs.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode_packets_jobs.argtypes = [vp, sz, vp, sz, vp, sz, vp, sz, u32, u32, vp, vp, vp, vp, ctypes.POINTER(sz), u32]
    L.symgpu_vorbis_fe_create_mc.restype = ctypes.c_int
    L.symgpu_vorbis_fe_create_mc.argtypes = [vp, sz, vp, sz, ctypes.POINTER(vp)]
    L.symgpu_vorbis_fe_config_mc.restype = ctypes.c_int
    L.symgpu_vorbis_fe_config_mc.argtypes = [vp, vp, vp, ctypes.POINTER(u32)]
    L.symgpu_vorbis_fe_decode_mc.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode_mc.argtypes = [vp, vp, sz, u32, u32, u32, vp, vp, vp]
    L.symgpu_vorbis_fe_decode_packets_mc.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode_packets_mc.argtypes = [vp, vp, sz, vp, sz, u32, u32, u32, vp, vp, vp, vp, ctypes.POINTER(sz)]
    L.symgpu_vorbis_fe_decode_packets_jobs_mc.restype = ctypes.c_int
    L.symgpu_vorbis_fe_decode_packets_jobs_mc.argtypes = [vp, sz, vp, sz, vp, sz, vp, sz, u32, u32, u32, vp, vp, vp, vp, ctypes.POINTER(sz), u32]
    L.symgpu_vorbis_channel_map.restype = ctypes.c_int
    L.symgpu_vorbis_channel_map.argtypes = [u32, vp]
    L.symgpu_pcm_pack_mapped_dev.restype = ctypes.c_int
    L.symgpu_pcm_pack_mapped_dev.argtypes = [vp, vp, vp, u32, u32, u32, u32, vp, ctypes.c_int, vp]
    L.symgpu_pcm_pack_mapped_host.restype = ctypes.c_int
    L.symgpu_pcm_pack_mapped_host.argtypes = [vp, vp, sz, vp, u32, u32, u32, u32, vp, ctypes.c_int, vp, sz]
    L.symgpu_aac_fe_tables.restype = None
    L.symgpu_aac_fe_tables.argtypes = [vp, vp, vp]
    _LIB = L
    return L


def mp3_pow43():
    out = np.zeros(8207, dtype=np.float32)
    lib().symgpu_mp3_pow43(out.ctypes.data_as(ctypes.c_void_p), 8207)
    return out
