/*
 * symgpu.h -- C ABI of libsymgpu.so, the B200 (sm_100a) batched audio-synthesis engine that
 * replaces the f32 DSP back-end of Symphonia's MP3 / AAC-LC / Vorbis decoders.
 *
 * The seam this ABI sits on is the point inside each reference decoder where the serial
 * bit-reader stage ends and the data-parallel synthesis stage begins:
 *
 *   MP3    symphonia-bundle-mp3/src/layer3/mod.rs:408 (read_main_data) | :421-477 (granule loop)
 *   AAC    symphonia-codec-aac/src/aac/mod.rs:217-220 -> ics/mod.rs:449-468 (Ics::synth_channel)
 *   Vorbis symphonia-codec-vorbis/src/lib.rs:248 (read_residue) | :250-315 (coupling/dot/synth)
 *
 * Everything left of the seam (frame sync, side info, Huffman / VQ decode) stays on the CPU in
 * the caller; everything right of it runs in one fused CUDA kernel per codec.  All entry points
 * take plain pointers and sizes.  "host" pointers are ordinary (ideally pinned) host memory and
 * the call performs the H2D / D2H copies itself; "dev" entry points take device pointers and
 * only enqueue the kernel on the context's CUDA stream (used when the spectra are already
 * resident in HBM).
 *
 * Error model (replaces symphonia_core::errors::Error, symphonia-core/src/errors.rs:43-57):
 * every function returns a symgpu_status; symgpu_strerror() returns a static string so a Rust
 * adapter can wrap it in Error::DecodeError(&'static str).  No C++ exception crosses the ABI.
 *
 * Threading (AudioDecoder: Send + Sync, symphonia-core/src/codecs/audio.rs:251): a context owns
 * one CUDA stream; calls on one context must be serialised by the caller (the trait's &mut self
 * already guarantees that per decoder).  Different contexts may be used concurrently.  The exception is
 * symgpu_mp3_submit / symgpu_mp3_submit_quantized / symgpu_mp3_wait: any number of decoder threads may call
 * them on ONE context at the same time, and the context gathers their frames into shared launches.
 */
#ifndef SYMGPU_H
#define SYMGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SYMGPU_ABI_VERSION 1

typedef enum symgpu_status {
    SYMGPU_OK = 0,
    SYMGPU_ERR_DECODE = 1,       /* Error::DecodeError  - malformed unit, caller drops packet   */
    SYMGPU_ERR_UNSUPPORTED = 2,  /* Error::Unsupported                                          */
    SYMGPU_ERR_LIMIT = 3,        /* Error::LimitError   - batch / stream limits exceeded        */
    SYMGPU_ERR_RESET = 4,        /* Error::ResetRequired                                        */
    SYMGPU_ERR_CUDA = 5,         /* device failure (sticky; context must be destroyed)          */
    SYMGPU_ERR_ARG = 6           /* null pointer / bad size - a bug in the caller               */
} symgpu_status;

typedef struct symgpu_ctx symgpu_ctx; /* opaque */

/* ---- context ------------------------------------------------------------------------------ */

/* Creates a context on CUDA device `device` (cudaSetDevice ordinal), builds every lookup table
 * on the host with libm (see DESIGN.md "tables") and uploads them.  Fails with SYMGPU_ERR_CUDA
 * when no usable sm_100 device is present: there is NO CPU fallback behind this ABI.
 * The calling thread is bound to the CPUs of the device's NUMA node (sysfs numa_node of the PCI device, intersected
 * with the thread's current affinity), so that pinned host buffers it allocates afterwards are node-local by first
 * touch -- one rank per GPU on a two-socket B200 node otherwise pushes half of its PCIe traffic across the socket link.
 * SYMGPU_NUMA_BIND=0 in the environment switches this off. */
symgpu_status symgpu_ctx_create(int device, symgpu_ctx** out);
/* NUMA node of CUDA device `device` (-1 if the platform does not say); binds the calling thread to that node's CPUs and
 * returns the node (-1 if nothing was changed); node a context bound its creating thread to (-1 none, -2 switched off). */
int symgpu_numa_node_of_device(int device);
int symgpu_bind_thread_to_device_numa(int device);
int symgpu_ctx_numa_node(const symgpu_ctx* ctx);
void symgpu_ctx_destroy(symgpu_ctx* ctx);

/* Static description of `status`. */
const char* symgpu_strerror(symgpu_status status);
/* Last CUDA error text seen by this context (static storage inside the context). */
const char* symgpu_last_cuda_error(const symgpu_ctx* ctx);
int symgpu_abi_version(void);

/* The host-built table blob (f32 words) exactly as uploaded, so that ranks can broadcast it
 * (ncclBroadcast / torch.distributed.broadcast) and tests can compare it with the oracle's
 * tables without a GPU.  Returns the number of bytes; `out` may be NULL to query the size. */
size_t symgpu_tables_host_blob(void* out, size_t cap);
/* Same for the tables of the power-of-two IMDCT codecs (FFT / IMDCT twiddles, AAC and Vorbis windows,
 * floor1 inverse-dB table); layout = struct CodecTables of symphonia_b200/csrc/tables.h. */
size_t symgpu_codec_tables_host_blob(void* out, size_t cap);
/* Replace the device tables of `ctx` with a blob received from rank 0. */
symgpu_status symgpu_tables_upload(symgpu_ctx* ctx, const void* blob, size_t bytes);
/* The same exchange without leaving the library: broadcasts the table blobs (MP3 and AAC / Vorbis) from rank `root` of
 * `nccl_comm` -- an ncclComm_t the host application created, passed as void* so that this header needs no nccl.h -- in
 * place over NCCL on the context's stream, and refreshes the constant-memory copies.  NULL: single GPU, nothing to do.
 * libnccl.so.2 is looked up with dlopen on first use (no link-time dependency); SYMGPU_ERR_UNSUPPORTED if it is absent.
 * Collective: every rank of the communicator must call it. */
symgpu_status symgpu_tables_broadcast(symgpu_ctx* ctx, void* nccl_comm, int root);

/* Blocks until every kernel / copy enqueued on the context's stream has finished. */
symgpu_status symgpu_sync(symgpu_ctx* ctx);
/* The context's cudaStream_t, as an opaque pointer (for CUDA-event timing by the caller). */
void* symgpu_cuda_stream(symgpu_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
uint64_t symgpu_launch_count(const symgpu_ctx* ctx);

/* ---- MPEG-1/2/2.5 Layer III ---------------------------------------------------------------- */

/* Block types, symphonia-bundle-mp3/src/layer3/common.rs:175-182. */
enum { SYMGPU_MP3_LONG = 0, SYMGPU_MP3_START = 1, SYMGPU_MP3_SHORT = 2, SYMGPU_MP3_END = 3 };

/* symgpu_mp3_gc.flags */
enum {
    SYMGPU_MP3_F_MIXED = 1 << 0,          /* BlockType::Short { is_mixed: true }                */
    SYMGPU_MP3_F_SCALEFAC_SCALE = 1 << 1, /* GranuleChannel::scalefac_scale                     */
    SYMGPU_MP3_F_PREFLAG = 1 << 2,        /* GranuleChannel::preflag                            */
    SYMGPU_MP3_F_SFC_LSB = 1 << 3,        /* scalefac_compress & 1 (MPEG-2 intensity scale)     */
    SYMGPU_MP3_F_MID_SIDE = 1 << 4,       /* frame: JointStereo(Layer3{mid_side})  header.rs:161 */
    SYMGPU_MP3_F_INTENSITY = 1 << 5,      /* frame: JointStereo(Layer3{intensity})              */
    SYMGPU_MP3_F_MPEG1 = 1 << 6,          /* frame: header.is_mpeg1()                           */
    SYMGPU_MP3_F_MUTE = 1 << 7            /* unit absent (mono ch1 / MPEG-2 gr1): skip, no PCM  */
};

/* One granule-channel: the fields of `GranuleChannel` (layer3/mod.rs:145-205) that the synthesis
 * stage reads, plus the three frame-header facts it needs.  64 bytes, 4 per frame laid out
 * [granule][channel].  `rzero` is the value returned by read_huffman_samples
 * (requantize.rs:236); the spectrum beyond it must be zero. */
typedef struct symgpu_mp3_gc {
    uint16_t rzero;            /* 0..576                                                        */
    uint8_t global_gain;       /*                                                               */
    uint8_t block_type;        /* SYMGPU_MP3_LONG..END                                          */
    uint8_t flags;             /* SYMGPU_MP3_F_*                                                */
    uint8_t sample_rate_idx;   /* 0..8, order of layer3/common.rs:9-55                          */
    uint8_t subblock_gain[3];  /*                                                               */
    uint8_t scalefacs[39];     /*                                                               */
    uint8_t reserved[16];      /* must be zero                                                  */
} symgpu_mp3_gc;

/* A run = `n_frames` consecutive frames of ONE stream, stored contiguously in the batch starting
 * at frame `first_frame`.  `stream` indexes the persistent per-stream synthesis state (hybrid
 * overlap + polyphase history; what `Layer3.overlap` / `Layer3.synthesis` hold,
 * layer3/mod.rs:254-259). */
typedef struct symgpu_mp3_run {
    uint32_t stream;
    uint32_t first_frame;
    uint32_t n_frames;
    uint8_t granules_per_frame; /* 2 = MPEG-1, 1 = MPEG-2 / 2.5 (header.n_granules()); 0 means 2 */
    uint8_t channels;           /* 1 or 2 (header.n_channels()); 0 means 2                      */
    uint16_t reserved;          /* must be zero                                                  */
} symgpu_mp3_run;

#define SYMGPU_MP3_LINES 576
#define SYMGPU_MP3_FRAME_FLOATS (2 * 2 * 576) /* spectra [gr][ch][576]; pcm [ch][gr*576 + i]  */

/* POW43[x] = f32 powf(x, 4/3) for x in 0..8206 (requantize.rs:23-32): the magnitude the CPU
 * Huffman stage writes for quantised value x (requantize.rs:128, :144).  Host libm, no GPU
 * needed.  Returns the table length (8207); copies min(cap, 8207) floats when `out` != NULL. */
size_t symgpu_mp3_pow43(float* out, size_t cap);

/* Allocates / zeroes device state for `n_streams` MP3 streams (Layer3::new, mod.rs:262-269). */
symgpu_status symgpu_mp3_streams_alloc(symgpu_ctx* ctx, uint32_t n_streams);
/* AudioDecoder::reset for one stream (decoder.rs:152-155): zero overlap + polyphase history. */
symgpu_status symgpu_mp3_stream_reset(symgpu_ctx* ctx, uint32_t stream);

/* Synthesises a batch of `n_frames` frames.
 *   units   [n_frames][2][2]      symgpu_mp3_gc
 *   spectra [n_frames][2][2][576] f32, values as left by read_huffman_samples
 *   runs    [n_runs]  (host)      frames of one stream are consecutive and in decode order; runs
 *                                 must tile [0, n_frames) without overlap and no stream may
 *                                 appear in two runs of the same call
 *   pcm     [n_frames][2][1152]   f32 planar per frame: plane(ch)[gr*576 .. gr*576+576]
 * Host variant: copies in, launches, copies out, and returns after the PCM is in `pcm`.  Batches of 512 frames or more are cut
 * into slices whose H2D copy, kernel and D2H copy overlap.  Smaller batches (one packet per call is the extreme) whose three
 * buffers are pinned, device-mapped host memory (cudaHostAlloc / cudaHostRegister) are handed to the kernel as they are -- one
 * launch, one synchronisation, no staging copy; pageable buffers are staged.  SYMGPU_ZERO_COPY=s forces staging, =2 hands
 * batches of any size to the kernel. */
symgpu_status symgpu_mp3_synth_host(symgpu_ctx* ctx, const symgpu_mp3_gc* units,
                                    const float* spectra, const symgpu_mp3_run* runs,
                                    uint32_t n_runs, uint32_t n_frames, float* pcm);
/* Device variant: `units`, `spectra` and `pcm` are device memory already resident in HBM; `runs`
 * is HOST memory (control plane: the library cuts runs into per-CTA tiles on the host).
 * Asynchronous on the context stream; call symgpu_sync() before reading `pcm`. */
symgpu_status symgpu_mp3_synth_dev(symgpu_ctx* ctx, const symgpu_mp3_gc* units,
                                   const float* spectra, const symgpu_mp3_run* runs,
                                   uint32_t n_runs, uint32_t n_frames, float* pcm);

/* ---- MP3: asynchronous, thread-safe submission (many single-stream decoders sharing one context) ------------------- *
 * The reference creates one decoder per stream (registry.rs:260-269) and calls decode() once per packet
 * (codecs/audio.rs:251-298); a server runs many of them on as many threads.  These three entry points may be called
 * concurrently from any number of threads on ONE context (every other entry point of a context still wants one caller at
 * a time, and must not run concurrently with these).  submit copies one frame into the context's pinned staging batch
 * and returns a ticket; wait returns that frame's PCM.  The first thread that waits for a ticket of the oldest
 * unfinished batch closes the batch and runs it -- one copy in, ONE launch, one copy out -- for every thread that has a
 * frame in it; the others sleep until it is done, while new submissions gather in the next batch.  Frames of a stream
 * are synthesised in submission order (a stream occurs once per batch; batches run in order).  A malformed frame is
 * refused by submit (SYMGPU_ERR_DECODE) and never reaches a batch.  Every ticket must be redeemed exactly once. */
typedef struct symgpu_ticket {
    uint64_t batch;
    uint32_t slot;
    uint32_t reserved;
} symgpu_ticket;
/* units [2][2], spectra [2][2][576] (one frame, as symgpu_mp3_synth_host takes them); granules_per_frame 2 | 1, channels 2 | 1. */
symgpu_status symgpu_mp3_submit(symgpu_ctx* ctx, uint32_t stream, const symgpu_mp3_gc* units, const float* spectra,
                                uint8_t granules_per_frame, uint8_t channels, symgpu_ticket* ticket);
/* Same with the Huffman stage's int16 values sign * x (|x| <= 8206); the POW43 lookup happens at submission. */
symgpu_status symgpu_mp3_submit_quantized(symgpu_ctx* ctx, uint32_t stream, const symgpu_mp3_gc* units, const int16_t* quant,
                                          uint8_t granules_per_frame, uint8_t channels, symgpu_ticket* ticket);
/* pcm [2][1152] of the ticket's frame.  Blocks until the frame's batch has run (running it if nobody else does). */
symgpu_status symgpu_mp3_wait(symgpu_ctx* ctx, symgpu_ticket ticket, float* pcm);
/* Launch batches run so far through submit / wait and the frames they held (frames / batches = achieved batching). */
void symgpu_mp3_async_stats(const symgpu_ctx* ctx, uint64_t* batches, uint64_t* frames);

/* ---- AAC-LC filterbank --------------------------------------------------------------------- */

/* Window sequences, symphonia-codec-aac/src/aac/common.rs:17-20. */
enum { SYMGPU_AAC_ONLY_LONG = 0, SYMGPU_AAC_LONG_START = 1, SYMGPU_AAC_EIGHT_SHORT = 2, SYMGPU_AAC_LONG_STOP = 3 };

/* One channel of one frame: the arguments of Dsp::synth (aac/dsp.rs:57-65) that are not sample
 * data, plus a reference to the channel's TNS filters.  16 bytes, 2 per frame. */
typedef struct symgpu_aac_unit {
    uint8_t window_sequence;   /* IcsInfo::window_sequence                                      */
    uint8_t window_shape;      /* 0 sine, 1 KBD (IcsInfo::window_shape)                         */
    uint8_t prev_window_shape; /* IcsInfo::prev_window_shape (ics/mod.rs:119, :172-177)         */
    uint8_t n_tns;             /* number of TNS filters with order > 0 to run on this channel   */
    uint32_t tns_first;        /* index of the first of them in the `tns` array                 */
    uint32_t reserved[2];      /* must be zero                                                  */
} symgpu_aac_unit;

/* One TNS all-pole filter, already resolved to a line range by the parser
 * (Tns::synth, aac/ics/tns.rs:149-199: start/end = w*128 + bands[min(.., tns_max_bands)]).
 * direction 0 filters upward from `start`, 1 downward from `end - 1`. */
typedef struct symgpu_aac_tns {
    uint16_t start, end;       /* [start, end) within the channel's 1024 lines                  */
    uint8_t order;             /* 1..20 (AAC-LC: <= 12)                                         */
    uint8_t direction;
    uint16_t reserved;
    float lpc[20];             /* TnsCoeffs::coef                                               */
} symgpu_aac_tns;

typedef struct symgpu_aac_run {
    uint32_t stream;           /* per-stream state slot: Ics.delay of both channels             */
    uint32_t first_frame;
    uint32_t n_frames;
    uint8_t channels;          /* 1 or 2; 0 means 2                                             */
    uint8_t reserved[3];
} symgpu_aac_run;

symgpu_status symgpu_aac_streams_alloc(symgpu_ctx* ctx, uint32_t n_streams);
symgpu_status symgpu_aac_stream_reset(symgpu_ctx* ctx, uint32_t stream); /* Ics::reset, ics/mod.rs:229-232 */

/* Synthesises `n_frames` AAC-LC frames (Pulse::synth, <= 4 lines, stays with the parser):
 *   units  [n_frames][2], tns [n_tns], coeffs [n_frames][2][1024] -> pcm [n_frames][2][1024]
 * (plane(ch) of frame f at pcm[f][ch]).  Same host/dev split as the MP3 entry points; `runs` is
 * host memory in both.  Runs must not overlap but may leave frames out (a stream that lost packets keeps an
 * unused tail in its slice): such frames are not decoded; their PCM is zero in the host variant and left
 * untouched in the device variant.  The same holds for the Vorbis entry points and their packets. */
symgpu_status symgpu_aac_synth_host(symgpu_ctx* ctx, const symgpu_aac_unit* units, const symgpu_aac_tns* tns,
                                    uint32_t n_tns, const float* coeffs, const symgpu_aac_run* runs,
                                    uint32_t n_runs, uint32_t n_frames, float* pcm);
symgpu_status symgpu_aac_synth_dev(symgpu_ctx* ctx, const symgpu_aac_unit* units, const symgpu_aac_tns* tns,
                                   uint32_t n_tns, const float* coeffs, const symgpu_aac_run* runs,
                                   uint32_t n_runs, uint32_t n_frames, float* pcm);

/* ---- Vorbis synthesis ---------------------------------------------------------------------- */

/* What floor-1 curve synthesis needs from Floor1Setup (codec-vorbis/src/floor.rs:546-560):
 * the X list, the precomputed neighbours (find_neighbors, :748-773) and the sort order. */
typedef struct symgpu_vorbis_floor1 {
    uint8_t multiplier;        /* floor1_multiplier, 1..4                                       */
    uint8_t n_posts;           /* floor1_x_list.len(), 2..65                                    */
    uint16_t x_list[65];
    uint8_t low[65], high[65]; /* floor1_x_list_neighbors                                       */
    uint8_t sort_order[65];    /* floor1_x_list_sort_order                                      */
    uint8_t reserved[5];
} symgpu_vorbis_floor1;        /* 332 bytes */

/* Identification-header facts of a stream (lib.rs:404-406).  Up to two channels with at most one
 * coupling step (magnitude = channel 0, angle = channel 1) are supported in this version. */
typedef struct symgpu_vorbis_stream {
    uint8_t bs0_exp, bs1_exp;  /* blocksize exponents, 6..13                                    */
    uint8_t channels;          /* 1 or 2                                                        */
    uint8_t coupled;           /* 1: inverse coupling of (ch0 magnitude, ch1 angle)             */
} symgpu_vorbis_stream;

/* One audio packet after entropy decode (lib.rs:248 | :250).  16 bytes. */
typedef struct symgpu_vorbis_unit {
    uint8_t block_flag;        /* mode.block_flag: 1 = long block                               */
    uint8_t prev_block_flag;   /* dsp.prev_block_flag.unwrap_or(block_flag)  (lib.rs:298)       */
    uint8_t do_not_decode[2];  /* per channel, after non-zero vector propagate (lib.rs:215-225) */
    uint16_t floor[2];         /* per channel: index of its floor-1 setup in `floors`, or 0xffff
                                  when the floor is unused (zero curve, floor.rs is_unused)     */
    uint8_t reserved[8];
} symgpu_vorbis_unit;

typedef struct symgpu_vorbis_run {
    uint32_t stream;           /* index into `streams` and of the per-stream overlap state      */
    uint32_t first_packet;
    uint32_t n_packets;
    uint32_t reserved;
} symgpu_vorbis_run;

/* Registers stream configurations (and zeroes their overlap state) / floor setups with a context. */
symgpu_status symgpu_vorbis_streams_set(symgpu_ctx* ctx, const symgpu_vorbis_stream* streams, uint32_t n_streams);
symgpu_status symgpu_vorbis_floors_set(symgpu_ctx* ctx, const symgpu_vorbis_floor1* floors, uint32_t n_floors);
/* The validation symgpu_vorbis_floors_set applies, without a context (host only): SYMGPU_OK or SYMGPU_ERR_ARG.  The Vorbis
 * front-end runs it when a stream is opened, so that an unusable setup is refused per stream (SYMGPU_ERR_UNSUPPORTED). */
symgpu_status symgpu_vorbis_floors_check(const symgpu_vorbis_floor1* floors, uint32_t n_floors);
/* The same, also writing each setup's dependency levels (72 bytes per setup: level[65], the largest level, 6 zero bytes). */
symgpu_status symgpu_vorbis_floors_levels(const symgpu_vorbis_floor1* floors, uint32_t n_floors, uint8_t* levels);
symgpu_status symgpu_vorbis_stream_reset(symgpu_ctx* ctx, uint32_t stream); /* dsp.rs:26-32, :128-131 */

/* Synthesises `n_packets` packets.  Every per-packet array uses fixed slots of `slot` floats per
 * channel, slot >= the largest blocksize_1 / 2 in the batch:
 *   units [n_packets], floor_y [n_packets][2][65] (Floor1.floor_y), residue [n_packets][2][slot]
 *   -> pcm [n_packets][2][slot], of which the first (prev_n + n) / 4 samples are the packet's output.
 * Floor curves are rendered on the device (floor1 synthesis step 1 + 2), then inverse coupling,
 * floor * residue, IMDCT, window, overlap-add. */
symgpu_status symgpu_vorbis_synth_host(symgpu_ctx* ctx, const symgpu_vorbis_unit* units, const uint16_t* floor_y,
                                       const float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                       uint32_t n_packets, uint32_t slot, float* pcm);
symgpu_status symgpu_vorbis_synth_dev(symgpu_ctx* ctx, const symgpu_vorbis_unit* units, const uint16_t* floor_y,
                                      const float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                      uint32_t n_packets, uint32_t slot, float* pcm);

/* ---- Vorbis with more than two channels / several coupling steps ------------------------------------------------------ *
 * The reference maps up to 8 channels (codec-vorbis/src/lib.rs:771-788) and applies every coupling step of the packet's
 * mapping in order (lib.rs:252-278).  Channels interact ONLY there: afterwards floor * residue, IMDCT and overlap-add are
 * per channel.  So the multichannel entry points run the inverse coupling of all steps as an element-wise pass over the
 * residue vectors (in place, on the device) and then synthesise the channel planes two at a time with the stereo kernel
 * (coupling off).  All per-packet arrays carry `channels` planes: floor_y [n_packets][channels][65], residue / pcm
 * [n_packets][channels][slot]; `channels` = the largest channel count among the streams of the call (planes a stream does
 * not have are left alone).  Stream indices of runs refer to symgpu_vorbis_mc_streams_set; a context holds either
 * classic or multichannel Vorbis streams, not both.  The device variant decouples `residue` in place. */
#define SYMGPU_VORBIS_MAX_CHANNELS 8
#define SYMGPU_VORBIS_MAX_COUPLINGS 16
typedef struct symgpu_vorbis_stream_mc {
    uint8_t bs0_exp, bs1_exp;  /* identification header                                          */
    uint8_t channels;          /* 1..8                                                           */
    uint8_t n_couplings;       /* mapping.couplings.len(), applied in this order                 */
    uint8_t magnitude_ch[SYMGPU_VORBIS_MAX_COUPLINGS];
    uint8_t angle_ch[SYMGPU_VORBIS_MAX_COUPLINGS];
} symgpu_vorbis_stream_mc;
typedef struct symgpu_vorbis_unit_mc {      /* 32 bytes */
    uint8_t block_flag, prev_block_flag;
    uint8_t do_not_decode[SYMGPU_VORBIS_MAX_CHANNELS];
    uint16_t floor[SYMGPU_VORBIS_MAX_CHANNELS]; /* floor-1 setup per channel, 0xffff = unused */
    uint8_t reserved[6];
} symgpu_vorbis_unit_mc;
symgpu_status symgpu_vorbis_mc_streams_set(symgpu_ctx* ctx, const symgpu_vorbis_stream_mc* streams, uint32_t n_streams);
symgpu_status symgpu_vorbis_mc_stream_reset(symgpu_ctx* ctx, uint32_t stream);
symgpu_status symgpu_vorbis_mc_synth_host(symgpu_ctx* ctx, const symgpu_vorbis_unit_mc* units, const uint16_t* floor_y,
                                          const float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                          uint32_t n_packets, uint32_t channels, uint32_t slot, float* pcm);
symgpu_status symgpu_vorbis_mc_synth_dev(symgpu_ctx* ctx, const symgpu_vorbis_unit_mc* units, const uint16_t* floor_y,
                                         float* residue, const symgpu_vorbis_run* runs, uint32_t n_runs,
                                         uint32_t n_packets, uint32_t channels, uint32_t slot, float* pcm);

/* ===================================================================================================
 * Output stage (SURVEY §8f N3): planar f32 PCM -> interleaved samples of the caller's format, with
 * the decoder's gapless trim, on the device -- so that the D2H copy carries i16 instead of f32.
 * (FLAC's integer samples have their own conversions, FromSample<i32>: see symgpu_flac_decode_*.)
 * Replaces, for the batch:
 *   AudioBuffer::trim(start, end)            symphonia-core/src/audio/buf.rs:404-433
 *     (called by the decoders at symphonia-bundle-mp3/src/decoder.rs:130-132 and
 *      symphonia-codec-vorbis/src/lib.rs:318-326)
 *   Audio::copy_to_slice_interleaved::<Sout> symphonia-core/src/audio/buf.rs:469-476
 *   FromSample<f32> for u8/i16/i24/i32/f32    symphonia-core/src/audio/conv.rs:592-607
 *   clamp_f32 / clamp_i24                    symphonia-core/src/util.rs:230-237, :258-266
 * Integer results are bit-exact: clamp to [-1, 1] (NaN passes through), scale by a power of two,
 * truncate toward zero with Rust's saturating `as` cast (NaN -> 0).
 * ================================================================================================= */
typedef enum symgpu_sample_format {
    SYMGPU_FMT_F32 = 0, /* f32, interleaved only                                   4 bytes / sample */
    SYMGPU_FMT_S16 = 1, /* (s.clamped() * 32768.0) as i16                          2 bytes / sample */
    SYMGPU_FMT_S24 = 2, /* i24::from((s.clamped() * 8388608.0) as i32).inner()     4 bytes / sample */
    SYMGPU_FMT_S32 = 3, /* (s.clamped() as f64 * 2147483648.0) as i32              4 bytes / sample */
    SYMGPU_FMT_U8 = 4   /* ((s.clamped() + 1.0) * 128.0) as u8                     1 byte  / sample */
} symgpu_sample_format;

/* One decoded packet of one stream.  32 bytes. */
typedef struct symgpu_pcm_span {
    uint64_t src;          /* float index, in `pcm`, of plane 0 of this packet                      */
    uint32_t plane_stride; /* floats from plane c to plane c + 1                                    */
    uint32_t frames;       /* decoded frames: 1152 (MP3), 1024 (AAC), (prev_n + n) / 4 (Vorbis)     */
    uint32_t trim_start;   /* Packet::trim_start                                                    */
    uint32_t trim_end;     /* Packet::trim_end                                                      */
    uint64_t dst_frame;    /* index of the packet's first surviving frame in `out`                  */
} symgpu_pcm_span;

/* Frames of a span that survive the trim: truncate(frames.saturating_sub(end)), then shift(start). */
uint32_t symgpu_pcm_span_kept(const symgpu_pcm_span* span);
size_t symgpu_sample_bytes(int format); /* 0 for an unknown format */

/* out[(dst_frame + i) * channels + c] = convert(pcm[src + c * plane_stride + trim_start + i]) for
 * every kept frame i of every span; 1 <= channels <= 8.  `spans` may be NULL: then the n_spans packets
 * are uniform, packet p at src = p * channels * plane_stride with `frames` frames, untrimmed, written
 * back to back (dst_frame = p * frames).
 * Device variant: pcm, spans and out are device memory; asynchronous on the context stream.
 * Host variant: host memory (pcm_floats / out_bytes give the extents to copy). */
symgpu_status symgpu_pcm_pack_dev(symgpu_ctx* ctx, const float* pcm, const symgpu_pcm_span* spans, uint32_t n_spans,
                                  uint32_t channels, uint32_t plane_stride, uint32_t frames, int format, void* out);
symgpu_status symgpu_pcm_pack_host(symgpu_ctx* ctx, const float* pcm, size_t pcm_floats, const symgpu_pcm_span* spans,
                                   uint32_t n_spans, uint32_t channels, uint32_t plane_stride, uint32_t frames,
                                   int format, void* out, size_t out_bytes);
/* The same with a channel map: output channel c reads plane plane_of_channel[c] (< channels; host memory in both variants), i.e.
 * out[(dst_frame + i) * channels + c] = convert(pcm[src + plane_of_channel[c] * plane_stride + trim_start + i]).  With the identity
 * map the output equals symgpu_pcm_pack_*. */
symgpu_status symgpu_pcm_pack_mapped_dev(symgpu_ctx* ctx, const float* pcm, const symgpu_pcm_span* spans, uint32_t n_spans,
                                         uint32_t channels, uint32_t plane_stride, uint32_t frames, const uint8_t* plane_of_channel,
                                         int format, void* out);
symgpu_status symgpu_pcm_pack_mapped_host(symgpu_ctx* ctx, const float* pcm, size_t pcm_floats, const symgpu_pcm_span* spans,
                                          uint32_t n_spans, uint32_t channels, uint32_t plane_stride, uint32_t frames,
                                          const uint8_t* plane_of_channel, int format, void* out, size_t out_bytes);

/* symgpu_mp3_synth_host with the output stage in the pipeline: the stereo PCM of frame f is written to
 * out as interleaved samples [f * 1152 .. f * 1152 + 1152) of `format` (no trim); only the packed
 * samples cross PCIe on the way back.  Runs must be 2-granule, 2-channel. */
symgpu_status symgpu_mp3_synth_host_packed(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const float* spectra,
                                           const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                                           int format, void* out);

/* Descriptor checks of the host entry points, callable on their own (no device needed): what the reference's
 * parsers guarantee about the units they hand to synthesis (3-bit subblock_gain, block types 0..3, rzero <= 576,
 * sample-rate index 0..8, equal block types on a joint-stereo pair -- stereo.rs:503-505; AAC window sequence 0..3,
 * window shape 0..1, TNS filters inside the 1024 lines with order <= 20 -- tns.rs:17-20).  SYMGPU_ERR_DECODE for a
 * malformed unit; the host entry points run them before anything is sent to the device (the device entry points
 * cannot: their descriptors are already in HBM). */
symgpu_status symgpu_mp3_units_check(const symgpu_mp3_gc* units, const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames);
symgpu_status symgpu_aac_units_check(const symgpu_aac_unit* units, const symgpu_aac_tns* tns, uint32_t n_tns, uint32_t n_frames);

/* ===================================================================================================
 * MPEG Layer I / II (SURVEY 8f N4): the polyphase synthesis bank alone, i.e. `synthesis::synthesis`
 * (symphonia-bundle-mp3/src/synthesis.rs:158-344) as the Layer I / II decoders call it after dequantising
 * their sub-band samples (layer1/mod.rs:184-194 with 12 time slots per frame, layer2/mod.rs:374-384 with 36).
 *   subbands [n_frames][2][32][n_slots]   = the decoders' samples[ch][n_slots * sb + s]
 *   pcm      [n_frames][2][1152]          plane(ch)[0 .. 32 * n_slots) written (384 or 1152 samples)
 * Streams use the Layer III state slots (symgpu_mp3_streams_alloc / symgpu_mp3_stream_reset): every layer
 * owns the same `synthesis: [SynthesisState; 2]` (layer1/mod.rs:63, layer2/mod.rs:220, layer3/mod.rs:257).
 * ================================================================================================= */
typedef struct symgpu_mpa12_run {
    uint32_t stream;
    uint32_t first_frame;
    uint32_t n_frames;
    uint8_t channels;     /* 1 or 2 */
    uint8_t reserved[3];
} symgpu_mpa12_run;
symgpu_status symgpu_mpa12_synth_host(symgpu_ctx* ctx, const float* subbands, const symgpu_mpa12_run* runs, uint32_t n_runs,
                                      uint32_t n_frames, uint32_t n_slots, float* pcm);
symgpu_status symgpu_mpa12_synth_dev(symgpu_ctx* ctx, const float* subbands, const symgpu_mpa12_run* runs, uint32_t n_runs,
                                     uint32_t n_frames, uint32_t n_slots, float* pcm);

/* ===================================================================================================
 * FLAC (SURVEY 8f N4): what FlacDecoder::decode_inner does after the Rice residuals are decoded --
 * integer prediction, wasted-bits shift, channel decorrelation, scaling to 32 bits.  Bit-exact (integers).
 * EXPERIMENTAL in this revision: see tests/test_flac_parity_gpu.py for what has and has not been verified.
 *   fixed_predict / lpc_predict         symphonia-bundle-flac/src/decoder.rs:663-752
 *   samples_shl (dropped_bps)           decoder.rs:384-394
 *   decorrelate_left_side / mid_side / right_side   decoder.rs:32-82
 *   output scaling `sample << (32 - bps)`            decoder.rs:232-241
 * `samples` is one int32 buffer; a sub-frame owns `n` consecutive samples at `offset`: on entry its warm-up
 * samples followed by the residuals (what decode_verbatim + decode_residual leave in the plane, decoder.rs:437-
 * 443, :459-481), or its constant in samples[offset], or the verbatim samples; on return the channel's PCM.
 * ================================================================================================= */
typedef enum symgpu_flac_subframe_type { SYMGPU_FLAC_CONSTANT = 0, SYMGPU_FLAC_VERBATIM = 1, SYMGPU_FLAC_FIXED = 2, SYMGPU_FLAC_LPC = 3 } symgpu_flac_subframe_type;
typedef enum symgpu_flac_assignment { SYMGPU_FLAC_INDEPENDENT = 0, SYMGPU_FLAC_LEFT_SIDE = 1, SYMGPU_FLAC_MID_SIDE = 2, SYMGPU_FLAC_RIGHT_SIDE = 3 } symgpu_flac_assignment;
typedef struct symgpu_flac_subframe {   /* 144 bytes */
    uint64_t offset;     /* first sample of the sub-frame in `samples`                                   */
    uint32_t n;          /* block size                                                                  */
    uint8_t type;        /* symgpu_flac_subframe_type                                                   */
    uint8_t order;       /* FIXED: 0..4, LPC: 1..32; must not exceed n (decoder.rs:429, :456)           */
    uint8_t shift;       /* LPC: qlp_coeff_shift, 0..15 (negative shifts are unsupported, decoder.rs:504) */
    uint8_t wasted;      /* dropped_bps: samples are shifted left by it after prediction (decoder.rs:382) */
    int32_t coeffs[32];  /* LPC: coeffs[j] multiplies sample i-1-j (the reference keeps them reversed)    */
} symgpu_flac_subframe;
typedef struct symgpu_flac_frame {      /* 16 bytes */
    uint32_t first_subframe; /* index of channel 0's sub-frame; channel c is first_subframe + c          */
    uint8_t channels;        /* 1..8; LEFT_SIDE / MID_SIDE / RIGHT_SIDE need 2                            */
    uint8_t assignment;      /* symgpu_flac_assignment                                                   */
    uint8_t bits_per_sample; /* 4..32 of the frame; the output is scaled by 32 - bits_per_sample          */
    uint8_t reserved;
    uint32_t reserved2[2];
} symgpu_flac_frame;
/* In place on `samples` (n_samples int32).  Host variant: host memory; device variant: frames, subframes and
 * samples in device memory, asynchronous on the context stream (descriptors are then not validated). */
symgpu_status symgpu_flac_restore_host(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                       const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                       size_t n_samples);
symgpu_status symgpu_flac_restore_dev(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                      const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                      size_t n_samples);
/* Restoration as symgpu_flac_restore_*, followed by FromSample<i32> into `format` (symphonia-core/src/audio/conv.rs:514-532),
 * interleaved: what a caller of the reference's FLAC decoder gets from AudioBuffer<i32> + copy_to_slice_interleaved::<S>.
 *   S32  s                      S24  s >> 8 (in a 4-byte container, as the f32 output stage stores it)
 *   S16  (s >> 16) as i16       U8   ((s as u32).wrapping_add(0x8000_0000) >> 24) as u8
 *   F32  (s as f64 / 2^31) as f32
 * Every rule is exact.  Frame f writes its n * channels samples from out[dst[f]] on (dst counts SAMPLES of `format`, so files with
 * different channel counts share one call): out[dst[f] + i * channels + c] = sample i of channel c.  The restored int32 planes are
 * not copied back.
 * Host variant: host memory; the descriptor checks of symgpu_flac_restore_host, plus a known format, one block size for all
 * sub-frames of a frame (SYMGPU_ERR_DECODE) and dst[f] + n * channels <= out_bytes / symgpu_sample_bytes(format)
 * (SYMGPU_ERR_LIMIT); a refused call sends nothing to the device and leaves `out` untouched.  Otherwise `out` is rewritten in
 * whole: samples no frame writes are zero.  `samples` is not modified.
 * Device variant: frames, subframes, samples, dst and out in device memory, asynchronous on the context stream.  It runs the
 * predictors in place on `samples`; n_samples bounds its reads and out_samples its writes (a frame that would leave either is not
 * written), and the descriptors are not otherwise validated. */
symgpu_status symgpu_flac_decode_host(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                      const symgpu_flac_subframe* subframes, uint32_t n_subframes, const int32_t* samples,
                                      size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_bytes);
symgpu_status symgpu_flac_decode_dev(symgpu_ctx* ctx, const symgpu_flac_frame* frames, uint32_t n_frames,
                                     const symgpu_flac_subframe* subframes, uint32_t n_subframes, int32_t* samples,
                                     size_t n_samples, const uint64_t* dst, int format, void* out, size_t out_samples);

/* The same synthesis fed with the QUANTISED spectra, i.e. what the Huffman stage decodes before the
 * reference turns it into f32 (read_huffman_samples: buf[i] = sign * POW43[x],
 * symphonia-bundle-mp3/src/layer3/requantize.rs:23-32, :128, :144):
 *   quant [n_frames][2][2][576] int16, |q| <= 8206, exactly 0 from rzero on;
 * the POW43 lookup runs on the device, so half the bytes cross PCIe on the way in.
 * format < 0: planar f32 PCM [n_frames][2][1152] as symgpu_mp3_synth_host; otherwise interleaved samples
 * of `format` as symgpu_mp3_synth_host_packed. */
symgpu_status symgpu_mp3_synth_host_quantized(symgpu_ctx* ctx, const symgpu_mp3_gc* units, const int16_t* quant,
                                              const symgpu_mp3_run* runs, uint32_t n_runs, uint32_t n_frames,
                                              int format, void* out);

/* ===================================================================================================
 * Packetisers (SURVEY 8f N2): file bytes -> packet tables, on the host, no context and no device needed.
 * C entry points over include/symgpu/packetizer.hpp (which C++ callers can use directly).  Nothing is copied:
 * a packet is a reference into `data`, so the file can go to the device in one piece.
 *   MPEG audio  MpaReader::try_new / next_packet   symphonia-bundle-mp3/src/demuxer.rs:414-487, :160-218
 *   ADTS        AdtsReader::next_packet            symphonia-codec-aac/src/adts.rs:278-309
 *   Ogg         PageReader + LogicalStream         symphonia-format-ogg/src/page.rs:166-271, logical.rs:104-205
 *   Vorbis      the Ogg mapper's header work       symphonia-format-ogg/src/mappings/vorbis.rs:45-405
 * All index functions follow the two-call pattern: with cap == 0 they only count (*n_out = what a full run
 * would write); otherwise they write at most cap records and still report the full count.
 * ================================================================================================= */
typedef struct symgpu_mpa_track {       /* 48 bytes: what try_new learns from the first frame                     */
    uint32_t first_header;   /* header word of the first frame (codec parameters)                                 */
    uint32_t sample_rate;
    uint8_t version;         /* 0 MPEG-1, 1 MPEG-2, 2 MPEG-2.5                                                     */
    uint8_t layer;           /* 1..3                                                                              */
    uint8_t channels;
    uint8_t tag;             /* 0 none, 1 Xing, 2 Info, 3 VBRI                                                     */
    uint8_t has_delay;       /* delay / padding come from a LAME extension                                        */
    uint8_t has_num_frames;  /* num_frames from a tag, or the reference's estimate when `seekable`                */
    uint8_t reserved[2];
    uint32_t delay, padding; /* samples                                                                           */
    uint32_t reserved2[2];
    uint64_t num_frames;     /* samples of audio, delay and padding already removed                               */
    uint64_t first_packet_pos;
} symgpu_mpa_track;
typedef struct symgpu_mpa_packet {      /* 48 bytes: one frame                                                     */
    uint64_t offset;         /* of the header word in `data`                                                      */
    uint32_t size;           /* whole frame                                                                       */
    uint32_t header;         /* the header word                                                                   */
    int64_t pts;             /* samples; the first packet starts at -delay                                        */
    uint32_t dur;            /* samples the frame decodes to                                                      */
    uint32_t trim_start;     /* leading samples to drop                                                           */
    uint64_t trim_end;       /* trailing samples to drop; may exceed dur (packet.rs:334-338 does not cap it)      */
    int32_t main_data_begin; /* Layer III bit-reservoir back pointer, -1 for Layers I / II                        */
    uint32_t reserved;
} symgpu_mpa_packet;
/* SYMGPU_ERR_DECODE: no frame in the data (track untouched). */
symgpu_status symgpu_mpa_index(const uint8_t* data, size_t n, int seekable, symgpu_mpa_track* track,
                               symgpu_mpa_packet* packets, size_t cap, size_t* n_out);

typedef struct symgpu_adts_packet {     /* 32 bytes: one raw data block (no ADTS header)                          */
    uint64_t offset;
    uint32_t size;
    uint32_t sample_rate;
    int64_t pts;             /* 1024 samples per packet                                                           */
    uint8_t channels;        /* 0: configured in-band                                                             */
    uint8_t profile;         /* MPEG-4 audio object type, 2 = LC                                                  */
    uint8_t reserved[6];
} symgpu_adts_packet;
/* Indexes up to the first thing the reference's reader would return an error for.  *stop: SYMGPU_OK = clean end of
 * data, SYMGPU_ERR_LIMIT = the last frame's payload is cut short, SYMGPU_ERR_DECODE / _UNSUPPORTED = a bad header
 * (adts.rs:155-191).  The function itself fails only on null arguments. */
symgpu_status symgpu_adts_index(const uint8_t* data, size_t n, symgpu_adts_packet* packets, size_t cap, size_t* n_out,
                                symgpu_status* stop);

typedef struct symgpu_piece {           /* 16 bytes: a byte range of `data`                                        */
    uint64_t offset;
    uint32_t len;
    uint32_t reserved;
} symgpu_piece;
typedef struct symgpu_ogg_packet {      /* 40 bytes: a packet = pieces[first_piece .. first_piece + n_pieces)      */
    uint32_t serial;         /* logical stream                                                                    */
    uint32_t page_sequence;  /* of the page the packet ends on                                                    */
    uint64_t page_absgp;     /* that page's granule position                                                      */
    uint64_t len;
    uint32_t first_piece;
    uint32_t n_pieces;
    uint8_t last_on_page;    /* the page's granule position is THIS packet's end                                  */
    uint8_t reserved[7];
} symgpu_ogg_packet;
/* Every page that verifies, every logical stream announced by a first-page flag; packets grouped by serial (ascending),
 * in stream order within a serial. */
symgpu_status symgpu_ogg_index(const uint8_t* data, size_t n, symgpu_ogg_packet* packets, size_t cap_packets,
                               size_t* n_packets, symgpu_piece* pieces, size_t cap_pieces, size_t* n_pieces);

typedef struct symgpu_vorbis_ident {    /* 8 bytes                                                                 */
    uint32_t sample_rate;
    uint8_t channels;
    uint8_t bs0_exp, bs1_exp; /* block sizes 2^6 .. 2^13, short <= long                                            */
    uint8_t reserved;
} symgpu_vorbis_ident;
/* The 30-byte identification packet.  SYMGPU_ERR_DECODE / _UNSUPPORTED as read_ident_header (mappings/vorbis.rs:293-360),
 * SYMGPU_ERR_ARG if n < 30. */
symgpu_status symgpu_vorbis_ident_parse(const uint8_t* packet, size_t n, symgpu_vorbis_ident* ident);
/* Walks a setup packet to its mode list: *n_modes (1..64) and bit i of *long_block_mask = mode i uses the long block. */
symgpu_status symgpu_vorbis_setup_modes(const uint8_t* packet, size_t n, const symgpu_vorbis_ident* ident, uint32_t* n_modes,
                                        uint64_t* long_block_mask);
/* The decoder's reading of a setup packet (symphonia-codec-vorbis/src/lib.rs:490-770, floor.rs:455-560): counts, modes, and for
 * every floor of type 1 the record symgpu_vorbis_floors_set takes (X list, neighbours, sort order, multiplier); floors of type
 * 0 are reported in floor_type and left zeroed.  Codebook CONTENTS are only syntax-checked.  floors: room for 64 records. */
typedef struct symgpu_vorbis_setup_info {   /* 160 bytes */
    uint32_t n_codebooks, n_floors, n_residues, n_mappings, n_modes;
    uint32_t reserved;
    uint64_t long_block_mask;       /* bit i: mode i uses the long block                  */
    uint8_t mode_mapping[64];       /* mapping of mode i                                  */
    uint8_t floor_type[64];         /* 0 or 1                                             */
} symgpu_vorbis_setup_info;
symgpu_status symgpu_vorbis_setup_parse(const uint8_t* packet, size_t n, const symgpu_vorbis_ident* ident, symgpu_vorbis_setup_info* info,
                                        symgpu_vorbis_floor1* floors);
/* Copies the packets' pieces back to back into `out` (cap bytes; the packets' `len` sum suffices) and writes table[i] = where packet i
 * now lies: a contiguous copy of a logical stream for the per-stream front-end calls.  SYMGPU_ERR_LIMIT if cap is too small. */
symgpu_status symgpu_ogg_gather(const uint8_t* data, size_t n, const symgpu_ogg_packet* packets, size_t n_packets, const symgpu_piece* pieces,
                                size_t n_pieces, uint8_t* out, size_t cap, symgpu_piece* table, size_t* used);
/* End trims of the stream packets of ONE logical stream against the granule positions of the pages they end on
 * (symphonia-format-ogg/src/logical.rs:164-302): page_sequence / page_absgp as in symgpu_ogg_packet, dur / discard from the
 * codec mapping (symgpu_vorbis_packet_durations), all in stream order. */
symgpu_status symgpu_ogg_page_end_trims(const uint32_t* page_sequence, const uint64_t* page_absgp, const uint32_t* dur,
                                        const uint32_t* discard, size_t n, uint32_t* trim_end);
/* Durations of a run of audio packets (VorbisPacketParser::parse_next_packet_dur, :62-106): heads[i] = the first
 * byte(s) of packet i packed little-endian (two bytes always suffice: 1 type bit + at most 6 mode bits), head_len[i] =
 * how many bytes of the packet exist (0, 1 or >= 2).  dur / discard in samples.  *prev_exp carries the previous block's
 * exponent across calls: 0 on entry = no previous block (stream start, or after a reset); updated on return. */
symgpu_status symgpu_vorbis_packet_durations(const symgpu_vorbis_ident* ident, uint32_t n_modes, uint64_t long_block_mask,
                                             const uint16_t* heads, const uint8_t* head_len, size_t n_packets, uint8_t* prev_exp,
                                             uint32_t* dur, uint32_t* discard);

/* ===================================================================================================
 * MP3 entropy front-end (SURVEY 8f N1): MPEG frame bytes -> the batch format of the synthesis entry points --
 * 4 x symgpu_mp3_gc + the QUANTISED spectrum (int16, as symgpu_mp3_synth_host_quantized takes it).  CPU only,
 * one object per stream (it owns the bit reservoir); no context, no device.
 *   MpaDecoder::decode_inner (header, size and spec checks)   symphonia-bundle-mp3/src/decoder.rs:84-131
 *   Layer3::decode up to the synthesis seam                    layer3/mod.rs:373-418
 *   BitResevoir::fill / consume                                layer3/mod.rs:42-108
 *   read_side_info, read_scale_factors_mpeg1 / _mpeg2          layer3/bitstream.rs:57-427
 *   read_main_data, read_huffman_samples (without POW43)       layer3/mod.rs:272-370, requantize.rs:47-237
 * ================================================================================================= */
typedef struct symgpu_mp3_fe symgpu_mp3_fe;
typedef struct symgpu_mp3_frame_info {  /* 16 bytes */
    uint32_t sample_rate;
    uint8_t channels;          /* 1 or 2                                                                    */
    uint8_t granules;          /* 2 (MPEG-1) or 1: symgpu_mp3_run.granules_per_frame                         */
    uint8_t sample_rate_idx;
    uint8_t version;           /* 0 MPEG-1, 1 MPEG-2, 2 MPEG-2.5                                             */
    uint32_t underflow_bytes;  /* main_data_begin pointed this many bytes before what the reservoir holds   */
    uint32_t main_data_bytes;  /* bytes of main data this frame consumed from the reservoir                  */
} symgpu_mp3_frame_info;
symgpu_status symgpu_mp3_fe_create(symgpu_mp3_fe** out);
void symgpu_mp3_fe_destroy(symgpu_mp3_fe* fe);
void symgpu_mp3_fe_reset(symgpu_mp3_fe* fe);   /* AudioDecoder::reset: empty reservoir, no signal spec yet */
/* One packet = one whole frame, header word first.
 *   units [2][2]       as the synthesis takes them; absent units (mono channel 1, MPEG-2 granule 1) get F_MUTE
 *   quant [2][2][576]  sign * x, |x| <= 8206; 0 from rzero on and in absent units
 * SYMGPU_ERR_DECODE: the reference would return an error for this packet and produce no audio (the reservoir is
 * cleared where the reference clears it); units / quant are then unspecified. */
symgpu_status symgpu_mp3_fe_decode(symgpu_mp3_fe* fe, const uint8_t* frame, size_t n, symgpu_mp3_gc* units, int16_t* quant,
                                   symgpu_mp3_frame_info* info);
/* A stream's packets in one call: packet i = data[packets[i].offset .. + size).  Good frames are written densely
 * (units / quant of the k-th good frame at index k) and frame_of[k] = its packet index; *n_good = how many.
 * `info` describes the first good frame.  Fails only on bad arguments. */
symgpu_status symgpu_mp3_fe_decode_packets(symgpu_mp3_fe* fe, const uint8_t* data, size_t n, const symgpu_mpa_packet* packets,
                                           size_t n_packets, symgpu_mp3_gc* units, int16_t* quant, uint32_t* frame_of,
                                           size_t* n_good, symgpu_mp3_frame_info* info);

/* ---- the same front-end as a PLAN + parallel jobs (what the device path executes) --------------------------------
 * A granule-channel's first bit follows from the side information alone (the part2_3_length fields before it), and
 * so does every step of the bit reservoir.  symgpu_mp3_entropy_plan therefore walks a stream's packets once WITHOUT
 * touching the Huffman data and emits
 *   md    the main data of the good frames, concatenated: a frame's reservoir is one contiguous window of it
 *   jobs  4 per good frame (64 bytes each, layout: symphonia_b200/csrc/mp3_entropy.h GcJob), independent of each other
 * which symgpu_mp3_entropy_run_cpu (host threads of the caller's choosing; the test model) or the device kernel turn into
 * units + quantised spectra, one job per thread.  A job that fails at decode time ("huffman decode overrun",
 * layer3/mod.rs:345-358) makes the reference drop the frame AND empty the reservoir, which changes the plan of the frames
 * behind it: pass the failed packets back in `bad` and plan again (symgpu_mp3_entropy_decode_cpu does this loop). */
typedef struct symgpu_mp3_gc_job { uint64_t opaque[8]; } symgpu_mp3_gc_job;
/* bad: n_packets flags or NULL: 1 = known to fail while its main data is read (reservoir emptied, as the reference does);
 * 2 = to be left out although its main data is consumed normally (a frame the synthesis stage refuses).  md_cap >= the packets' total size is always enough.
 * frame_of[k] = packet index of good frame k; jobs / frame_of may be NULL to count only.  *md_len, *n_good: results. */
symgpu_status symgpu_mp3_entropy_plan(const uint8_t* data, size_t n, const symgpu_mpa_packet* packets, size_t n_packets,
                                      const uint8_t* bad, uint8_t* md, size_t md_cap, size_t* md_len, symgpu_mp3_gc_job* jobs,
                                      uint32_t* frame_of, size_t* n_good, symgpu_mp3_frame_info* info);
/* Runs jobs [0, n_jobs): unit / quant slot of a job = its out_index (frame * 4 + granule * 2 + channel, frames counted from
 * the first job's frame).  failed[f] = 1 when a job of good frame f failed.  Pure function of its inputs: callers may
 * split the job range over threads. */
symgpu_status symgpu_mp3_entropy_run_cpu(const uint8_t* md, size_t md_len, const symgpu_mp3_gc_job* jobs, size_t n_jobs,
                                         symgpu_mp3_gc* units, int16_t* quant, uint8_t* failed);
/* The same over `n_threads` host threads (0 = hardware concurrency): jobs are cut into contiguous ranges of whole frames. */
symgpu_status symgpu_mp3_entropy_run_cpu_mt(const uint8_t* md, size_t md_len, const symgpu_mp3_gc_job* jobs, size_t n_jobs,
                                            symgpu_mp3_gc* units, int16_t* quant, uint8_t* failed, uint32_t n_threads);
/* plan -> run -> re-plan until no job fails; results as symgpu_mp3_fe_decode_packets (a fresh stream: no state carried). */
symgpu_status symgpu_mp3_entropy_decode_cpu(const uint8_t* data, size_t n, const symgpu_mpa_packet* packets, size_t n_packets,
                                            symgpu_mp3_gc* units, int16_t* quant, uint32_t* frame_of, size_t* n_good,
                                            symgpu_mp3_frame_info* info, uint32_t* n_rounds);

/* ---- the device path of the front-end.  EXPERIMENTAL in this revision: compiled for sm_100a, not yet run on a GPU
 * (tests/test_mp3_entropy_gpu.py is opt-in, SYMGPU_TEST_ENTROPY=1). ------------------------------------------------ */
/* One thread per job, the same decode functions as symgpu_mp3_entropy_run_cpu.  All pointers are device memory;
 * d_failed[n_jobs / 4] must be zeroed by the caller; asynchronous on the context stream. */
symgpu_status symgpu_mp3_entropy_dev(symgpu_ctx* ctx, const uint8_t* d_md, size_t md_len, const symgpu_mp3_gc_job* d_jobs, size_t n_jobs,
                                     symgpu_mp3_gc* d_units, int16_t* d_quant, uint32_t* d_failed);
typedef struct symgpu_mp3_file {        /* one stream's bytes and packet table (symgpu_mpa_index), all host memory          */
    const uint8_t* data;
    size_t n;
    const symgpu_mpa_packet* packets;
    size_t n_packets;
    uint32_t stream;                    /* synthesis state slot (symgpu_mp3_streams_alloc)                                  */
    uint32_t reserved;
} symgpu_mp3_file;
/* File bytes -> planar f32 PCM with nothing but the side-information pass on the CPU: plan, upload main data + jobs,
 * entropy kernel, POW43 lookup, synthesis kernel, PCM back.  pcm [sum of good frames][2][1152] (pcm_frames_cap >= total
 * packets is always enough); good_per_file[f] frames of file f, in order; frame_of = their packet indices, concatenated.
 * Frames the reference refuses are left out as symgpu_mp3_fe_decode_packets leaves them out; additionally a joint-stereo
 * frame whose channels disagree on the window sequence (refused by the reference's stereo stage) is left out whole. */
symgpu_status symgpu_mp3_decode_files_host(symgpu_ctx* ctx, const symgpu_mp3_file* files, uint32_t n_files, float* pcm, size_t pcm_frames_cap,
                                           uint32_t* good_per_file, uint32_t* frame_of, uint32_t* n_rounds);

/* ===================================================================================================
 * MPEG Layer I / II sample decoders (SURVEY 8f N1 for the Layer I / II path): a packet becomes the sub-band samples
 * symgpu_mpa12_synth_* take.  CPU only, stateless apart from the stream's signal specification.
 *   Layer1::decode up to the synthesis call   symphonia-bundle-mp3/src/layer1/mod.rs:19-176
 *   Layer2::decode up to the synthesis call   layer2/mod.rs:45-369; scale factors layer12.rs:9-75
 * ================================================================================================= */
/* One packet.  subbands [2][32][n_slots] f32 (n_slots = 12 Layer I, 36 Layer II: samples[ch][n_slots * sb + s]), fully
 * written (zeros where nothing is allocated and in the absent channel of a mono frame).  `layer` = the stream's layer
 * (1 or 2): a packet of another layer is refused as the reference's decoder refuses it (decoder.rs:113-128). */
symgpu_status symgpu_mpa12_fe_decode(const uint8_t* frame, size_t n, int layer, float* subbands, symgpu_mp3_frame_info* info);
/* A stream's packets: good frames densely in `subbands` ([n_good][2][32][n_slots]), frame_of[k] = packet index.  The signal
 * specification is fixed by the first packet (decoder.rs:96-108). */
symgpu_status symgpu_mpa12_fe_decode_packets(const uint8_t* data, size_t n, const symgpu_mpa_packet* packets, size_t n_packets, int layer,
                                             float* subbands, uint32_t* frame_of, size_t* n_good, symgpu_mp3_frame_info* info);
/* The decoders' constants (for tests): 64 scale factors, then C and D of the 17 quantisation classes in the order of
 * ISO 11172-3 Table 3-B.4 (3, 5, 7, 9, 15, ... 65535 levels).  Returns 98 = the number of floats. */
size_t symgpu_mpa12_constants(float* out, size_t cap);

/* ===================================================================================================
 * FLAC front-end (SURVEY 8f N1 for the FLAC row): a packet (one frame) becomes the descriptors and the residual /
 * warm-up / verbatim samples symgpu_flac_restore_* take.  CPU only, stateless.
 *   sync_frame, read_frame_header (CRC-8, UTF-8 coded sequence number)   symphonia-bundle-flac/src/frame.rs:66-233, :281-333
 *   FlacDecoder::decode_inner up to the restoration                       decoder.rs:139-228
 *   read_subframe, decode_constant / _verbatim / _fixed_linear / _linear  decoder.rs:340-520
 *   decode_residual, decode_rice_partition, rice_signed_to_i32            decoder.rs:522-640
 * ================================================================================================= */
typedef struct symgpu_flac_frame_info {  /* 24 bytes */
    uint64_t sequence;        /* frame number (fixed block size streams) or first sample number (variable)              */
    uint32_t block_size;
    uint32_t sample_rate;     /* 0: not in the frame header, take it from the stream information                        */
    uint8_t by_sample;        /* sequence counts samples                                                                */
    uint8_t reserved[7];
} symgpu_flac_frame_info;
/* A stream's packets: packet i = data[packets[i].offset .. + len).  For every packet the reference decodes, in order:
 *   frames[k], infos[k], frame_of[k] = i; its sub-frames appended to `subs` (frames[k].first_subframe), each sub-frame's n
 *   samples appended to `samples` (subs[].offset) -- residuals behind the warm-up samples, a constant in the first slot, or
 *   the verbatim samples, exactly the input of symgpu_flac_restore_*.
 * stream_bps / stream_channels / max_block: from the stream information block (0 = unknown; a frame that relies on a
 * missing value, has more channels than the stream or a larger block is refused as the reference refuses it).
 * SYMGPU_ERR_LIMIT if subs_cap / samples_cap are too small (a refused packet's partial output is discarded). */
symgpu_status symgpu_flac_fe_decode_packets(const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                            uint32_t stream_bps, uint32_t stream_channels, uint32_t max_block,
                                            symgpu_flac_frame* frames, symgpu_flac_frame_info* infos, uint32_t* frame_of,
                                            symgpu_flac_subframe* subs, size_t subs_cap, int32_t* samples, size_t samples_cap,
                                            size_t* n_good, size_t* n_subs, size_t* n_samples);

/* FLAC native container (include/symgpu/packetizer.hpp FlacIndexer): "fLaC", metadata blocks, frames split where the
 * CRC-16 vouches for the boundary.  Same packets as the reference's parser (symphonia-bundle-flac/src/parser.rs) on
 * well-formed files; a plain checksum-validated splitter on damaged ones (DESIGN 5b). */
typedef struct symgpu_flac_stream_info {   /* 56 bytes: STREAMINFO, symphonia-common/src/xiph/audio/flac/mod.rs:78-186 */
    uint64_t n_samples;        /* 0 = unknown                                                                        */
    uint64_t first_frame_pos;
    uint32_t sample_rate;
    uint32_t frame_min, frame_max;
    uint16_t block_min, block_max;
    uint8_t channels, bits_per_sample, has_md5, reserved;
    uint8_t md5[16];
    uint8_t reserved2[4];
} symgpu_flac_stream_info;
typedef struct symgpu_flac_packet {        /* 24 bytes */
    uint64_t offset;
    uint64_t ts;               /* first sample of the frame (parser.rs:566-584)                                       */
    uint32_t size;
    uint32_t dur;              /* samples                                                                            */
} symgpu_flac_packet;
/* SYMGPU_ERR_UNSUPPORTED: no "fLaC" marker; SYMGPU_ERR_DECODE: bad or missing STREAMINFO / cut metadata.  Two-call pattern. */
symgpu_status symgpu_flac_index(const uint8_t* data, size_t n, symgpu_flac_stream_info* info, symgpu_flac_packet* packets, size_t cap,
                                size_t* n_out);

/* ===================================================================================================
 * Vorbis entropy front-end (SURVEY 8f N1): audio packets -> the batch format of symgpu_vorbis_synth_* (unit, floor-1 Y
 * values, residue vectors BEFORE inverse coupling).  CPU only; one object per stream (codebooks, setup, previous block).
 *   VorbisCodebook::read, synthesize_codewords, VQ unpack   symphonia-codec-vorbis/src/codebook.rs:16-400
 *   Floor1::read_channel                                     floor.rs:655-722
 *   Residue::read_residue (types 0, 1, 2)                    residue.rs:142-543
 *   VorbisDecoder::decode_inner up to inverse coupling       lib.rs:146-250
 * Two ways to open a stream, both refusing floor type 0 and setups symgpu_vorbis_floors_check refuses (SYMGPU_ERR_UNSUPPORTED):
 *   symgpu_vorbis_fe_create     what symgpu_vorbis_synth_* takes: 1 or 2 channels, every mapping uncoupled or coupled by the one
 *                               step (magnitude 0, angle 1), the same number of steps in every mode's mapping.  Used with the
 *                               two-plane entry points (config, decode, decode_packets, decode_packets_jobs).
 *   symgpu_vorbis_fe_create_mc  what symgpu_vorbis_mc_synth_* takes: 1 to 8 channels (more: SYMGPU_ERR_UNSUPPORTED, the reference has
 *                               no channel map for them; 0: SYMGPU_ERR_DECODE), up to SYMGPU_VORBIS_MAX_COUPLINGS steps per mapping,
 *                               every mode's mapping with the same coupling list.  Used with the *_mc entry points, which write
 *                               `planes` channel planes (stream channels <= planes <= 8: streams of different channel counts can
 *                               share one batch; planes beyond the stream's are zero, not decoded, without a floor).
 * A front-end from create_mc takes the two-plane entry points only if create would have accepted the stream (else SYMGPU_ERR_ARG).
 * ================================================================================================= */
typedef struct symgpu_vorbis_fe symgpu_vorbis_fe;
/* ident: the 30-byte identification packet; setup: the setup packet (together: the stream's extra data). */
symgpu_status symgpu_vorbis_fe_create(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out);
void symgpu_vorbis_fe_destroy(symgpu_vorbis_fe* fe);
void symgpu_vorbis_fe_reset(symgpu_vorbis_fe* fe);   /* AudioDecoder::reset: no previous block */
/* The stream record and the floor records to register with the context (floors: room for 64; *n_floors written). */
symgpu_status symgpu_vorbis_fe_config(const symgpu_vorbis_fe* fe, symgpu_vorbis_stream* stream, symgpu_vorbis_floor1* floors, uint32_t* n_floors);
/* One audio packet.  floor_y [2][65], residue [2][slot] (slot >= blocksize_1 / 2; fully written, zeros where nothing was coded);
 * unit->floor[] index the records of symgpu_vorbis_fe_config (+ floor_base).  SYMGPU_ERR_DECODE where the reference errors
 * (not an audio packet, bad mode number); a packet that merely ends early is decoded as far as it goes, as in the reference. */
symgpu_status symgpu_vorbis_fe_decode(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base,
                                      symgpu_vorbis_unit* unit, uint16_t* floor_y, float* residue);
/* The same as independent jobs on n_threads host threads (every thread builds its own front-end from the headers): outputs stay at their
 * packet's index (units[i], floor_y[130 i], residue[2 slot i]; a refused packet's unit is zeroed), accepted[0 .. *n_good) lists the
 * decoded packets in order and the previous block flags are chained over those -- always identical to the serial form (DESIGN 10.9). */
symgpu_status symgpu_vorbis_fe_decode_packets_jobs(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, const uint8_t* data, size_t n,
                                                   const symgpu_piece* packets, size_t n_packets, uint32_t slot, uint32_t floor_base,
                                                   symgpu_vorbis_unit* units, uint16_t* floor_y, float* residue, uint32_t* accepted, size_t* n_good,
                                                   uint32_t n_threads);
/* A stream's audio packets in one call (packet i = data[packets[i].offset .. + len)): units[k], floor_y[130k..], residue[2*slot*k..],
 * packet_of[k] = i for every packet the front-end accepts, in order; refused packets are left out. */
symgpu_status symgpu_vorbis_fe_decode_packets(symgpu_vorbis_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                              uint32_t slot, uint32_t floor_base, symgpu_vorbis_unit* units, uint16_t* floor_y, float* residue,
                                              uint32_t* packet_of, size_t* n_good);
/* The multichannel forms: records of symgpu_vorbis_mc_streams_set (couplings in mapping order) / _floors_set; per packet a
 * symgpu_vorbis_unit_mc, floor_y [planes][65], residue [planes][slot] (packet k of a batch at 65 * planes * k / planes * slot * k). */
symgpu_status symgpu_vorbis_fe_create_mc(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, symgpu_vorbis_fe** out);
symgpu_status symgpu_vorbis_fe_config_mc(const symgpu_vorbis_fe* fe, symgpu_vorbis_stream_mc* stream, symgpu_vorbis_floor1* floors, uint32_t* n_floors);
symgpu_status symgpu_vorbis_fe_decode_mc(symgpu_vorbis_fe* fe, const uint8_t* packet, size_t n, uint32_t slot, uint32_t floor_base, uint32_t planes,
                                         symgpu_vorbis_unit_mc* unit, uint16_t* floor_y, float* residue);
symgpu_status symgpu_vorbis_fe_decode_packets_mc(symgpu_vorbis_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                                 uint32_t slot, uint32_t floor_base, uint32_t planes, symgpu_vorbis_unit_mc* units, uint16_t* floor_y,
                                                 float* residue, uint32_t* packet_of, size_t* n_good);
symgpu_status symgpu_vorbis_fe_decode_packets_jobs_mc(const uint8_t* ident, size_t n_ident, const uint8_t* setup, size_t n_setup, const uint8_t* data,
                                                      size_t n, const symgpu_piece* packets, size_t n_packets, uint32_t slot, uint32_t floor_base,
                                                      uint32_t planes, symgpu_vorbis_unit_mc* units, uint16_t* floor_y, float* residue, uint32_t* accepted,
                                                      size_t* n_good, uint32_t n_threads);
/* The reference's channel order (map_vorbis_channel, lib.rs:771-788; Vorbis I 4.3.9): Vorbis channel i of a `channels`-channel
 * stream is output plane plane_of_channel[i].  symgpu_vorbis_*_synth_* write planes in Vorbis order; symgpu_pcm_pack_mapped_* with
 * the inverse permutation produces the reference's order.  channels 1..8, else SYMGPU_ERR_ARG. */
symgpu_status symgpu_vorbis_channel_map(uint32_t channels, uint8_t* plane_of_channel);

/* ===================================================================================================
 * AAC-LC entropy front-end (SURVEY 8f N1): one raw_data_block per packet (an ADTS frame's payload, or an MP4 sample) ->
 * the batch format of symgpu_aac_synth_* (two channel units, resolved TNS filters, 2 x 1024 dequantised lines after
 * joint stereo and pulse restoration).  CPU only; one object per stream (window history, element layout, noise generator).
 *   AacDecoder::try_new (no extra data), set_pair, decode_ga   symphonia-codec-aac/src/aac/mod.rs:52-229
 *   ChannelPair::decode_ga_sce / decode_ga_cpe                  aac/cpe.rs:51-161
 *   IcsInfo::decode, Ics::decode (sections, scale factors, spectrum, PNS)   aac/ics/mod.rs:120-447
 *   Pulse::read / synth, Tns::read, the line ranges of Tns::synth           aac/ics/pulse.rs:35-105, aac/ics/tns.rs:35-199
 * 1 or 2 channels (mod.rs:101-108); a packet whose elements do not cover exactly the configured channels is
 * SYMGPU_ERR_UNSUPPORTED (the reference renders the channels it found; the batch format carries all of a frame).
 * ================================================================================================= */
typedef struct symgpu_aac_fe symgpu_aac_fe;
symgpu_status symgpu_aac_fe_create(uint32_t sample_rate, uint32_t channels, symgpu_aac_fe** out);
/* MPEG-4 AudioSpecificConfig as the reference reads it (symphonia-common/src/mpeg/audio/mod.rs:230-439): the extra data of AAC in MP4 /
 * Matroska.  24 bytes. */
typedef struct symgpu_aac_asc {
    uint32_t sample_rate;
    uint32_t ext_sample_rate;  /* of an explicit SBR / PS extension (has_ext)                                              */
    uint16_t samples;          /* 1024 or 960 for the general-audio object types, else 0                                   */
    uint8_t object_type;       /* MPEG-4 audio object type index after an SBR / PS prefix: 2 = AAC-LC                      */
    uint8_t channels;          /* channel count of the configuration index (7 -> 8); 0 = defined in-band                   */
    uint8_t sbr_present, ps_present, has_ext, ext_channels;
    uint8_t reserved[8];
} symgpu_aac_asc;
/* SYMGPU_ERR_DECODE (invalid index, zero rate, data ends) / SYMGPU_ERR_UNSUPPORTED (object types and options the reference refuses). */
symgpu_status symgpu_aac_asc_parse(const uint8_t* buf, size_t n, symgpu_aac_asc* out);
/* AacDecoder::try_new with extra data (aac/mod.rs:59-108): parses it, then requires AAC-LC, no SBR, at most two channels, 1024-sample
 * frames ("aac too complex" otherwise).  *asc (optional) receives what was parsed. */
symgpu_status symgpu_aac_fe_create_asc(const uint8_t* extra, size_t n, symgpu_aac_fe** out, symgpu_aac_asc* asc);
void symgpu_aac_fe_destroy(symgpu_aac_fe* fe);
void symgpu_aac_fe_reset(symgpu_aac_fe* fe);   /* AudioDecoder::reset: window history forgotten (pair with symgpu_aac_stream_reset) */
/* units [2], tns: room for 16 records (*n_tns written; units[].tns_first = tns_base + position), coeffs [2][1024] (channel 1
 * zero for a mono stream).  SYMGPU_ERR_DECODE / _UNSUPPORTED where the reference's decode returns that error; the stream
 * state is then left as the reference leaves it (changed up to the point of failure). */
symgpu_status symgpu_aac_fe_decode(symgpu_aac_fe* fe, const uint8_t* packet, size_t n, uint32_t tns_base, symgpu_aac_unit* units,
                                   symgpu_aac_tns* tns, uint32_t* n_tns, float* coeffs);
/* A stream's packets in one call: packet i = data[packets[i].offset .. + len).  For every packet the front-end accepts, in order:
 * units[2k..], coeffs[2048k..], frame_of[k] = i, its TNS records appended to `tns` (tns_base + position); refused packets are left
 * out, as a caller of the reference drops them.  SYMGPU_ERR_LIMIT if tns_cap is too small (16 per packet always suffice). */
symgpu_status symgpu_aac_fe_decode_packets(symgpu_aac_fe* fe, const uint8_t* data, size_t n, const symgpu_piece* packets, size_t n_packets,
                                           uint32_t tns_base, symgpu_aac_unit* units, symgpu_aac_tns* tns, size_t tns_cap, float* coeffs,
                                           uint32_t* frame_of, size_t* n_good, size_t* n_tns);
/* The blocks of ONE stream as independent jobs on n_threads host threads (the decomposition a device front-end would use, DESIGN 10.9):
 * every block decoded from a fresh state, noise generators jumped ahead over the prefix sums of each block's draws, blocks that drew
 * noise decoded again from the right state, window history chained afterwards.  units [2 n_packets], coeffs [2048 n_packets], tns
 * compacted as in symgpu_aac_fe_decode_packets.  SYMGPU_OK: identical to the serial front-end.  SYMGPU_ERR_RESET: the stream needs the
 * serial path (a block is refused, the element layout changes, or a pulse reads a scale left behind by an earlier block). */
symgpu_status symgpu_aac_fe_decode_packets_jobs(uint32_t sample_rate, uint32_t channels, const uint8_t* data, size_t n, const symgpu_piece* packets,
                                                size_t n_packets, uint32_t tns_base, symgpu_aac_unit* units, symgpu_aac_tns* tns, size_t tns_cap,
                                                float* coeffs, size_t* n_tns, uint32_t n_threads);
/* The dequantisation tables the front-end uses (for tests): x^(4/3) [8192], 2^((i-156)/4) [256], 0.5^((i-155)/4) [256]. */
void symgpu_aac_fe_tables(float* pow43, float* normal_scf, float* intensity_scf);

#ifdef __cplusplus
}
#endif
#endif /* SYMGPU_H */
