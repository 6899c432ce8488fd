/* sed_b200.h -- C ABI of the B200-native sound-event-detection inference hot path.
 *
 * Plain pointers and sizes only; every pointer is a DEVICE pointer unless stated otherwise, `stream`
 * is a cudaStream_t passed as void*.  Every entry returns 0 on success or one of SED_ERR_*; the
 * message for the calling thread's last failure is returned by sed_last_error_string().  Nothing here
 * allocates or frees memory the caller can see, and all work is asynchronous on `stream`.
 *
 * The reference (yazdayy/sound-event-detection) has no FFI: its hot path is the Python nn.Module
 * forward() of pytorch/models.py calling ATen ops.  Each entry below names the reference code it
 * replaces (file:line under /root/reference).  INTEGRATION.md shows the ctypes binding.
 */
#ifndef SED_B200_H_
#define SED_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define SED_OK 0
#define SED_ERR_BAD_SHAPE 1
#define SED_ERR_UNSUPPORTED 2
#define SED_ERR_CUDA 3
#define SED_ERR_NULL 4
#define SED_ERR_DRIVER 5

#define SED_DTYPE_F16 0
#define SED_DTYPE_BF16 1

#define SED_CONV_STORE 0    /* conv -> BN -> ReLU                        (ConvBlock first conv)        */
#define SED_CONV_POOL 1     /* conv -> BN -> ReLU -> avg_pool2d(2,2)     (ConvBlock second conv)       */
#define SED_CONV_FREQMEAN 2 /* conv -> BN -> ReLU -> mean over W (W==8)  (conv_block4 + models.py:668) */

/* ABI version of this header (bumped on any signature change). */
int sed_abi_version(void);

/* Message describing the last non-zero return on the calling thread (host pointer, never NULL). */
const char* sed_last_error_string(void);

/* Fused front-end: reflect-pad, frame, window, real DFT, power, mel projection, clamped 10*log10,
 * optional per-mel affine (eval-mode bn0).
 * Replaces STFT.forward pytorch/stft.py:223-247, Spectrogram.forward :651-670,
 * LogmelFilterBank.forward + power_to_db :698-734 and bn0 pytorch/models.py:642-644; with wave_dtype = 1 also
 * int16_to_float32 utils/utilities.py:78-79 (x = q / 32767); with clip_stride < L also the window slicing +
 * pad_truncate_sequence of the streaming loop pytorch/predict.py:302-305.
 *   wave: clip b = wave + b*clip_stride, L samples, f32 (wave_dtype 0) or int16 PCM (wave_dtype 1); samples at
 *   index >= total_len (counted from `wave`) read as zero.  Dense batch: clip_stride = L, total_len = B*L.
 *   clip_offset: optional device table [B] of clip starts in samples (overrides b*clip_stride) -- the windows of
 *   many padded clips as one batch, pytorch/main_strong.py:786-805.
 *   window [n_fft] f32 (row 0 of the loaded conv_real kernel); twiddle [n_fft][2] f32 = exp(-2 pi i k / n_fft);
 *   banded mel matrix: for mel bin m the non-zero weights melW[mel_lo[m] .. mel_lo[m]+mel_len[m]) are stored at
 *   mel_val[mel_off[m] ..]; db_offset = 10*log10(max(amin, ref)); bn_scale/bn_shift [n_mels] or NULL;
 *   out [B, T, n_mels] f32 with T = L / hop + 1.  n_fft in {256, 512, 1024}. */
int sed_frontend_logmel(const void* wave, int wave_dtype, int B, int L, long clip_stride, const long* clip_offset,
                        long total_len, int n_fft, int hop, const float* window, const float* twiddle, const int* mel_lo, const int* mel_len,
                        const int* mel_off, const float* mel_val, int n_mels, float amin, float db_offset, int is_log,
                        const float* bn_scale, const float* bn_shift, float* out, void* stream);

/* Power spectrogram only.  Replaces Spectrogram.forward pytorch/stft.py:651-670 (power == 2).
 *   out [B, T, n_fft/2+1] f32 (the reference's [B,1,T,F] layout). */
int sed_spectrogram_f32(const float* wave, int B, int L, int n_fft, int hop, const float* window,
                        const float* twiddle, float* out, void* stream);

/* Mel projection + power_to_db on existing spectrogram rows.
 * Replaces LogmelFilterBank.forward pytorch/stft.py:698-734 (top_db == None).
 *   spec [rows, F] f32 -> out [rows, n_mels] f32. */
int sed_logmel_rows_f32(const float* spec, long rows, int F, const int* mel_lo, const int* mel_len,
                        const int* mel_off, const float* mel_val, int n_mels, float amin, float db_offset,
                        int is_log, float* out, void* stream);

/* conv_block1.conv1 (Cin = 1) + bn1 + ReLU.  Replaces pytorch/models.py:128 for the first block.
 *   x [NB, H, 64] f32 (log-mel after bn0); w9 [64][9] f32; scale/shift [64] folded BatchNorm;
 *   out [NB, H, 64, 64] NHWC 16-bit (dtype). */
int sed_conv_first_f32(const float* x, int NB, int H, int W, const float* w9, const float* scale,
                       const float* shift, void* out, int dtype, void* stream);

/* 3x3 stride-1 pad-1 convolution (no bias) + folded BatchNorm + ReLU [+ 2x2 avg-pool | + mean over W]
 * on the tcgen05 tensor cores.  Replaces ConvBlock.forward pytorch/models.py:125-141 (one conv each
 * call) and torch.mean(x, dim=3) models.py:668.
 *   x [NB, H, W, cin] NHWC 16-bit; wpacked [cout][9][cin] 16-bit (tap = 3*kh + kw);
 *   scale/shift [cout] f32; out NHWC 16-bit: [NB,H,W,cout] | [NB,H/2,W/2,cout] | [NB,H,cout];
 *   out_f32: optional float32 copy [NB,H,cout] of the FREQMEAN result (NULL otherwise).
 *   out_stride_n / out_stride_h (FREQMEAN only; 0, 0 = default H, 1): output row of (image n, row h) is
 *   n*out_stride_n + h*out_stride_h -- (1, batch) writes the features time-major for the GRU.
 *   Supported (cin,cout,mode): (64,64,POOL) (64,128,STORE) (128,128,POOL) (128,256,STORE)
 *   (256,256,POOL) (256,512,STORE) (512,512,FREQMEAN).
 *   variant 0 = single-CTA haloed-patch operand reuse, 1 = one TMA box per tap, 2 = CTA pairs (cta_group::2). */
int sed_conv3x3_bn_relu(const void* x, int NB, int H, int W, int cin, const void* wpacked, const float* scale,
                        const float* shift, int cout, int mode, void* out, void* out_f32, long out_stride_n,
                        long out_stride_h, int dtype, int variant, void* stream);

/* conv_block1 in one kernel: conv1 (1 -> 64) + bn1 + ReLU computed on the fly as the tensor-core operand of
 * conv2 (64 -> 64) + bn2 + ReLU + 2x2 avg-pool.  Replaces ConvBlock.forward pytorch/models.py:125-141 for
 * conv_block1 (models.py:663); the [NB, H, W, 64] intermediate never reaches HBM.
 *   producer 0: conv1 on the CUDA cores (packed f32x2 FMAs) -- measured slower (1.07 ms per 148 clips) than
 *   sed_conv_first_f32 + sed_conv3x3_bn_relu (0.28 + 0.53 ms); producer 1: conv1 as a split-fp16 tensor-core GEMM
 *   whose accumulators are drained from TMEM into conv2's shared-memory operand.
 *   x [NB, H, W] f32 (log-mel after bn0, W % 16 == 0); w1_scaled [64][9] f32 = conv1 weights x folded bn1 scale;
 *   shift1 [64] folded bn1 shift; w2packed [64][9][64] 16-bit; scale2/shift2 [64]; out [NB, H/2, W/2, 64] 16-bit. */
int sed_conv_block1(const float* x, int NB, int H, int W, const float* w1_scaled, const float* shift1,
                    const void* w2packed, const float* scale2, const float* shift2, void* out, int producer, int dtype,
                    void* stream);

/* out[M, N] = a[M, K] * w[N, K]^T + bias (optional ReLU) on the tensor cores; K in {256, 512},
 * N % 128 == 0.  Replaces the nn.Linear calls inside nn.GRU (input projection, models.py:670) and
 * MultiHead (w_qs/w_ks/w_vs/fc, models.py:863-865, 876).
 *   a16 [M,K], w16 [N,K] 16-bit; bias [N] f32 or NULL; out [M,N] f32; out16 [M,N] 16-bit or NULL.
 *   out_layout 0: row-major.  1: 128-row transposed blocks (M % 128 == 0, out16 NULL): the float4 holding columns
 *   4c..4c+3 of row r is float4 number ((r/128) * N/4 + c) * 128 + r%128 -- the layout sed_bigru streams. */
int sed_linear(const void* a16, long M, int K, const void* w16, const float* bias, int N, int relu, float* out,
               void* out16, int out_layout, int dtype, void* stream);

/* Bytes of device scratch sed_bigru needs for a batch of B clips (16-bit hidden-state exchange buffer). */
long sed_bigru_workspace_bytes(int B);

/* Bidirectional GRU recurrence, hidden 256, gate order r,z,n, h0 = 0.
 * Replaces nn.GRU.forward pytorch/models.py:670 given the input projections.
 *   gi = x W_ih^T + b_ih (f32, columns [dir][gate][256]) for rows ordered time-major over the batch padded to
 *   Bp = 128*ceil(B/128) clips (row r = t*Bp + clip), stored as 128-row transposed blocks (sed_linear out_layout 1,
 *   M = T*Bp, N = 1536): rows of padding clips may hold anything;
 *   whh_packed [2*768, 256] 16-bit, row (dir*768 + 96*q + 32*g + jj) = W_hh[dir][g*256 + 32*q + jj];
 *   bhh [2][768] f32; out = [forward | backward] f32 for the same padded time-major rows (r = t*Bp + clip,
 *   512 columns), in the same 128-row transposed-block layout (T*Bp*512 floats; feed it to sed_attpool_blocks);
 *   workspace: sed_bigru_workspace_bytes(B) bytes (kept for ABI stability; the hidden state is exchanged through
 *   distributed shared memory). */
int sed_bigru(const float* gi, const void* whh_packed, const float* bhh, int B, int T, float* out, void* workspace,
              int dtype, void* stream);

/* sed_attpool for an input in 128-clip transposed blocks (the output layout of sed_bigru, or of sed_linear
 * out_layout 1 over time-major rows r = t*Bp + clip, Bp = 128*ceil(B/128), 512 columns).  Same outputs as sed_attpool.
 *   scratch: sed_attpool_blocks_scratch_bytes(B, T) bytes of device memory, contents irrelevant.
 *   stage 0: everything for clips [clip_begin, clip_begin + n_clips) (pass 0, B for the whole batch);
 *   stage 1: only the projections of ALL clips into `scratch`; stage 2: only the per-clip pooling / output pass of clips
 *   [clip_begin, clip_begin + n_clips) from a `scratch` filled by stage 1 -- lets a caller overlap the device->host copy of
 *   one range with the pooling of the next.  Output tensors are always indexed by the absolute clip. */
long sed_attpool_blocks_scratch_bytes(int B, int T);
int sed_attpool_blocks(const float* x_blocks, int B, int T, const float* w_att, const float* b_att, const float* w_cla,
                       const float* b_cla, int ratio, int frames_out, void* scratch, float* clip, float* frame,
                       float* cla_t, float* norm_att_t, int stage, int clip_begin, int n_clips, void* stream);

/* Linear(512 -> classes) + sigmoid per frame, x`ratio` interpolation, clipwise mean (use_max = 0) or max (1)
 * over frames: the head of Cnn_9layers_FrameAvg / FrameMax / Gru_FrameAvg / Transformer_FrameAvg
 * (pytorch/models.py:276-288, 361-373, 547-556, 963-972).
 *   x [B, T, 512] f32; w [classes, 512]; b [classes]; classes <= 32; clip [B, classes]; frame [B, T*ratio, classes]. */
int sed_fcpool(const float* x, int B, int T, const float* w, const float* b, int classes, int ratio, int use_max,
               float* clip, float* frame, void* stream);

/* Overlap-add of per-window framewise outputs followed by the reference's block-wise averaging.
 * Replaces merge + avg_merge utils/utilities.py:405-446 as driven by pytorch/predict.py:323-349 (bug-compatible:
 * the first and last overlap_interval frames are never divided, inner blocks use the reference's divisor rule).
 *   frames [n_recordings, n_windows, frames_per_window, classes] f32; window k starts at frame k*overlap_interval;
 *   merged [n_recordings, (n_windows-1)*overlap_interval + frames_per_window, classes] f32 (recordings independent:
 *   the per-file loops of pytorch/predict.py:264 and pytorch/main_strong.py:768 as one launch). */
int sed_window_merge_avg(const float* frames, int n_windows, int frames_per_window, int classes, int overlap_interval,
                         int sample_duration, int n_recordings, float* merged, void* stream);

/* Frame-wise probabilities -> sound events per (clip, class): double-threshold hysteresis, smoothing, salt removal.
 * Replaces activity_detection utils/vad.py:11-45 (+ helpers :108-199) as called per clip and class by
 * frame_prediction_to_event_prediction utils/utilities.py:82-153 / pytorch/predict.py:57-121 (quirks kept:
 * asymmetric +1 on gap boundaries, low-threshold extension, smooth(1) then smooth(n_smooth), fin-bgn <= n_salt dropped).
 *   frames [n_clips, n_frames, classes] f32; high/low [classes] f64 (low may be NULL); n_smooth/n_salt [classes] i32;
 *   events [n_clips, classes, max_events, 2] i32 = (bgn, fin) in frames; counts [n_clips, classes] i32 = number of
 *   events found (may exceed max_events; only the first max_events are stored). */
int sed_events(const float* frames, int n_clips, int n_frames, int classes, const double* high, const double* low,
               const int* n_smooth, const int* n_salt, int max_events, int* events, int* counts, void* stream);

/* ---- Live streaming: audio that is still arriving, many streams per batch ----------------------------------------
 * The rolling window of pytorch/predict.py:297-349 run incrementally: each stream (slot) owns a mirrored audio ring,
 * a merge accumulator ring and per-class event state, all in caller-allocated device memory; the caller keeps the
 * counters and runs, per push, sed_live_ingest -> the model on the ready windows (sed_frontend_logmel reads them in
 * place through its clip_offset table) -> sed_live_merge -> sed_live_events.  sed_b200.LiveStreamer is the driver.
 *
 * Table of sed_live_merge / sed_live_events: [n_entries, SED_LIVE_TABLE_COLS] i32, one row per stream with work:
 *   slot, k0 (windows merged before), m (windows in this push, rows row0 .. row0+m-1 of the model output), row0,
 *   lo (frames returned before), n_final (frames final after this push), out_row (row of frame lo in `out`),
 *   ev_off / ev_cap (events of class c go to events[ev_off + c*ev_cap ..], at most ev_cap), closing (0 / 1). */
#define SED_LIVE_TABLE_COLS 10
#define SED_LIVE_EVENT_STATE_INTS 19 /* ints of event state per (slot, class) */

/* Write chunks into their slots' rings.  Replaces the growing `audio_full` slices of pytorch/predict.py:297-305.
 *   src: packed chunks (dtype 0 = f32, 1 = int16 PCM); table [n_entries, 4] i64 = (slot, offset in src or -1 for
 *   zeros, length <= max_len, absolute position of the first sample in the stream); arena [n_slots, 2*ring_samples]
 *   of src's type: sample p of a slot is stored at p mod ring_samples and at p mod ring_samples + ring_samples. */
int sed_live_ingest(const void* src, int dtype, const long* table, int n_entries, long max_len, long ring_samples,
                    void* arena, void* stream);

/* Incremental merge + avg_merge of the windows of one push.  Replaces merge / avg_merge utils/utilities.py:405-446
 * as driven window by window by pytorch/predict.py:323-349, bit for bit: the first window covering a frame sets it,
 * later windows add in ascending order, final frames are divided by avg_merge's divisor.
 *   window_frames [rows, frames_per_window, classes] f32 (model output of the push); acc [n_slots, ring_frames,
 *   classes] f32; out [rows_out, classes] f32 receives frames lo .. n_final-1 of each entry at out_row;
 *   max_span >= (k0+m-1)*overlap_interval + frames_per_window - lo of every entry with m > 0 (and n_final - lo). */
int sed_live_merge(const float* window_frames, const int* table, int n_entries, int max_span, int frames_per_window,
                   int classes, int overlap_interval, int sample_duration, int ring_frames, float* acc, float* out,
                   void* stream);

/* Resumable activity_detection utils/vad.py:11-199 on the frames sed_live_merge finalized (`frames` = its `out`):
 * events are reported as soon as no later frame can change them, close flushes the rest (quirks as sed_events).
 *   state [n_slots, classes, SED_LIVE_EVENT_STATE_INTS] i32 (reset when lo == 0); high/low/n_smooth/n_salt as
 *   sed_events (low may be NULL); events i32 pairs (bgn, fin) at the table's ev_off / ev_cap; counts
 *   [n_entries, classes] i32 (may exceed ev_cap: only ev_cap are stored). */
int sed_live_events(const float* frames, const int* table, int n_entries, int classes, const double* high,
                    const double* low, const int* n_smooth, const int* n_salt, void* state, int* events, int* counts,
                    void* stream);

/* ---- Sample-rate conversion and downmix ---------------------------------------------------------------------------
 * Replaces librosa.load(path, sr=sample_rate, mono=True) of pytorch/predict.py:288-295 for decoded audio: the
 * channels are averaged (numpy's x.astype(float32).mean(axis=1), int16 PCM as q / 32767), then
 *   y[j] = sum_i x[i] * taps[j*down + half - i*up]   (0 <= j < ceil(n_in*up/down); x[i] = 0 outside [0, n_in))
 * is summed over ascending i in float32 FMAs -- scipy.signal.resample_poly(x, up, down, window=h) with taps = up*h.
 * Both device entries take the taps sed_resample_filter returns (n_taps = 2*half + 1 floats on the device; any
 * odd-length filter works), int16 (dtype 1) or float32 (dtype 0) frames of 1 <= channels <= 8 interleaved samples. */

/* HOST helper: the polyphase filter for in_rate -> out_rate (both 1 .. 384000).  up = out_rate/g, down = in_rate/g
 * (g = gcd), half = 64*max(up, down), *n_taps = 2*half + 1; taps_or_NULL (host, *n_taps floats) receives
 * float32(up * h), h = scipy.signal.firwin(n_taps, 0.9475937167399596 / max(up, down), window=('kaiser',
 * 14.769656459379492)) computed in float64 (resampy's kaiser_best design).  Call with NULL for the sizes first.
 * SED_ERR_UNSUPPORTED when max(up, down) > 4096. */
int sed_resample_filter(int in_rate, int out_rate, int* up, int* down, int* n_taps, float* taps_or_NULL);

/* Many recordings in one launch.  table [n_rows, 4] i64 = (first frame in src, n_in frames, first sample in dst,
 * n_out samples); max_out >= every n_out.  dst f32: only the n_out samples of each row are written. */
int sed_resample(const void* src, int dtype, int channels, const long* table, int n_rows, long max_out,
                 const float* taps, int up, int down, int half, float* dst, void* stream);

/* Live ingest with resampling: computes model-rate samples of live streams into the mirrored rings of
 * sed_live_ingest (arena f32 [n_slots, 2*ring_samples]).  table [n_entries, 6] i64 = (slot, first output j0, outputs
 * (<= max_len), first frame of the stream's chunk in src or -1 to write zeros, n_prev = input frames before this
 * push, n_end = input frames after it).  Input i reads the chunk for n_prev <= i < n_end, the slot's history
 * hist[slot*history_len + i mod history_len] (f32) for 0 <= i < n_prev, and zero otherwise: an output must only need
 * i >= n_prev - history_len.  After the outputs, history_table [n_history, 4] i64 = (slot, first frame of the chunk
 * in src, n_prev, frames) stores the last min(frames, history_len) downmixed inputs of each chunk into its history:
 * pass it with the last call of a push (n_history = 0 otherwise; table may be NULL when n_entries = 0). */
int sed_live_resample(const void* src, int dtype, int channels, const long* table, int n_entries, long max_len,
                      const float* taps, int up, int down, int half, long ring_samples, float* arena, float* hist,
                      int history_len, const long* history_table, int n_history, void* stream);

/* ---- Peer-memory result buffers (multi-GPU gather without a collective on the data path) -------------------------
 * The reference gathers replica outputs on GPU 0 inside torch.nn.DataParallel (pytorch/main_strong.py:541,
 * pytorch/predict.py:239).  Here the destination rank owns ONE buffer for the results of all ranks; every other rank
 * (one process per GPU) maps it through CUDA IPC and passes its slice as the `clip` / `frame` output pointers of
 * sed_attpool* / sed_fcpool, whose stores then travel over NVLink to the destination GPU: the gather is fused into
 * the pooling head's epilogue.  These five entries are the only ones that allocate; they are explicit alloc / free
 * calls made by the caller, host-synchronous, and work on the calling thread's current CUDA device.
 *   sed_peer_alloc : cudaMalloc of `bytes` on the current device (a dedicated allocation, exportable as a whole)
 *   sed_peer_export: 64-byte IPC handle (HOST buffer) of an allocation made by sed_peer_alloc
 *   sed_peer_open  : map another process's allocation into this process (peer access enabled lazily)
 *   sed_peer_close / sed_peer_free: undo sed_peer_open / sed_peer_alloc
 *   sed_peer_copy  : asynchronous copy-engine transfer between any two device pointers visible to this process
 *                    (local or peer-mapped) on `stream` -- the push variant: results leave over NVLink by DMA while
 *                    the SMs already run the next batch */
int sed_peer_alloc(long bytes, void** dev_ptr);
int sed_peer_free(void* dev_ptr);
int sed_peer_export(const void* dev_ptr, unsigned char* handle64);
int sed_peer_open(const unsigned char* handle64, void** dev_ptr);
int sed_peer_close(void* dev_ptr);
int sed_peer_copy(void* dst, const void* src, long bytes, void* stream);
/* Stream-ordered 32-bit flags (driver stream memory operations; no kernel runs, no SM is occupied) on LOCAL device
 * memory: a producer rank writes step + 1 into a local word and copies the word into the consumer's flag array with
 * sed_peer_copy behind its data; the consumer's stream waits until the flag is cyclically >= the value.  With them the
 * ranks never meet in a collective: each runs at its own pace, only the consumer waits for what it consumes. */
int sed_stream_write32(void* dev_ptr, unsigned int value, void* stream);
int sed_stream_wait_geq32(void* dev_ptr, unsigned int value, void* stream);

#ifdef SED_PROFILE
/* Developer builds only (make -C sound-event-detection_b200/csrc profile -> libsed_b200_profile.so): sed_bigru that
 * also records clock64() stamps of CTA 0 for recurrence steps 8..15 (stamps: device buffer of 8*12 long long). */
int sed_bigru_profile(const float* gi, const void* whh_packed, const float* bhh, int B, int T, float* out,
                      void* workspace, int dtype, long long* stamps, void* stream);
#endif

/* softmax(q k^T / 8) v for 8 heads of 64.  Replaces ScaledDotProductAttention.forward
 * pytorch/models.py:808-820 and the head split/merge :863-875.
 *   qkv rows of 1536 f32 = [q | k | v], head h = columns h*64..h*64+63; out16 rows of 512 16-bit values.
 *   Row of (clip b, step t) = b*row_stride_b + t*row_stride_t in both tensors: (0, 0) selects the clip-major
 *   default (1, T); (Bp, 1) is time-major over a batch padded to Bp clips. */
int sed_mha_core(const float* qkv, int B, int T, long row_stride_t, long row_stride_b, void* out16, int dtype,
                 void* stream);

/* The same attention on the tensor cores, for T <= 128 pooled steps (clips up to 10.24 s): per (clip, head)
 * S = Q K^T and O = P V are tcgen05 MMAs with S / O in TMEM and the softmax in registers; operands arrive by TMA
 * straight from the 16-bit output of the QKV projection, so no float32 q | k | v tensor exists.  Replaces
 * pytorch/models.py:808-820, 863-875 like sed_mha_core.
 *   qkv16 [T * Bp, 1536] 16-bit, row of (step t, clip b) = t * Bp + b (time-major over the batch padded to Bp),
 *   columns [q | k | v]; qk_lo16 [T * Bp, 1024] 16-bit or NULL: the residuals q - q16 | k - k16 written by
 *   sed_linear_split16 -- with them the logits are accumulated as q_hi k_hi + q_lo k_hi + q_hi k_lo (float32-grade:
 *   the softmax exponentiates them, so operand rounding there is amplified by the logit magnitude);
 *   ctx16 [T * Bp, 512] 16-bit in the same row order (rows of clips >= B are left untouched). */
int sed_mha_attention(const void* qkv16, const void* qk_lo16, int B, int T, long Bp, void* ctx16, int dtype,
                      void* stream);

/* sed_linear without activation whose result leaves as split 16-bit operands: out_hi [M, N] = the rounded values,
 * out_lo [M, lo_cols] = (value - out_hi) rounded, for the first lo_cols columns (a multiple of 128, N <= 1536). */
int sed_linear_split16(const void* a16, long M, int K, const void* w16, const float* bias, int N, void* out_hi,
                       void* out_lo, int lo_cols, int dtype, void* stream);

/* Frame-attention pooling + framewise interpolation/padding.
 * Replaces AttBlock.forward pytorch/models.py:161-169, interpolate :84-95, pad_framewise_output :65-81.
 *   x [B, T, 512] f32; w_att/w_cla [25][512]; b_att/b_cla [25];
 *   clip [B,25]; frame [B, frames_out, 25] (frames_out >= T*ratio, padded with the last frame);
 *   cla_t / norm_att_t [B,25,T] or NULL. */
int sed_attpool(const float* x, int B, int T, const float* w_att, const float* b_att, const float* w_cla,
                const float* b_cla, int ratio, int frames_out, float* clip, float* frame, float* cla_t,
                float* norm_att_t, void* stream);

/* ---- Weight preparation: what the reference gets for free by keeping nn.Module parameters.  One-time work per
 * checkpoint; with these a caller needs no tensor library to go from a reference-layout state_dict (raw float32
 * arrays) to the packed operands the entries above take (examples/sed_infer.c does exactly that). ---- */

/* Eval-mode BatchNorm as y = x*scale + shift: scale = weight / sqrt(running_var + eps), shift = bias - running_mean*scale,
 * folded in float64, results float32.  Replaces nn.BatchNorm2d.forward in eval mode (bn0 pytorch/models.py:642-644,
 * bn1/bn2 of ConvBlock :128-129; eps = 1e-5).  All arrays [channels] f32 on the device. */
int sed_fold_bn(const float* weight, const float* bias, const float* running_mean, const float* running_var,
                int channels, double eps, float* scale, float* shift, void* stream);

/* nn.Conv2d weight [cout, cin, 3, 3] f32 (pytorch/models.py:103-111) -> wpacked [cout][3*kh+kw][cin] 16-bit (round to
 * nearest even), the operand layout of sed_conv3x3_bn_relu / sed_conv_block1. */
int sed_pack_conv3x3(const float* w_oihw, int cout, int cin, void* wpacked, int dtype, void* stream);

/* conv_block1.conv1 weight [64, 1, 3, 3] f32 times the folded bn1 scale [64] (float64 product, float32 result)
 * -> w1_scaled [64][9] for sed_conv_block1. */
int sed_pack_conv_first(const float* w1, const float* scale1, float* w1_scaled, void* stream);

/* nn.GRU weight_hh_l0 / weight_hh_l0_reverse [768, 256] f32 (rows [r | z | n]) -> whh_packed [2*768, 256] 16-bit in the
 * row order sed_bigru documents. */
int sed_pack_gru_whh(const float* whh_fwd, const float* whh_bwd, void* whh_packed, int dtype, void* stream);

/* float32 -> 16-bit (round to nearest even) for the nn.Linear / weight_ih operands of sed_linear. */
int sed_cast_16(const float* src, long n, void* dst, int dtype, void* stream);

/* Range guard of the 16-bit path.  The reference computes in float32 (no range limit); here every conversion of an
 * activation or weight to 16 bits saturates, so a value beyond the format's range is stored as exactly +-MAX (fp16:
 * 65504).  Adds to *count (device, 8 bytes, zeroed by the caller) the number of stored values of x[0..n) with
 * |x| >= MAX or non-finite, i.e. the conversions that clipped.  Used on packed weights at load time and on the
 * activation buffers by PackedModel.saturation_report (a checkpoint whose BatchNorm statistics do not bound the
 * activations trips it; results would silently differ from the reference otherwise). */
int sed_count_saturated16(const void* x, long n, int dtype, unsigned long long* count, void* stream);

/* Front-end constants, HOST pointers: twiddle_host [n_fft][2] f32 = (cos, sin)(-2 pi k / n_fft) computed in float64;
 * the banded form of the loaded mel matrix melW_host [F, n_mels] f32 (LogmelFilterBank.melW, pytorch/stft.py:688-693):
 * mel_lo/mel_len/mel_off [n_mels], mel_val [val_capacity] (F*n_mels always suffices), *n_val = values written. */
int sed_frontend_twiddle(int n_fft, float* twiddle_host);
int sed_band_mel(const float* melW_host, int F, int n_mels, int* mel_lo, int* mel_len, int* mel_off, float* mel_val,
                 int val_capacity, int* n_val);

#ifdef __cplusplus
}
#endif
#endif /* SED_B200_H_ */
