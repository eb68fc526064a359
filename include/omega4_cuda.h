/* omega4_cuda.h -- C ABI of libomega4_cuda.so: the B200 (sm_100a) implementation of OMEGA-4's
 * per-frame analysis hot path.  Plain C linkage, plain pointers and sizes, no C++/torch types.
 *
 * The reference (magicat777/Audio-Analyzer-OMEGA) is 100 % Python and has no FFI; its boundary for
 * this path is a set of Python classes (SURVEY.md section 8b).  Each entry point below names the
 * reference interface it replaces (paths relative to the reference root); the thin Python shims in
 * audio-analyzer-omega_b200/omega4_b200/ keep those classes' signatures and call these functions
 * through ctypes (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions
 *   - every function returns OMEGA4_OK (0) or a negative error code; omega4_last_error() returns a
 *     thread-local message for the last failure.  Nothing here falls back to the CPU.
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  Calls are
 *     asynchronous on that stream in OMEGA4_MEM_DEVICE mode and synchronous in OMEGA4_MEM_HOST mode.
 *   - `mem` says where the DATA pointers of that call live (samples, frames, outputs).  Table
 *     pointers in omega4_plan_desc are always host memory and are copied at plan creation.
 *   - sample/frame pointers must be 16-byte aligned in device mode.
 */
#ifndef OMEGA4_CUDA_H
#define OMEGA4_CUDA_H

#ifdef __cplusplus
extern "C" {
#endif

#define OMEGA4_ABI_VERSION 4

#define OMEGA4_OK 0
#define OMEGA4_ERR_INVALID (-1)   /* bad argument */
#define OMEGA4_ERR_CUDA (-2)      /* a CUDA runtime call failed */
#define OMEGA4_ERR_UNSUPPORTED (-3)
#define OMEGA4_ERR_NO_DEVICE (-4)

#define OMEGA4_MEM_HOST 0
#define OMEGA4_MEM_DEVICE 1

#define OMEGA4_MAX_RES 8
#define OMEGA4_METER_WINDOW 2048                 /* FFT_SIZE_BASE, omega4/config/config.py:12 */
#define OMEGA4_METER_STATE_DOUBLES (8 + 3600 + 60) /* carry state per channel for omega4_meter_stats */
#define OMEGA4_N_METERS 5                        /* momentary, short_term, integrated, range, true_peak */

/* omega4_analyze flags */
#define OMEGA4_FLAG_TIME_KERNELS 1               /* record CUDA events around every kernel launch */
#define OMEGA4_FLAG_FRESH_METERS 2               /* ignore meter_state contents on entry */
#define OMEGA4_FLAG_CONCURRENT_METERS 4          /* run the K-weighting + statistics kernels on an internal side
                                                    stream, concurrently with the FFT kernels (helps small batches
                                                    that under-fill the GPU; measured slower at 2048 channels) */

#define OMEGA4_FLAG_NO_BLOCKDFT 8                /* evaluate every resolution with the full FFT kernel even where the fused
                                                    output needs only a few bins (default: hop-block partial DFT there) */

#define OMEGA4_FLAG_NO_TENSOR 16                 /* run the hop-block partial DFT GEMM on the CUDA cores (fp32 FFMA) instead
                                                    of the tensor cores (tcgen05 kind::tf32, 3xTF32 split precision) */
#define OMEGA4_FLAG_TENSOR 32                    /* force the tensor-core GEMM when the plan default is off (OMEGA4_TENSOR=0) */

/* Environment knobs read by the library (developer / A-B measurement; defaults are the product path):
     OMEGA4_BLOCKDFT_FD=1       plan build: cosine-sum (frequency-domain) windowing for every hop-block resolution
                                instead of the exact-windowing GEMM operand (DESIGN.md 4.1b)
     OMEGA4_BLOCKDFT_UNFUSED=1  plan build: write the GEMM result Q and assemble frames in a separate kernel
     OMEGA4_KW_F64=1            per call: float64-state K-weighting kernel instead of the float32-state one
     OMEGA4_TENSOR=0            plan build: hop-block GEMM on the CUDA cores unless OMEGA4_FLAG_TENSOR is passed
     OMEGA4_HOST_CHUNK_MB=n     plan build: device bytes per slot of the host-buffer pipeline (default 1024)
     OMEGA4_STREAM_GRAPH=0      omega4_stream_hop: launch eagerly instead of replaying the captured CUDA graph
     OMEGA4_TP_F32=1            per call: float32 true-peak kernel for the batch path too (see OMEGA4_FLAG_EXACT_TRUE_PEAK)
     OMEGA4_TC_ONE_TILE_PER_CTA=1  per call: hop-block GEMM with one tile per CTA instead of the persistent walk */

#define OMEGA4_FLAG_SERIAL_STATS 64               /* keep the deque-statistics kernel on the caller's stream (default: it
                                                    runs on an internal side stream underneath the FFT kernels) */

#define OMEGA4_FLAG_FRESH_BARS 128                /* omega4_analyze_io: ignore bars_state contents on entry */

#define OMEGA4_FLAG_EXACT_TRUE_PEAK 256           /* batch entry points: evaluate the transforms of the 4x true peak in
                                                    float32 (4e-6 dBTP from the reference) instead of half precision on
                                                    two frame pairs at a time (<= 0.025 dBTP, bar 0.05; truepeak16_kernel.cuh).
                                                    The explicit-frame entry points always use float32. */

typedef struct omega4_plan omega4_plan;

/* Everything that defines the reference's behaviour is DATA computed on the host with the
 * reference's own formulas (SURVEY.md section 7 step 3) and handed over here. */
typedef struct omega4_plan_desc {
    int sample_rate;
    int hop;                       /* CHUNK_SIZE = 512 */
    int n_res;                     /* number of FFT resolutions, <= OMEGA4_MAX_RES */
    const int* fft_sizes;          /* [n_res] powers of two in 512 .. 32768 */
    const float* windows;          /* concatenated float32 windows, sum(fft_sizes) entries
                                      (MultiResolutionFFT._setup_windows, multi_resolution_fft.py:171-193) */
    const float* bin_weights;      /* concatenated per-bin weights, sum(fft_size/2+1) entries, or NULL
                                      (_apply_psychoacoustic_weighting, :304-333) */
    int target_bins;               /* T of combine_results_optimized (:335) */
    const int* tb_count;           /* [n_res] target bins fed by each resolution */
    const int* tb_idx;             /* concatenated target-bin indices */
    const int* tb_lo;              /* concatenated lower FFT-bin index of the np.interp segment */
    const float* tb_frac;          /* concatenated interpolation fractions */
    const float* res_weight;       /* [n_res] FFTConfig.weight (:149-154) */
    int meter_window;              /* must be OMEGA4_METER_WINDOW */
    const double* meter_hann;      /* [meter_window] float64 np.hanning (omega4_main.py:953) */
    const double* kw_coeffs;       /* hp_b[3] hp_a[3] shelf_b[3] shelf_a[3]
                                      (create_k_weighting_filter, professional_meters.py:48-72) */
    double gate_threshold;         /* -70.0 (:36) */
} omega4_plan_desc;

int omega4_abi_version(void);
const char* omega4_last_error(void);
int omega4_device_count(void);

/* ---- plan ------------------------------------------------------------------------------- */
omega4_plan* omega4_plan_create(const omega4_plan_desc* desc, int device);
void omega4_plan_destroy(omega4_plan* plan);

/* Frequency weighting of the meters (SURVEY.md section 8f rank 2): ProfessionalMetering.weighting_mode
 * 'K' / 'A' / 'C' / 'Z' (professional_meters.py:74-127, 129-229).  A weighting is a cascade of up to
 * four zero-phase sections, each scipy.signal.filtfilt(b, a, x) of order 1 or 2 with scipy's default
 * odd padding (padlen 3 * (order + 1)):
 *   K: 2 sections, blend = 1      -> out = f0 + 0.3 (f1 - f0)            (:137-151; the plan's default)
 *   A: hp1, hp2, lp1, lp2, gain 2.5                                      (:166-190)
 *   C: hp, lp, gain 1                                                    (:205-216)
 *   Z: n_sections = 0, rms_gate = 0                                      (:228-229)
 * rms_gate: frames with rms < 1e-6 weigh to zeros (:132-134, :158-160, :197-199).
 * Affects omega4_analyze and omega4_meter_frames on this plan from the next call on; NULL restores K. */
typedef struct omega4_weighting {
    int n_sections;
    int order[4];
    double b[4][3];
    double a[4][3];
    int blend;
    int rms_gate;
    double gain;
} omega4_weighting;
int omega4_plan_set_weighting(omega4_plan* plan, const omega4_weighting* weighting);

/* ProfessionalMetering.gate_threshold (professional_meters.py:36, read at :267 on every calculate_lufs):
 * values <= gate_threshold are left out of the integrated loudness and the loudness range.  Takes effect
 * from the next omega4_analyze / omega4_meter_stats call on this plan (the plan descriptor's value until then). */
int omega4_plan_set_gate_threshold(omega4_plan* plan, double gate_threshold);

/* The whole hot path over a batch: replaces, per channel and hop,
 *   MultiResolutionFFT.process_audio_chunk + combine_results_optimized (multi_resolution_fft.py:228,335)
 *   ProfessionalMetering.calculate_lufs on the Hann-windowed last 2048 samples (professional_meters.py:231)
 * as the caller omega4_main.py:928-1082 drives them, on the shared schedule of SURVEY.md section 7:
 * hop k of a channel ends at sample (k+1)*hop; resolution N contributes once hist_samples+(k+1)*hop >= N.
 *   samples        [n_ch] rows, row c starts at samples + c*ch_stride; `hist_samples` valid samples
 *                  precede each row start (carry of a previous time tile), 0 for a fresh stream
 *   combined       [n_ch][n_hops][target_bins] float32, or NULL
 *   magnitudes     [n_res] pointers (entries may be NULL) to [n_ch][n_hops][N/2+1] float32, or NULL
 *   meters         [n_ch][n_hops][5] float32 (M, S, I, LRA, TP), or NULL
 *   lufs_inst/tp_db [n_ch][n_hops] float64 per-frame values, or NULL (internal scratch is used)
 *   meter_state    [n_ch][OMEGA4_METER_STATE_DOUBLES] carried deque state, or NULL (fresh meters) */
int omega4_analyze(omega4_plan* plan, void* stream, int mem,
                   const float* samples, long long ch_stride, int n_ch, int n_hops, int hist_samples,
                   float* combined, float* const* magnitudes, float* meters,
                   double* lufs_inst, double* tp_db, double* meter_state, int flags);

/* Same path fed with the capture side's wire format (SURVEY.md section 8f rank 4): interleaved
 * little-endian int16 frames, x = int16 / 32768 as AudioCaptureManager._capture_loop decodes "s16le"
 * (omega4/audio/capture.py:571-574).  Stream g starts at frames + g*stream_stride (int16 units, first
 * NEW frame; hist_frames frames precede it); n_interleaved channels per frame (1 = the capture's mono
 * chunks, 2 / 8 = stereo / 7.1 files).  Outputs are indexed by planar channel g*n_interleaved + c,
 * n_ch = n_streams*n_interleaved, exactly as omega4_analyze's.  Halves the host->device bytes. */
int omega4_analyze_s16(omega4_plan* plan, void* stream, int mem,
                       const short* frames, long long stream_stride, int n_streams, int n_interleaved,
                       int n_hops, int hist_frames,
                       float* combined, float* const* magnitudes, float* meters,
                       double* lufs_inst, double* tp_db, double* meter_state, int flags);

/* The same path with every optional input / output in one descriptor, plus the application's post-processing
 * fused behind the combine step: what process_audio_spectrum hands the display is `band_values`
 * (omega4_main.py:992-1056 -> omega4_bars_*), so a caller that only draws bars and meters asks for
 * band_values + meters and never moves the combined spectrum off the device.
 *   samples / frames_s16   exactly one is non-NULL (float32 planar rows, or interleaved int16 as omega4_analyze_s16)
 *   stride                 ch_stride (float units) or stream_stride (int16 units); n_ch planar channels in total
 *   bars                   an omega4_bars object on the plan's device with spectrum_len == target_bins, or NULL
 *   band_values, peak_values  [n_ch][n_hops][omega4_bars_count(bars)] (peak_values may be NULL)
 *   bars_state             [n_ch][1 + count] float32 smoothing state carried between calls, or NULL (fresh)
 * Every other field means what the omega4_analyze argument of the same name means. */
typedef struct omega4_bars omega4_bars;
typedef struct omega4_io {
    const float* samples;
    const short* frames_s16;
    int n_interleaved;
    long long stride;
    int n_ch, n_hops, hist;
    float* combined;
    float* const* magnitudes;
    float* meters;
    double* lufs_inst;
    double* tp_db;
    double* meter_state;
    omega4_bars* bars;
    float* band_values;
    float* peak_values;
    float* bars_state;
    int flags;
} omega4_io;
int omega4_analyze_io(omega4_plan* plan, void* stream, int mem, const omega4_io* io);

/* ---- streaming entry points: one round trip per application frame -------------------------- */
/* MultiResolutionFFT.process_audio_chunk (multi_resolution_fft.py:228-302) for the resolutions whose ring has
 * filled, and combine_results_optimized (:335-408) over exactly those, in ONE host round trip: frames[r] is the
 * latest fft_size[r] samples of resolution r's ring (HOST float32) or NULL when that ring is not ready;
 * magnitudes[r] receives |X| x weights (fft_size[r]/2+1 values); combined ([target_bins], may be NULL) the
 * combination of the ready resolutions (zeros when none is).  Synchronous; staging buffers are pinned and
 * owned by the plan. */
int omega4_stream_hop(omega4_plan* plan, const float* const* frames, float* const* magnitudes, float* combined);

/* ProfessionalMetering.calculate_lufs (professional_meters.py:231-281) on ONE float64 frame of
 * OMEGA4_METER_WINDOW samples in one host round trip: weighting + mean square, true peak, deque statistics.
 * state: HOST [OMEGA4_METER_STATE_DOUBLES], read (unless fresh) and written; meters: HOST float[5]
 * (M, S, I, LRA, TP); lufs_inst / tp_db: this frame's values, or NULL. */
int omega4_meter_update(omega4_plan* plan, const double* frame, double* state, int fresh, float* meters,
                        double* lufs_inst, double* tp_db);

/* combine_results_optimized (multi_resolution_fft.py:335-408) on caller-supplied magnitudes:
 * magnitudes[r] = [n_rows][N_r/2+1] or NULL when resolution r is absent from `results`. */
int omega4_combine(omega4_plan* plan, void* stream, int mem,
                   const float* const* magnitudes, int n_rows, float* combined);

/* ProfessionalMetering on explicit float64 frames of OMEGA4_METER_WINDOW samples
 * (apply_k_weighting :129, calculate_lufs :237-246, calculate_true_peak :283).
 * lufs_inst / tp_db: [n_frames]; weighted: [n_frames][W] K-weighted frames or NULL. */
int omega4_meter_frames(omega4_plan* plan, void* stream, int mem,
                        const double* frames, int n_frames,
                        double* lufs_inst, double* tp_db, double* weighted);

/* The deque statistics of calculate_lufs (professional_meters.py:248-279) over per-frame series. */
int omega4_meter_stats(omega4_plan* plan, void* stream, int mem,
                       const double* lufs_inst, const double* tp_db, int n_ch, int n_frames,
                       int first_frame, double* state, float* meters, int fresh);

/* ---- plan-less entry points --------------------------------------------------------------- */
/* Batched windowed rFFT + magnitude: BatchedFFTProcessor._process_size_group_{gpu,cpu}
 * (batched_fft_processor.py:197-285) and GPUAcceleratedFFT.compute_fft / process_fft_batch
 * (gpu_accelerated_fft.py:92-177, 300-340).  frames [batch][n] float32; window [n] HOST float32 or
 * NULL; magnitude [batch][n/2+1]; complex_out interleaved (re,im) [batch][n/2+1][2] or NULL. */
int omega4_rfft_batch(int device, void* stream, int mem, const float* frames, int batch, int n,
                      const float* window, float* magnitude, float* complex_out);

/* PrecomputedFrequencyMapper.map_spectrum_to_bars (freq_mapper.py:165-196): bar = mean(spectrum[s:e])
 * with optional compensation curve; bands [n_bars][2] HOST int32; comp [len] HOST or NULL.
 * db = 1 additionally converts 20*log10(max(x,1e-10)) (panels/spectrogram_waterfall.py:85),
 * db = 2 converts 20*log10(x + 1e-10) (plugins/panels/spectrogram.py:72). */
int omega4_band_map(int device, void* stream, int mem, const float* spectrum, int n_rows, int len,
                    const int* bands, int n_bars, const float* comp, float* bars_out, int db);

/* SpectrogramWaterfall.update + _normalize_spectrum (omega4/panels/spectrogram_waterfall.py:71-121), data side:
 * per row  dB = 20 log10(max(spectrum[lo:hi], 1e-10))  (db_form 0; db_form 1 = the plugin panel's
 * 20 log10(x + 1e-10), plugins/panels/spectrogram.py:72), (max, min) of the row into the panel's peak history,
 * with auto_gain current_peak / current_floor = 95th / 5th percentile of the last 20 maxima / minima, then
 * clip((dB + gain_adjustment - floor) / (peak - floor), 0, 1) (zeros when peak <= floor).
 *   spectra     [n_ch][n_rows][len] magnitudes, rows in time order
 *   state       [n_ch][OMEGA4_WATERFALL_STATE] float32 carried between calls (the last 19 (max, min) pairs, their
 *               count, current_peak, current_floor), or NULL; fresh != 0 ignores its contents on entry
 *               (a new panel: no history, peak 0, floor -80, :38-39)
 *   db_out, norm_out  [n_ch][n_rows][hi - lo] or NULL;  rowstat_out [n_ch][n_rows][4] = row max dB, row min dB,
 *               current_peak, current_floor after the row, or NULL */
#define OMEGA4_WATERFALL_STATE 41
int omega4_waterfall(int device, void* stream, int mem, const float* spectra, int n_ch, int n_rows, int len,
                     int lo, int hi, int db_form, int auto_gain, float gain_adjustment, float* state, int fresh,
                     float* db_out, float* norm_out, float* rowstat_out);

/* BassZoomPanel._process_bass_detail_internal (omega4/panels/bass_zoom.py:141-214) after its 8192-point
 * FFT (omega4_rfft_batch), without the wall-clock peak hold: per bar mean(|X|[first .. first+count)) * comp,
 * dynamic scaling 0.85/max * log10(max(1, 10 max))/2, compression above 0.7, attack/release smoothing
 * against the previous bars, clamp [0,1].  magnitudes [n_ch][n_frames][n_bins]; bar_bins [n_bars][2]
 * (first bin, count; count 0 = bar keeps its value) and comp [n_bars] are HOST tables; state
 * [n_ch][n_bars] carries bass_bar_values between calls (NULL: zeros); bars_out [n_ch][n_frames][n_bars]. */
int omega4_bass_bars(int device, void* stream, int mem, const float* magnitudes, int n_ch, int n_frames,
                     int n_bins, const int* bar_bins, const float* comp, int n_bars, float* state, float* bars_out);

/* Device-side synthetic multi-stream audio for the headless batch driver (sweep + counter-hash noise). */
int omega4_synth_fill(int device, void* stream, float* out_device, int n_streams, int n_channels,
                      long long n_samples, long long row_stride, int first_stream, int sample_rate,
                      long long clip_samples);

/* ---- application post-processing (SURVEY.md section 8f rank 1) ---------------------------- */
/* The block of ProfessionalLiveAudioAnalyzer.process_audio_spectrum between the combined spectrum and
 * `band_values` (omega4_main.py:992-1056): np.percentile(spectrum, 98) normalisation x 0.8,
 * apply_frequency_compensation (:855-926, as a per-bin gain table), optional max normalisation,
 * mel band mean -> sqrt -> clamp [0,1] over PrecomputedFrequencyMapper's band table (the loop stops
 * at the first band reaching past the spectrum, :1012-1013), per-band exponential smoothing
 * against the previous frame (:1041-1056).  Tables are host pointers, copied at creation. */
typedef struct omega4_bars_desc {
    int spectrum_len;              /* T: length of one combined spectrum (self.bars) */
    int n_bars;                    /* entries in `bands` */
    const int* bands;              /* [n_bars][2] (start, end) FFT-bin pairs (freq_mapper.py:83-124) */
    const float* gain;             /* [T] frequency-compensation gains, or NULL (freq_compensation_enabled off) */
    const double* smooth;          /* [n_bars] smoothing factor per band (:1046-1052), or NULL (smoothing off) */
    double percentile;             /* 98 */
    float scale;                   /* 0.8 */
    int normalize_max;             /* normalization_enabled (:1005) */
} omega4_bars_desc;
omega4_bars* omega4_bars_create(const omega4_bars_desc* desc, int device);
void omega4_bars_destroy(omega4_bars* bars);
/* number of bars produced per frame: bands whose end <= spectrum_len, at most n_bars */
int omega4_bars_count(const omega4_bars* bars);
/* spectrum [n_ch][n_hops][T] -> band_values [n_ch][n_hops][count] (+ peak_values = unsmoothed, or NULL).
 * state [n_ch][1 + count] float32 carries prev_band_values between calls (state[0] != 0: present);
 * NULL or fresh != 0 starts every channel without a previous frame. */
int omega4_bars_run(omega4_bars* bars, void* stream, int mem, const float* spectrum, int n_ch, int n_hops,
                    float* state, int fresh, float* band_values, float* peak_values);

/* ---- ITU-R BS.1770-4 program loudness and EBU Tech 3342 loudness range (extension) ---------- */
/* Not part of the reference's behaviour: ProfessionalMetering (omega4_analyze's five meters) is not textbook
 * BS.1770 and stays as it is.  This object measures, per stream of C planar channels, the K-weighted
 * (high-shelf, then high-pass, run continuously from zero state) energy of every 100 ms sub-block of
 * sub = sample_rate / 10 samples, z_j = sum_c G_c sum y_c^2, and from it
 *   momentary  M_j = -0.691 + 10 log10(sum_{i=j-3..j} z_i / (4 sub))     NaN for j < 3
 *   short-term S_j = -0.691 + 10 log10(sum_{i=j-29..j} z_i / (30 sub))   NaN for j < 29;  -inf for zero energy
 * at the end of each sub-block j (counted from the stream start), the running sample peak per channel, and on
 * request the integrated loudness (gated at -70 LUFS and 10 LU below) and the loudness range (short-term values
 * gated at -70 and 20 LU below; v[floor(0.95 (n-1) + 0.5)] - v[floor(0.10 (n-1) + 0.5)] of the sorted survivors).
 * DESIGN.md section 4.7.  One call at a time per object (it owns its scratch buffers). */
#define OMEGA4_LOUDNESS_MAX_CH 32
typedef struct omega4_loudness omega4_loudness;
typedef struct omega4_loudness_desc {
    int sample_rate;               /* a multiple of 10 */
    int channels;                  /* C per stream, 1 .. OMEGA4_LOUDNESS_MAX_CH */
    const double* ch_weights;      /* [channels] G_c >= 0 (1 1 for stereo; 1 1 1 0 1.41 1.41 for 5.1 L R C LFE Ls Rs) */
    const double* shelf_b;         /* [3] K-weighting stage 1 (high-shelf), a[0] = 1 */
    const double* shelf_a;
    const double* hp_b;            /* [3] stage 2 (high-pass), a[0] = 1 */
    const double* hp_a;
    int sub;                       /* sample_rate / 10 */
} omega4_loudness_desc;
omega4_loudness* omega4_loudness_create(const omega4_loudness_desc* desc, int device);
void omega4_loudness_destroy(omega4_loudness* h);
/* doubles of carried state per stream: 30 + 6 C (sample count, last 29 sub-block energies, per channel the
 * filter state, the partial sub-block's energy and the sample peak) */
int omega4_loudness_state_doubles(const omega4_loudness* h);
/* Continue n_streams streams by n_samples samples each:
 *   samples      [n_streams * C] planar rows (stream-major: row s * C + c), row r at samples + r * ch_stride
 *   state        [n_streams][omega4_loudness_state_doubles] read (unless fresh) and written; every stream of one
 *                state array has received the same number of samples T (each push advances all of them)
 *   fresh        != 0: start every stream anew (T = 0), ignoring the contents of state
 *   momentary, short_term  [n_streams][out_stride] float32 LUFS, or NULL: column i of row s receives step
 *                floor(T / sub) + i of stream s.  A push of n samples after T emits
 *                floor((T + n) / sub) - floor(T / sub) steps, so the caller knows the count without a sync.
 *   sample_peak  [n_streams][C] float32 20 log10(max |x|) in dBFS over everything pushed since the start
 *                (-inf for silence), or NULL
 * Tile lengths are arbitrary (no multiple of sub or of 512 needed).  Values above -70 LUFS, the integrated loudness
 * and the loudness range agree across tilings to ~1e-6 LU.  Far below the gate they may not: where digital silence
 * follows a signal, a sub-block more than 100 ms into the silence reads either -inf (when the filter restarted from
 * zero over a silent 100 ms warm-up) or a finite value below -120 LUFS (the filter's decaying ringing, when it
 * continued from an earlier sub-block), and where the filter restarts depends on the push boundaries
 * (DESIGN.md section 4.7). */
int omega4_loudness_push(omega4_loudness* h, void* stream, int mem, const float* samples, long long ch_stride,
                         int n_streams, long long n_samples, double* state, int fresh, long long out_stride,
                         float* momentary, float* short_term, float* sample_peak);
/* momentary, short_term [n_streams][stride] series of n_steps steps each, counted from the stream start ->
 * out [n_streams][4] float32: integrated loudness (-inf when no block passes the gates), loudness range (0 when no
 * short-term value passes), max M, max S (NaN when n_steps leaves them undefined). */
int omega4_loudness_summary(omega4_loudness* h, void* stream, int mem, const float* momentary, const float* short_term,
                            int n_streams, int n_steps, long long stride, float* out);
/* number of kernels this library launched through `h` since creation (two per push, one per summary) */
long long omega4_loudness_launches(const omega4_loudness* h);

/* ---- one-third-octave band levels per channel (IEC 61260-1 bands; extension) ----------------- */
/* Not part of the reference's behaviour.  Per channel row: the base-10 one-third-octave bands x = -17 .. 13
 * (f_m = 1000 * 10^(x/10) Hz, edges f_m * 10^(-/+0.05)) whose upper edge lies below fs / 2, each filtered by the
 * 6th-order digital Butterworth band-pass that scipy.signal.butter(3, [f1, f2], "bandpass", fs=fs, output="sos")
 * designs (-3.01 dB at the edges), run continuously over the whole stream from zero state in float64.  At the end
 * of each 100 ms block j of sub = sample_rate / 10 samples (counted from the stream start) each band reads
 *   L = 10 log10(2 / sub * sum_{n in j} y^2)   dBFS (a full-scale sine in the band reads 0 dBFS; -inf for zero energy)
 * and column n_bands holds the same on the unfiltered input (the overall level).  Per row and column the object
 * also keeps Leq = 10 log10(2 sum y^2 / T) over all T samples pushed (an incomplete last block included) and
 * Lmax, the largest completed-block level; both -inf before any energy.  No channel summation, no weighting.
 * The band frequencies follow IEC 61260-1; conformance to its filter class acceptance limits is not claimed.
 * DESIGN.md section 4.8.  One call at a time per object (it owns its staging buffers). */
#define OMEGA4_OCTAVE_MAX_BANDS 31
typedef struct omega4_octave omega4_octave;
typedef struct omega4_octave_desc {
    int sample_rate;               /* a multiple of 10 in [8000, 192000] */
    int n_bands;                   /* 1 .. OMEGA4_OCTAVE_MAX_BANDS */
    const double* sos;             /* [n_bands][3][6] b0 b1 b2 a0 a1 a2 per section, a0 = 1, host memory, copied.  Each
                                      band's numerators are g [1, -2, 1], g [1, 2, 1] or g [1, 0, -1] with three zeros at
                                      z = 1 and three at z = -1 in all (scipy's pairing or tables.third_octave_sos); the
                                      poles must lie inside the unit circle.  The kernel runs every section with
                                      numerator [1, 0, -1] and applies the product of the b0 to the energy. */
    int sub;                       /* sample_rate / 10 */
} omega4_octave_desc;
omega4_octave* omega4_octave_create(const omega4_octave_desc* desc, int device);
void omega4_octave_destroy(omega4_octave* h);
/* doubles of carried state per row: 1 + 9 (n_bands + 1) (the sample count T, then per column the 6 filter values,
 * the partial block's energy, the energy of the completed blocks and the largest block energy) */
int omega4_octave_state_doubles(const omega4_octave* h);
/* Continue n_rows channel rows by n_samples samples each (one kernel launch):
 *   samples   [n_rows] rows, row r at samples + r * ch_stride (ch_stride >= n_samples; float alignment suffices)
 *   state     [n_rows][omega4_octave_state_doubles] doubles, read (unless fresh) and written; every row of one
 *             state array has received the same number of samples T
 *   fresh     != 0: start every row anew (T = 0), ignoring the contents of state
 *   levels    [n_rows][out_stride][n_bands + 1] float32 dBFS, or NULL: column i of row r receives block
 *             floor(T / sub) + i.  A push of n samples after T completes floor((T + n) / sub) - floor(T / sub)
 *             blocks, so the caller knows the count without a sync; blocks at column >= out_stride are not written
 *             (in host mode an out_stride below the count is an error).
 *   leq, lmax [n_rows][n_bands + 1] float32 dBFS over everything pushed since the start, or NULL
 * Tile lengths are arbitrary: the carried state is exact, so any cut of a stream into pushes gives bit-identical
 * levels, Leq and Lmax. */
int omega4_octave_push(omega4_octave* h, void* stream, int mem, const float* samples, long long ch_stride, int n_rows,
                       long long n_samples, double* state, int fresh, long long out_stride, float* levels, float* leq,
                       float* lmax);
/* number of kernels this library launched through `h` since creation (one per push with samples) */
long long omega4_octave_launches(const omega4_octave* h);

/* ---- introspection ------------------------------------------------------------------------ */
/* number of kernels this library launched through `plan` since creation */
long long omega4_plan_launches(const omega4_plan* plan);
/* After an omega4_analyze(..., OMEGA4_FLAG_TIME_KERNELS) call has completed: per-kernel device
 * times of that call.  names: array of max_n char[32] buffers.  Returns the number of kernels. */
int omega4_plan_kernel_times(omega4_plan* plan, char* names, float* ms, int max_n);

#ifdef __cplusplus
}
#endif
#endif /* OMEGA4_CUDA_H */
