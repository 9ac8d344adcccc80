/* gooey_batch.h — additive batch entry points of libgooey_b200.so.
 *
 * libgooey renders one engine / one voice per call, sample by sample, on one
 * CPU thread.  These entry points render THOUSANDS of independent voices or
 * engines in one call on an NVIDIA B200.  They sit beside (not instead of) the
 * reference's own C FFI (include/gooey.h): single-engine render/bounce keep
 * working as a batch of one.
 *
 * Plain C ABI: pointers and sizes only.  Every function returns 0 on success
 * and a negative GOOEY_E_* code on failure; gooey_b200_last_error() returns a
 * thread-local description.  There is NO CPU fallback: without a CUDA device
 * every compute entry fails with GOOEY_E_NO_DEVICE.
 */
#ifndef GOOEY_BATCH_H
#define GOOEY_BATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GOOEY_E_OK 0
#define GOOEY_E_INVALID (-1)
#define GOOEY_E_NO_DEVICE (-2)
#define GOOEY_E_CUDA (-3)

/* Instrument ids (reference: src/ffi.rs:1843-1853). */
#define GOOEY_INSTRUMENT_KICK 0u
#define GOOEY_INSTRUMENT_SNARE 1u
#define GOOEY_INSTRUMENT_HIHAT 2u
#define GOOEY_INSTRUMENT_TOM 3u
#define GOOEY_INSTRUMENT_BASS 4u
/* libgooey_b200 voice kinds beyond the five sequenced instruments (GooeyVoicePatch.instrument):
 * the poly synth (params = PolyConfig, 14 normalized values, src/instruments/poly_synth.rs:20-47) and the granulator
 * (GranulatorConfig::default; buffer, seed and parameters arrive as events: gooey_voice_batch_set_buffer / _share_buffer /
 * _set_seed / _set_param below). */
#define GOOEY_B200_VOICE_POLY 5u
#define GOOEY_B200_VOICE_GRANULATOR 6u

/* One voice patch = the argument list of the reference's `<Voice>::with_config`
 * (Rust API, instrument level):
 *   kick  : KickConfig::new_full order, 18 normalized values (src/instruments/kick.rs:118-160)
 *   snare : SnareConfig::new_full order, 19 values, filter_type at [13] (src/instruments/snare.rs:135-180)
 *   hihat : pitch, decay, attack, tone, volume; aux bit0 = pink noise, bit1 = 12 dB slope
 *           (HiHat2Config, src/instruments/hihat2.rs:41-70; default white / 24 dB)
 *   tom   : tune, bend, tone, color, decay, membrane, membrane_q, volume in 0-100 units
 *           (Tom2Config, src/instruments/tom2.rs:105-115); aux bit0 = 1 to apply it, 0 = Tom2::new defaults
 *   bass  : BassConfig order, 15 normalized values (src/instruments/bass.rs)
 * `tuning` (0.5 neutral) is params[23] when aux bit8 is set.
 */
typedef struct GooeyVoicePatch {
  uint32_t instrument;
  uint32_t aux;
  float params[24];
} GooeyVoicePatch;

typedef struct GooeyVoiceBatch GooeyVoiceBatch;

const char* gooey_b200_last_error(void);
/* Number of visible CUDA devices (0 = the library cannot compute). */
int gooey_b200_device_count(void);
/* Kernels launched by this process since load (bench.py reports it as gpu_launches). */
uint64_t gooey_b200_launch_count(void);
/* Device time (ms, CUDA events on the launching stream) of the most recent render call's kernels. */
float gooey_b200_last_kernel_ms(void);
/* Accumulated device time of one back-end kernel ("wave_kernel<KickW>" / "<SnareW>" / "<HatW>" / "<TomW>",
 * "coop_kernel<TomC>", "back_kernel", and for poly synths "poly_wave_kernel" or, under GOOEY_B200_BACKEND=serial,
 * "slow_kernel<PolyV>") since load or the last reset: launches, summed launch durations (ms, CUDA events on the launching
 * stream) and voice-frames written. */
int gooey_b200_kernel_stat(const char* kernel, uint64_t* launches, double* total_ms, double* voice_frames);
/* ';'-separated names of the kernels that have statistics (thread-local storage, valid until the next call) */
const char* gooey_b200_kernel_stat_names(void);
void gooey_b200_kernel_stats_reset(void);

/* Voice-level batch: n voices built `with_config`, then driven by per-voice events. */
int gooey_voice_batch_new(float sample_rate, uint32_t n_voices, const GooeyVoicePatch* patches, int device,
                          GooeyVoiceBatch** out_batch);
void gooey_voice_batch_free(GooeyVoiceBatch* b);
/* `voice.trigger_with_velocity(t_frame, velocity)` at frame `frame` (frames count from the batch's current position).
 * A poly voice has no such trigger and ignores it: it sounds only through gooey_voice_batch_note_on. */
int gooey_voice_batch_trigger(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, float velocity);
/* Same trigger for every voice; velocities may be NULL (=1.0). */
int gooey_voice_batch_trigger_all(GooeyVoiceBatch* b, uint32_t frame, const float* velocities);
/* FFI-style normalized parameter edit (`gooey_engine_set_*_param` ids) taking effect at `frame`; snap != 0 also snaps.
 * Poly voices: ids 0-13 = PolySynth::set_param (PolyConfig order); granulators: ids 0-11 as gooey_engine_granulator_set_param
 * (with snap = gooey_engine_granulator_snap_params).  The value is clamped to 0..1 and glides to its target unless snapped.
 * Unknown ids are ignored.  (Until libgooey_b200 played poly voices and granulators in batches, this call did nothing for
 * those two kinds.) */
int gooey_voice_batch_set_param(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t param, float value, int snap);
/* Poly voices and granulators.  Each call queues its events at `frame`, counted like gooey_voice_batch_trigger's.
 * GOOEY_E_INVALID, with a message and nothing queued, for a voice out of range, a voice of another kind, or the refusals
 * named below.
 *   note_on      PolySynth::trigger_note(note, velocity): note 0-127 (the reference's u8; above 127 is refused), velocity
 *                unclamped.  A seventh note steals the oldest of the six sub-voices.
 *   release      PolySynth::release_all.
 *   set_buffer   Granulator::set_buffer: copies `len` samples at `sample_rate` to the device.  Refused: samples NULL,
 *                len 0, a non-finite sample, or a sample_rate that is not finite and > 0.  Kills the voice's grains.
 *   share_buffer libgooey_b200 addition: dst_voice plays the buffer most recently set on or shared to src_voice (also a
 *                granulator; refused if it holds none) without a second device copy, so 1600 granulators over one 60 s
 *                source keep one copy.  The batch keeps each buffer while a voice or a queued event refers to it.
 *   set_seed     Granulator::set_seed (0 selects the reference's fixed non-zero seed). */
int gooey_voice_batch_note_on(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t note, float velocity);
int gooey_voice_batch_release(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame);
int gooey_voice_batch_set_buffer(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, const float* samples, uint32_t len, float sample_rate);
int gooey_voice_batch_share_buffer(GooeyVoiceBatch* b, uint32_t dst_voice, uint32_t frame, uint32_t src_voice);
int gooey_voice_batch_set_seed(GooeyVoiceBatch* b, uint32_t voice, uint32_t frame, uint32_t seed);
/* Render `frames` samples of every voice: out_host[v * frames + i] (host memory; copies are part of the call). */
int gooey_voice_batch_render(GooeyVoiceBatch* b, uint32_t frames, float* out_host);
/* Same as 16-bit PCM, `(s * 32767).round() as i16` (bounce.rs:105-113), quantised on the device: out_host[v * frames + i]. */
int gooey_voice_batch_render_pcm16(GooeyVoiceBatch* b, uint32_t frames, int16_t* out_host);
/* Same, leaving the result in device memory: out_dev[v * stride + i], stride >= frames. */
int gooey_voice_batch_render_device(GooeyVoiceBatch* b, uint32_t frames, float* out_dev, size_t stride);

/* ---- batches of Rust-API engines (reference: src/engine/mod.rs:109-253 Engine, src/bounce.rs:41-59 bounce_to_buffer) ----
 * One GooeyRsBatch holds n independent `Engine`s.  Per engine: named instruments (`Engine::add_instrument(name,
 * Box::new(<Voice>::with_config(sr, cfg)))`), sequencers that name their instrument (`Sequencer::with_pattern /
 * with_velocity_pattern(bpm, sr, pattern, name)`), `set_bpm`, `set_master_gain` (default 0.25) and the global effect chain,
 * which starts as [SoftLimiter(1.0)] (`clear_global_effects`, `add_global_effect(effect)`).
 * gooey_rs_batch_bounce = `bounce_to_buffer(&mut engine, BounceLength::Samples(samples))` of every engine in one device
 * pass: out_host[engine * samples + i], mono.  Bars / Beats lengths are converted by the host mirror (bounce.rs:20-32).
 *
 * Global effects: gooey_rs_batch_add_effect appends `effect_id` (the FFI effect ids of gooey.h) built at the batch's
 * sample rate from its constructor arguments after the sample rate, in the reference's order:
 *   0 LowpassFilterEffect (cutoff, resonance) · 1 DelayEffect (timing = DelayTiming index, bpm, feedback, mix, cutoff) ·
 *   2 TubeSaturation (drive, warmth, mix) · 3 TubeCompressor (threshold dB, ratio, attack ms, release ms, mix) ·
 *   4 TiltFilterEffect () · 5 SoftLimiter (threshold) · 6 SpringReverbEffect (decay, mix, damping) ·
 *   7 Waveshaper (drive, mix) · 8 FeedbackWaveshaper (drive, feedback, cutoff, mix) · 9 PlateReverbEffect (decay, mix, damping).
 * Each effect runs its mono `process` (the channel-0 path; the compressor is its own side-chain).  Effects keep their
 * state from one bounce to the next; clear_global_effects drops them.  set_bpm does not reach a DelayEffect: it keeps
 * the tempo it was built with.  GOOEY_E_INVALID (chain unchanged) for a bad engine, an unknown id, n_args other than
 * the kind's count, NULL args with n_args > 0, or a chain already GOOEY_RS_MAX_EFFECTS long.
 * gooey_rs_batch_add_limiter(b, e, th) = gooey_rs_batch_add_effect(b, e, 5, &th, 1). */
#define GOOEY_RS_MAX_EFFECTS 8
typedef struct GooeyRsBatch GooeyRsBatch;
int gooey_rs_batch_new(float sample_rate, uint32_t n_engines, int device, GooeyRsBatch** out_batch);
void gooey_rs_batch_free(GooeyRsBatch* b);
int gooey_rs_batch_add_instrument(GooeyRsBatch* b, uint32_t engine, const char* name, const GooeyVoicePatch* patch);
int gooey_rs_batch_add_sequencer(GooeyRsBatch* b, uint32_t engine, const char* instrument_name, float bpm, const uint8_t* enabled,
                                 const float* velocity, uint32_t steps);
int gooey_rs_batch_set_bpm(GooeyRsBatch* b, uint32_t engine, float bpm);
float gooey_rs_batch_get_bpm(const GooeyRsBatch* b, uint32_t engine);
int gooey_rs_batch_set_master_gain(GooeyRsBatch* b, uint32_t engine, float gain);
int gooey_rs_batch_clear_global_effects(GooeyRsBatch* b, uint32_t engine);
int gooey_rs_batch_add_limiter(GooeyRsBatch* b, uint32_t engine, float threshold);
int gooey_rs_batch_add_effect(GooeyRsBatch* b, uint32_t engine, uint32_t effect_id, const float* args, uint32_t n_args);
int gooey_rs_batch_bounce(GooeyRsBatch* b, uint32_t samples, float* out_host);
int gooey_rs_batch_bounce_device(GooeyRsBatch* b, uint32_t samples, float* out_dev, size_t stride);
/* Mono PCM WAV writer of bounce_to_wav (bounce.rs:80-133; ffi.rs:7942-7980): bit_depth 16 or 24, sample = round(s * (2^(bits-1) - 1)). */
int gooey_b200_write_wav(const char* utf8_path, const float* samples, uint32_t n, uint32_t sample_rate, uint32_t bit_depth);

/* 32-bit float WAV (WAVE_FORMAT_IEEE_FLOAT), 1 or 2 interleaved channels: the container of ffi.rs:8030-8048. */
int gooey_b200_write_wav_f32(const char* utf8_path, const float* interleaved, uint32_t frames, uint32_t channels, uint32_t sample_rate);
/* Pinned host memory for the drains above, allocated on the NUMA node `device` is attached to (*out_numa_node: the node, or
 * -1 when the placement could not be applied).  Free with gooey_b200_host_free. */
void* gooey_b200_host_alloc(size_t bytes, int device, int* out_numa_node);
void gooey_b200_host_free(void* p);

/* Host-only (no device needed): frames and velocities at which a bounce of an engine with this tempo, swing and step
 * pattern fires its triggers — the schedule the host resolves into kernel event tables (reference:
 * Sequencer::tick_with_settings, src/engine/sequencer.rs:883-952).  Returns the number of triggers (may exceed capacity). */
uint32_t gooey_b200_sequencer_schedule(float sample_rate, float bpm, float swing, const uint8_t* enabled, const float* velocity, uint32_t steps,
                                       uint32_t frames, uint32_t* out_frames, float* out_velocity, uint32_t capacity);

/* Host-only (no device): the pad hits a sampler rack's 16-step pattern resolves to over a sequence of render calls — the schedule the host
 * hands to the device (reference: SamplerRack::activate_start_if_due / tick_sequencer, src/instruments/sampler.rs:232-275; the transport,
 * src/mixer/clip_grid.rs:174-191, 656-660).  pending_beat < 0: the pattern already runs.  Returns the number of hits (may exceed capacity). */
uint32_t gooey_b200_sampler_schedule(float sample_rate, float bpm, float swing, const uint8_t* enabled, const uint8_t* pads, const float* velocity,
                                     int transport_running, double transport_beat, double pending_beat, int bounce, const uint32_t* calls, uint32_t n_calls,
                                     uint32_t* out_frames, uint32_t* out_pads, float* out_velocity, uint32_t capacity, double* out_transport_beat);

#ifdef __cplusplus
}
#endif
#endif /* GOOEY_BATCH_H */
