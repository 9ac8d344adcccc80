//! Rust host side of libgooey_b200: raw bindings of `include/gooey_batch.h` and safe wrappers that mirror
//! `gooey::bounce` (reference `src/bounce.rs`) for whole batches of engines.
//!
//! The reference resolves nothing ahead of time: `Engine::tick` walks sequencers and instruments sample by sample.
//! Here the host describes each engine (instruments as `with_config` argument lists, sequencer patterns, master gain,
//! global effect chain) once; the library resolves the sequencer schedule into per-voice trigger tables (bit-exact with
//! `Sequencer::tick_with_settings`) and renders every engine of the batch in one pass on a B200.
//!
//! This crate cannot be compiled in the repository's own image (no Rust toolchain there); it is the binding a libgooey
//! maintainer adds, kept next to the header it binds so the two stay in step.

pub mod bounce;

use std::ffi::{c_char, c_float, c_int, CStr, CString};

/// `GooeyVoicePatch` (include/gooey_batch.h): instrument id, aux bits, `with_config` arguments.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct GooeyVoicePatch {
    pub instrument: u32,
    pub aux: u32,
    pub params: [f32; 24],
}

pub const GOOEY_INSTRUMENT_KICK: u32 = 0;
pub const GOOEY_INSTRUMENT_SNARE: u32 = 1;
pub const GOOEY_INSTRUMENT_HIHAT: u32 = 2;
pub const GOOEY_INSTRUMENT_TOM: u32 = 3;
pub const GOOEY_INSTRUMENT_BASS: u32 = 4;

#[repr(C)]
pub struct GooeyRsBatch {
    _private: [u8; 0],
}
#[repr(C)]
pub struct GooeyVoiceBatch {
    _private: [u8; 0],
}

extern "C" {
    pub fn gooey_b200_last_error() -> *const c_char;
    pub fn gooey_b200_device_count() -> c_int;

    pub fn gooey_rs_batch_new(sample_rate: c_float, n_engines: u32, device: c_int, out: *mut *mut GooeyRsBatch) -> c_int;
    pub fn gooey_rs_batch_free(b: *mut GooeyRsBatch);
    pub fn gooey_rs_batch_add_instrument(b: *mut GooeyRsBatch, engine: u32, name: *const c_char, patch: *const GooeyVoicePatch) -> c_int;
    pub fn gooey_rs_batch_add_sequencer(
        b: *mut GooeyRsBatch, engine: u32, instrument_name: *const c_char, bpm: c_float, enabled: *const u8, velocity: *const c_float, steps: u32,
    ) -> c_int;
    pub fn gooey_rs_batch_set_bpm(b: *mut GooeyRsBatch, engine: u32, bpm: c_float) -> c_int;
    pub fn gooey_rs_batch_set_master_gain(b: *mut GooeyRsBatch, engine: u32, gain: c_float) -> c_int;
    pub fn gooey_rs_batch_clear_global_effects(b: *mut GooeyRsBatch, engine: u32) -> c_int;
    pub fn gooey_rs_batch_add_limiter(b: *mut GooeyRsBatch, engine: u32, threshold: c_float) -> c_int;
    pub fn gooey_rs_batch_add_effect(b: *mut GooeyRsBatch, engine: u32, effect_id: u32, args: *const c_float, n_args: u32) -> c_int;
    pub fn gooey_rs_batch_bounce(b: *mut GooeyRsBatch, samples: u32, out_host: *mut c_float) -> c_int;

    pub fn gooey_voice_batch_new(sample_rate: c_float, n: u32, patches: *const GooeyVoicePatch, device: c_int, out: *mut *mut GooeyVoiceBatch) -> c_int;
    pub fn gooey_voice_batch_free(b: *mut GooeyVoiceBatch);
    pub fn gooey_voice_batch_trigger(b: *mut GooeyVoiceBatch, voice: u32, frame: u32, velocity: c_float) -> c_int;
    pub fn gooey_voice_batch_set_param(b: *mut GooeyVoiceBatch, voice: u32, frame: u32, param: u32, value: c_float, snap: c_int) -> c_int;
    pub fn gooey_voice_batch_note_on(b: *mut GooeyVoiceBatch, voice: u32, frame: u32, note: u32, velocity: c_float) -> c_int;
    pub fn gooey_voice_batch_release(b: *mut GooeyVoiceBatch, voice: u32, frame: u32) -> c_int;
    pub fn gooey_voice_batch_set_buffer(b: *mut GooeyVoiceBatch, voice: u32, frame: u32, samples: *const c_float, len: u32, sample_rate: c_float) -> c_int;
    pub fn gooey_voice_batch_share_buffer(b: *mut GooeyVoiceBatch, dst_voice: u32, frame: u32, src_voice: u32) -> c_int;
    pub fn gooey_voice_batch_set_seed(b: *mut GooeyVoiceBatch, voice: u32, frame: u32, seed: u32) -> c_int;
    pub fn gooey_voice_batch_render(b: *mut GooeyVoiceBatch, frames: u32, out_host: *mut c_float) -> c_int;

    pub fn gooey_b200_write_wav(path: *const c_char, samples: *const c_float, n: u32, sample_rate: u32, bit_depth: u32) -> c_int;
    pub fn gooey_b200_write_wav_f32(path: *const c_char, interleaved: *const c_float, frames: u32, channels: u32, sample_rate: u32) -> c_int;
    pub fn gooey_voice_batch_render_pcm16(b: *mut GooeyVoiceBatch, frames: u32, out_host: *mut i16) -> c_int;

    // FFI engines (`include/gooey.h`): the handles are the reference's `*mut GooeyEngine`; these are the batch calls a host adds
    pub fn gooey_b200_set_device(device: c_int) -> c_int;
    pub fn gooey_batch_bounce(engines: *const *mut GooeyEngineOpaque, n: u32, bars: u32, out_buffers: *mut *mut c_float, out_lengths: *mut u32) -> c_int;
    pub fn gooey_batch_bounce_host(engines: *const *mut GooeyEngineOpaque, n: u32, bars: u32, out_host: *mut c_float, pitch: usize, out_frames: *mut u32) -> c_int;
    pub fn gooey_batch_bounce_pcm16(engines: *const *mut GooeyEngineOpaque, n: u32, bars: u32, out_host: *mut i16, pitch: usize, out_frames: *mut u32) -> c_int;
    pub fn gooey_batch_bounce_to_wav(engines: *const *mut GooeyEngineOpaque, n: u32, bars: u32, utf8_paths: *const *const c_char) -> c_int;
    pub fn gooey_batch_render(engines: *const *mut GooeyEngineOpaque, n: u32, frames: u32, out_host: *mut c_float) -> c_int;
    pub fn gooey_b200_host_alloc(bytes: usize, device: c_int, out_numa_node: *mut c_int) -> *mut std::ffi::c_void;
    pub fn gooey_b200_host_free(p: *mut std::ffi::c_void);

    // sample-playback sources: the reference's own names (`src/ffi.rs:6007-6168`, `:7184-7535`, `:8006-8048`); a host that already
    // binds libgooey's FFI needs no new declarations for them — listed here for the Rust-side batch host
    pub fn gooey_engine_loop_load(e: *mut GooeyEngineOpaque, channel: u32, samples: *const c_float, frames: u32, channels: u32, sample_rate: c_float) -> bool;
    pub fn gooey_engine_loop_set_playing(e: *mut GooeyEngineOpaque, channel: u32, playing: bool);
    pub fn gooey_engine_loop_set_gain(e: *mut GooeyEngineOpaque, channel: u32, gain: c_float);
    pub fn gooey_engine_loop_set_start(e: *mut GooeyEngineOpaque, channel: u32, normalized: c_float);
    pub fn gooey_engine_loop_set_end(e: *mut GooeyEngineOpaque, channel: u32, normalized: c_float);
    pub fn gooey_engine_loop_set_speed(e: *mut GooeyEngineOpaque, channel: u32, speed: c_float);
    pub fn gooey_engine_loop_set_source_bpm(e: *mut GooeyEngineOpaque, channel: u32, source_bpm: c_float);
    pub fn gooey_engine_loop_set_pitch_mode(e: *mut GooeyEngineOpaque, channel: u32, mode: u32);
    pub fn gooey_engine_loop_render_to_wav(e: *mut GooeyEngineOpaque, channel: u32, frame_count: u32, preroll_frame_count: u32, path: *const c_char) -> bool;
    pub fn gooey_b200_loop_share_buffer(dst: *mut GooeyEngineOpaque, dst_channel: u32, src: *const GooeyEngineOpaque, src_channel: u32) -> bool;
    pub fn gooey_engine_sampler_register(e: *mut GooeyEngineOpaque) -> i32;
    pub fn gooey_engine_sampler_set_slot_buffer(
        e: *mut GooeyEngineOpaque, rack: u32, slot: u32, samples: *const c_float, frames: u32, channels: u32, sample_rate: c_float,
    ) -> bool;
    pub fn gooey_engine_sampler_trigger(e: *mut GooeyEngineOpaque, rack: u32, slot: u32, velocity: c_float) -> bool;
}

/// Opaque `GooeyEngine` of `include/gooey.h` (the reference's handle type, `src/ffi.rs:670`).
#[repr(C)]
pub struct GooeyEngineOpaque {
    _private: [u8; 0],
}

/// `gooey_engine_bounce_to_wav` (ffi.rs:7942-7980) for a whole batch of FFI engines: one device pass, 16-bit PCM quantised on
/// the device, one mono WAV per engine.
///
/// # Safety
/// every pointer must be a live handle returned by `gooey_engine_new` of libgooey_b200.
pub unsafe fn batch_bounce_to_wav(engines: &[*mut GooeyEngineOpaque], bars: u32, paths: &[&str]) -> Result<(), String> {
    if engines.len() != paths.len() {
        return Err(String::from("one path per engine"));
    }
    let c: Vec<CString> = paths.iter().map(|p| cstr(p)).collect::<Result<_, _>>()?;
    let p: Vec<*const c_char> = c.iter().map(|s| s.as_ptr()).collect();
    check(gooey_batch_bounce_to_wav(engines.as_ptr(), engines.len() as u32, bars, p.as_ptr()))
}

/// The library's thread-local error text, as the `Err(String)` the reference's Rust API uses.
pub(crate) fn last_error() -> String {
    unsafe {
        let p = gooey_b200_last_error();
        if p.is_null() { String::from("libgooey_b200: unknown error") } else { CStr::from_ptr(p).to_string_lossy().into_owned() }
    }
}
pub(crate) fn check(rc: c_int) -> Result<(), String> {
    if rc == 0 { Ok(()) } else { Err(format!("libgooey_b200 error {rc}: {}", last_error())) }
}
pub(crate) fn cstr(s: &str) -> Result<CString, String> {
    CString::new(s).map_err(|_| String::from("name contains a NUL byte"))
}
