//! `gooey::bounce` for batches (reference `src/bounce.rs:9-133`): same `BounceLength`, `WavConfig` and function names;
//! the engine argument is a description (`EngineSpec`) instead of a live `Engine`, because the audio state lives on the GPU.

use crate::*;
use std::path::Path;

/// Identical to the reference's enum (bounce.rs:9-16).
pub enum BounceLength {
    Bars(usize),
    Beats(f64),
    Samples(usize),
}

impl BounceLength {
    /// bounce.rs:20-32 — f64 arithmetic, `round` half away from zero.
    pub fn to_samples(&self, bpm: f32, sample_rate: f32) -> usize {
        match self {
            BounceLength::Bars(bars) => (*bars as f64 * (4.0 * (60.0 / bpm as f64) * sample_rate as f64)).round() as usize,
            BounceLength::Beats(beats) => (beats * ((60.0 / bpm as f64) * sample_rate as f64)).round() as usize,
            BounceLength::Samples(n) => *n,
        }
    }
}

/// bounce.rs:62-74.
pub struct WavConfig {
    pub bit_depth: u16,
}
impl Default for WavConfig {
    fn default() -> Self {
        Self { bit_depth: 16 }
    }
}

/// One sequencer: `Sequencer::with_velocity_pattern(bpm, sr, steps, instrument_name)` (sequencer.rs:556-582).
pub struct SequencerSpec {
    pub bpm: f32,
    pub instrument_name: String,
    pub steps: Vec<(bool, f32)>,
}

/// What `Engine::new` + `add_instrument` + `add_sequencer` + `set_master_gain` + the global effect chain describe.
pub struct EngineSpec {
    pub bpm: f32,
    pub instruments: Vec<(String, GooeyVoicePatch)>,
    pub sequencers: Vec<SequencerSpec>,
    pub master_gain: f32,
    /// the global chain in order; `Engine::new` starts with `[SoftLimiter(1.0)]`
    pub global_effects: Vec<GlobalEffect>,
}

impl EngineSpec {
    pub fn new() -> Self {
        Self { bpm: 120.0, instruments: Vec::new(), sequencers: Vec::new(), master_gain: 0.25, global_effects: vec![GlobalEffect::SoftLimiter(1.0)] }
    }
}

/// One global effect, by its reference type and constructor arguments after the sample rate (the device builds it at
/// the batch's sample rate).  `DelayEffect`'s first argument is the `DelayTiming` index (3 = eighth).
#[derive(Clone, Copy, Debug)]
pub enum GlobalEffect {
    LowpassFilterEffect { cutoff: f32, resonance: f32 },
    DelayEffect { timing: u32, bpm: f32, feedback: f32, mix: f32, cutoff: f32 },
    TubeSaturation { drive: f32, warmth: f32, mix: f32 },
    TubeCompressor { threshold_db: f32, ratio: f32, attack_ms: f32, release_ms: f32, mix: f32 },
    TiltFilterEffect,
    SoftLimiter(f32),
    SpringReverbEffect { decay: f32, mix: f32, damping: f32 },
    Waveshaper { drive: f32, mix: f32 },
    FeedbackWaveshaper { drive: f32, feedback: f32, cutoff: f32, mix: f32 },
    PlateReverbEffect { decay: f32, mix: f32, damping: f32 },
}

impl GlobalEffect {
    /// (FFI effect id, constructor arguments) as `gooey_rs_batch_add_effect` takes them
    fn ffi(&self) -> (u32, Vec<f32>) {
        use GlobalEffect::*;
        match *self {
            LowpassFilterEffect { cutoff, resonance } => (0, vec![cutoff, resonance]),
            DelayEffect { timing, bpm, feedback, mix, cutoff } => (1, vec![timing as f32, bpm, feedback, mix, cutoff]),
            TubeSaturation { drive, warmth, mix } => (2, vec![drive, warmth, mix]),
            TubeCompressor { threshold_db, ratio, attack_ms, release_ms, mix } => (3, vec![threshold_db, ratio, attack_ms, release_ms, mix]),
            TiltFilterEffect => (4, vec![]),
            SoftLimiter(threshold) => (5, vec![threshold]),
            SpringReverbEffect { decay, mix, damping } => (6, vec![decay, mix, damping]),
            Waveshaper { drive, mix } => (7, vec![drive, mix]),
            FeedbackWaveshaper { drive, feedback, cutoff, mix } => (8, vec![drive, feedback, cutoff, mix]),
            PlateReverbEffect { decay, mix, damping } => (9, vec![decay, mix, damping]),
        }
    }
}

/// A device-resident batch of engines.  Voice state persists across bounces, as it does in the reference.
pub struct EngineBatch {
    raw: *mut GooeyRsBatch,
    sample_rate: f32,
    bpm: Vec<f32>,
}

impl EngineBatch {
    pub fn new(sample_rate: f32, specs: &[EngineSpec], device: i32) -> Result<Self, String> {
        let mut raw = std::ptr::null_mut();
        check(unsafe { gooey_rs_batch_new(sample_rate, specs.len() as u32, device, &mut raw) })?;
        let batch = EngineBatch { raw, sample_rate, bpm: specs.iter().map(|s| s.bpm).collect() };
        for (i, s) in specs.iter().enumerate() {
            let e = i as u32;
            check(unsafe { gooey_rs_batch_set_bpm(raw, e, s.bpm) })?;
            for (name, patch) in &s.instruments {
                let n = cstr(name)?;
                check(unsafe { gooey_rs_batch_add_instrument(raw, e, n.as_ptr(), patch) })?;
            }
            for q in &s.sequencers {
                let n = cstr(&q.instrument_name)?;
                let en: Vec<u8> = q.steps.iter().map(|p| p.0 as u8).collect();
                let ve: Vec<f32> = q.steps.iter().map(|p| p.1).collect();
                check(unsafe { gooey_rs_batch_add_sequencer(raw, e, n.as_ptr(), q.bpm, en.as_ptr(), ve.as_ptr(), en.len() as u32) })?;
            }
            check(unsafe { gooey_rs_batch_set_master_gain(raw, e, s.master_gain) })?;
            check(unsafe { gooey_rs_batch_clear_global_effects(raw, e) })?;
            for fx in &s.global_effects {
                let (id, args) = fx.ffi();
                check(unsafe { gooey_rs_batch_add_effect(raw, e, id, args.as_ptr(), args.len() as u32) })?;
            }
        }
        Ok(batch)
    }

    /// `bounce_to_buffer` of every engine in one device pass.  Engines must resolve `length` to one sample count.
    pub fn bounce_to_buffers(&mut self, length: &BounceLength) -> Result<Vec<Vec<f32>>, String> {
        let n = self.bpm.len();
        if n == 0 {
            return Ok(Vec::new());
        }
        let total = length.to_samples(self.bpm[0], self.sample_rate);
        if self.bpm.iter().any(|b| length.to_samples(*b, self.sample_rate) != total) {
            return Err(String::from("engines of one batch bounce must have equal length; group them by tempo"));
        }
        let mut flat = vec![0.0f32; n * total];
        if total > 0 {
            check(unsafe { gooey_rs_batch_bounce(self.raw, total as u32, flat.as_mut_ptr()) })?;
        }
        Ok((0..n).map(|i| flat[i * total..(i + 1) * total].to_vec()).collect())
    }
}

impl Drop for EngineBatch {
    fn drop(&mut self) {
        unsafe { gooey_rs_batch_free(self.raw) }
    }
}

/// Single-engine convenience with the reference's name: a batch of one.
pub fn bounce_to_buffer(spec: &EngineSpec, sample_rate: f32, length: BounceLength) -> Result<Vec<f32>, String> {
    let mut b = EngineBatch::new(sample_rate, std::slice::from_ref(spec), 0)?;
    Ok(b.bounce_to_buffers(&length)?.pop().unwrap_or_default())
}

/// bounce.rs:80-133 — mono 16/24-bit PCM, `(s * scale).round()`.
pub fn bounce_to_wav(spec: &EngineSpec, sample_rate: f32, length: BounceLength, path: &Path, config: WavConfig) -> Result<(), String> {
    if config.bit_depth != 16 && config.bit_depth != 24 {
        return Err(format!("Unsupported bit depth: {}. Use 16 or 24.", config.bit_depth));
    }
    let buffer = bounce_to_buffer(spec, sample_rate, length)?;
    let p = cstr(path.to_str().ok_or_else(|| String::from("path is not UTF-8"))?)?;
    check(unsafe { gooey_b200_write_wav(p.as_ptr(), buffer.as_ptr(), buffer.len() as u32, sample_rate as u32, config.bit_depth as u32) })
}
