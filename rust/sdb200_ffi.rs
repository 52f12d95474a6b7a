//! Reference-side binding of libsdb200.so — SOURCE ONLY (no rustc/cargo in the build image; see DESIGN.md).
//!
//! Drop this file into the reference as `src/sdb200.rs`, add `pub mod sdb200;` to `src/lib.rs`, link with
//! `println!("cargo:rustc-link-lib=dylib=sdb200")` from a build script, and replace the three hot-path calls in
//! `src/bin/sample/main.rs:100-109`:
//!
//!   let images = sd.sample_image(context, unconditional_context, scale, n_steps);
//! becomes
//!   let sdb = sdb200::StableDiffusion::new(0)?;
//!   sdb.load_dump_dir(&model_name)?;          // in place of load_stable_diffusion(&model_name, &device)
//!   sdb.finalize_weights()?;
//!   let images = sdb.sample_image(&context_f32, [n, l], &uncond_f32, lu, scale, n_steps, None, 0)?;
//!
//! The signatures keep the reference's argument meaning (src/model/stablediffusion/mod.rs:51-57,
//! src/model/unet/mod.rs:109-114, src/model/autoencoder/mod.rs:68) with plain fp32 slices in place of
//! `Tensor<B, D>` (same contiguous row-major contents: NCHW / [n, L, 768]).

use std::ffi::{c_char, c_int, c_void, CStr, CString};

#[repr(C)]
pub struct SdbCtx {
    _private: [u8; 0],
}

/// The update rule of `StableDiffusion::sample_ex` (SDB_SAMPLER_* in include/sdb200.h). `Ddim { eta: 0.0 }` is the reference's.
#[derive(Clone, Copy, Debug)]
pub enum Sampler {
    /// DDIM with `eta` in [0, 1] (the `sigma` of src/model/stablediffusion/mod.rs:119, scaled by eta).
    Ddim { eta: f64 },
    /// DPM-Solver++(2M), data prediction, multistep.
    DpmPp2M,
}
const SDB_SAMPLER_DDIM: c_int = 0;
const SDB_SAMPLER_DPMPP_2M: c_int = 1;

extern "C" {
    fn sdb_create(device: c_int, out: *mut *mut SdbCtx) -> c_int;
    fn sdb_destroy(ctx: *mut SdbCtx) -> c_int;
    fn sdb_last_error(ctx: *mut SdbCtx) -> *const c_char;
    fn sdb_set_tensor(ctx: *mut SdbCtx, name: *const c_char, host: *const f32, dims: *const i64, ndim: c_int) -> c_int;
    fn sdb_load_dump_dir(ctx: *mut SdbCtx, path: *const c_char) -> c_int;
    fn sdb_finalize_weights(ctx: *mut SdbCtx) -> c_int;
    fn sdb_clip_forward(ctx: *mut SdbCtx, tokens: *const i32, n: c_int, l: c_int, out: *mut f32) -> c_int;
    fn sdb_encode_image(ctx: *mut SdbCtx, img: *const f32, n: c_int, h: c_int, w: c_int, latent: *mut f32) -> c_int;
    fn sdb_unet_forward(ctx: *mut SdbCtx, x: *const f32, timestep: i32, context: *const f32, n: c_int, h: c_int,
                        w: c_int, l: c_int, out: *mut f32) -> c_int;
    fn sdb_decode_latent(ctx: *mut SdbCtx, latent: *const f32, n: c_int, h: c_int, w: c_int, img: *mut f32) -> c_int;
    fn sdb_sample_image(ctx: *mut SdbCtx, context: *const f32, n: c_int, l: c_int, uncond: *const f32, lu: c_int,
                        guidance_scale: f64, n_steps: c_int, init_latent: *const f32, seed: u64, h: c_int, w: c_int,
                        rgb: *mut u8) -> c_int;
    fn sdb_sample_latent(ctx: *mut SdbCtx, context: *const f32, n: c_int, l: c_int, uncond: *const f32, lu: c_int,
                         guidance_scale: f64, n_steps: c_int, init_latent: *const f32, seed: u64, h: c_int, w: c_int,
                         latent_out: *mut f32) -> c_int;
    fn sdb_latent_to_image(ctx: *mut SdbCtx, latent: *const f32, n: c_int, h: c_int, w: c_int, rgb: *mut u8) -> c_int;
    fn sdb_forward_diffuser(ctx: *mut SdbCtx, latent: *const f32, timestep: i32, context: *const f32, n: c_int, l: c_int,
                            uncond: *const f32, lu: c_int, guidance_scale: f64, h: c_int, w: c_int, pred: *mut f32,
                            out_uncond: *mut f32, out_cond: *mut f32) -> c_int;
    fn sdb_img2img(ctx: *mut SdbCtx, rgb: *const u8, mask: *const u8, context: *const f32, n: c_int, l: c_int,
                   uncond: *const f32, lu: c_int, guidance_scale: f64, n_steps: c_int, strength: f64, noise: *const f32,
                   seed: u64, h: c_int, w: c_int, latent_out: *mut f32, rgb_out: *mut u8) -> c_int;
    #[allow(dead_code)]
    fn sdb_img2img_dev(ctx: *mut SdbCtx, d_rgb: *const c_void, d_mask: *const c_void, d_context: *const c_void, n: c_int,
                       l: c_int, d_uncond: *const c_void, lu: c_int, guidance_scale: f64, n_steps: c_int, strength: f64,
                       d_noise: *const c_void, seed: u64, h: c_int, w: c_int, d_latent_out: *mut c_void,
                       d_rgb_out: *mut c_void, stream: *mut c_void) -> c_int;
    fn sdb_sample_ex(ctx: *mut SdbCtx, context: *const f32, n: c_int, l: c_int, uncond: *const f32, lu: c_int,
                     guidance_scale: f64, n_steps: c_int, sampler: c_int, eta: f64, init_latent: *const f32,
                     step_noise: *const f32, seed: u64, h: c_int, w: c_int, latent_out: *mut f32, rgb_out: *mut u8) -> c_int;
    #[allow(dead_code)]
    fn sdb_sample_ex_dev(ctx: *mut SdbCtx, d_context: *const c_void, n: c_int, l: c_int, d_uncond: *const c_void, lu: c_int,
                         guidance_scale: f64, n_steps: c_int, sampler: c_int, eta: f64, d_init_latent: *const c_void,
                         d_step_noise: *const c_void, seed: u64, h: c_int, w: c_int, d_latent_out: *mut c_void,
                         d_rgb_out: *mut c_void, stream: *mut c_void) -> c_int;
    #[allow(dead_code)]
    fn sdb_randn(ctx: *mut SdbCtx, seed: u64, count: i64, out: *mut f32) -> c_int;
    fn sdb_nccl_unique_id(id128: *mut c_void) -> c_int;
    fn sdb_broadcast_weights(ctx: *mut SdbCtx, id128: *const c_void, rank: c_int, world: c_int) -> c_int;
    #[allow(dead_code)]
    fn sdb_sample_image_dev(ctx: *mut SdbCtx, d_context: *const c_void, n: c_int, l: c_int, d_uncond: *const c_void,
                            lu: c_int, guidance_scale: f64, n_steps: c_int, d_init_latent: *const c_void, h: c_int,
                            w: c_int, d_rgb: *mut c_void, stream: *mut c_void) -> c_int;
}

#[derive(Debug)]
pub struct SdbError(pub String);

pub struct StableDiffusion {
    ctx: *mut SdbCtx,
}

impl StableDiffusion {
    /// Replaces `StableDiffusionConfig::new().init(&device)` (src/model/stablediffusion/mod.rs:22-39).
    pub fn new(device: i32) -> Result<Self, SdbError> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { sdb_create(device, &mut ctx) };
        if rc != 0 {
            return Err(SdbError(unsafe { CStr::from_ptr(sdb_last_error(std::ptr::null_mut())) }.to_string_lossy().into()));
        }
        Ok(Self { ctx })
    }

    fn check(&self, rc: c_int) -> Result<(), SdbError> {
        if rc == 0 {
            Ok(())
        } else {
            Err(SdbError(unsafe { CStr::from_ptr(sdb_last_error(self.ctx)) }.to_string_lossy().into()))
        }
    }

    /// Replaces `load_tensor` + `Param::from_tensor` (src/model/load.rs:30-47): `name` is the dump-dir path
    /// without the `.npy` suffix, e.g. "unet/input_blocks/rt1/res/conv_in/weight".
    pub fn set_tensor(&self, name: &str, data: &[f32], dims: &[i64]) -> Result<(), SdbError> {
        let cname = CString::new(name).unwrap();
        self.check(unsafe { sdb_set_tensor(self.ctx, cname.as_ptr(), data.as_ptr(), dims.as_ptr(), dims.len() as c_int) })
    }

    /// Replaces `load_stable_diffusion(path, device)` (src/model/stablediffusion/load.rs:16-33): reads the dump-dir tree.
    pub fn load_dump_dir(&self, path: &str) -> Result<(), SdbError> {
        let cpath = CString::new(path).unwrap();
        self.check(unsafe { sdb_load_dump_dir(self.ctx, cpath.as_ptr()) })
    }

    pub fn finalize_weights(&self) -> Result<(), SdbError> {
        self.check(unsafe { sdb_finalize_weights(self.ctx) })
    }

    /// `Autoencoder::encode_image(x)` (src/model/autoencoder/mod.rs:60-66): [n, 3, h, w] -> [n, 4, h/8, w/8].
    pub fn encode_image(&self, img: &[f32], [n, h, w]: [usize; 3]) -> Result<Vec<f32>, SdbError> {
        let mut latent = vec![0f32; n * 4 * (h / 8) * (w / 8)];
        self.check(unsafe { sdb_encode_image(self.ctx, img.as_ptr(), n as c_int, h as c_int, w as c_int, latent.as_mut_ptr()) })?;
        Ok(latent)
    }

    /// `CLIP::forward(tokens)` (src/model/clip/mod.rs:56-75): ids [n, l] (l <= 77, unpadded) -> [n, l, 768].
    pub fn clip_forward(&self, tokens: &[i32], [n, l]: [usize; 2]) -> Result<Vec<f32>, SdbError> {
        let mut out = vec![0f32; n * l * 768];
        self.check(unsafe { sdb_clip_forward(self.ctx, tokens.as_ptr(), n as c_int, l as c_int, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `UNet::forward(x, timesteps, context)` (src/model/unet/mod.rs:109-114).
    pub fn unet_forward(&self, x: &[f32], [n, h, w]: [usize; 3], timestep: i32, context: &[f32], l: usize) -> Result<Vec<f32>, SdbError> {
        let mut out = vec![0f32; n * 4 * h * w];
        self.check(unsafe {
            sdb_unet_forward(self.ctx, x.as_ptr(), timestep, context.as_ptr(), n as c_int, h as c_int, w as c_int, l as c_int, out.as_mut_ptr())
        })?;
        Ok(out)
    }

    /// `Autoencoder::decode_latent(latent)` (src/model/autoencoder/mod.rs:68-71).
    pub fn decode_latent(&self, latent: &[f32], [n, h, w]: [usize; 3]) -> Result<Vec<f32>, SdbError> {
        let mut img = vec![0f32; n * 3 * 64 * h * w];
        self.check(unsafe { sdb_decode_latent(self.ctx, latent.as_ptr(), n as c_int, h as c_int, w as c_int, img.as_mut_ptr()) })?;
        Ok(img)
    }

    /// `StableDiffusion::sample_image(context, unconditional_context, scale, n_steps) -> Vec<Vec<u8>>`
    /// (src/model/stablediffusion/mod.rs:51-67). `init_latent = None` draws N(0,1) on the device from `seed`.
    #[allow(clippy::too_many_arguments)]
    pub fn sample_image(&self, context: &[f32], [n, l]: [usize; 2], unconditional_context: &[f32], lu: usize,
                        unconditional_guidance_scale: f64, n_steps: usize, init_latent: Option<&[f32]>, seed: u64)
                        -> Result<Vec<Vec<u8>>, SdbError> {
        let (h, w) = (64usize, 64usize); // the reference hard-codes 512x512 (stablediffusion/mod.rs:74-75,116)
        let mut rgb = vec![0u8; n * 8 * h * 8 * w * 3];
        self.check(unsafe {
            sdb_sample_image(self.ctx, context.as_ptr(), n as c_int, l as c_int, unconditional_context.as_ptr(), lu as c_int,
                             unconditional_guidance_scale, n_steps as c_int,
                             init_latent.map_or(std::ptr::null(), |s| s.as_ptr()), seed, h as c_int, w as c_int, rgb.as_mut_ptr())
        })?;
        Ok(rgb.chunks(8 * h * 8 * w * 3).map(|c| c.to_vec()).collect())
    }
}

impl StableDiffusion {
    /// `StableDiffusion::sample_latent(context, unconditional_context, scale, n_steps) -> Tensor<B, 4>`
    /// (src/model/stablediffusion/mod.rs:102-160); returns the final latent [n, 4, 64, 64].
    #[allow(clippy::too_many_arguments)]
    pub fn sample_latent(&self, context: &[f32], [n, l]: [usize; 2], unconditional_context: &[f32], lu: usize,
                         unconditional_guidance_scale: f64, n_steps: usize, init_latent: Option<&[f32]>, seed: u64)
                         -> Result<Vec<f32>, SdbError> {
        let (h, w) = (64usize, 64usize);
        let mut latent = vec![0f32; n * 4 * h * w];
        self.check(unsafe {
            sdb_sample_latent(self.ctx, context.as_ptr(), n as c_int, l as c_int, unconditional_context.as_ptr(), lu as c_int,
                              unconditional_guidance_scale, n_steps as c_int,
                              init_latent.map_or(std::ptr::null(), |s| s.as_ptr()), seed, h as c_int, w as c_int, latent.as_mut_ptr())
        })?;
        Ok(latent)
    }

    /// `StableDiffusion::latent_to_image(latent) -> Vec<Vec<u8>>` (src/model/stablediffusion/mod.rs:69-100).
    pub fn latent_to_image(&self, latent: &[f32], [n, h, w]: [usize; 3]) -> Result<Vec<Vec<u8>>, SdbError> {
        let mut rgb = vec![0u8; n * 8 * h * 8 * w * 3];
        self.check(unsafe { sdb_latent_to_image(self.ctx, latent.as_ptr(), n as c_int, h as c_int, w as c_int, rgb.as_mut_ptr()) })?;
        Ok(rgb.chunks(8 * h * 8 * w * 3).map(|c| c.to_vec()).collect())
    }

    /// `forward_diffuser(latent, timestep, context, unconditional_context, scale)` (src/model/stablediffusion/mod.rs:162-192):
    /// the guided noise prediction of one step.
    #[allow(clippy::too_many_arguments)]
    pub fn forward_diffuser(&self, latent: &[f32], [n, h, w]: [usize; 3], timestep: i32, context: &[f32], l: usize,
                            unconditional_context: &[f32], lu: usize, unconditional_guidance_scale: f64) -> Result<Vec<f32>, SdbError> {
        let mut pred = vec![0f32; n * 4 * h * w];
        self.check(unsafe {
            sdb_forward_diffuser(self.ctx, latent.as_ptr(), timestep, context.as_ptr(), n as c_int, l as c_int,
                                 unconditional_context.as_ptr(), lu as c_int, unconditional_guidance_scale, h as c_int, w as c_int,
                                 pred.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut())
        })?;
        Ok(pred)
    }

    /// img2img (SDEdit) and, with `mask`, latent-blend inpainting on the sample_latent sampler (DESIGN.md §7 row f5; the reference
    /// has no img2img). `rgb` is [n, 8h, 8w, 3] u8 like the images sample_image returns, `mask` [n, 8h, 8w] (nonzero = repaint),
    /// `strength` in [0, 1] the share of the n_steps schedule that runs, `noise = None` draws N(0,1) on the device from `seed`.
    #[allow(clippy::too_many_arguments)]
    pub fn img2img(&self, rgb: &[u8], [n, h, w]: [usize; 3], mask: Option<&[u8]>, context: &[f32], l: usize,
                   unconditional_context: &[f32], lu: usize, unconditional_guidance_scale: f64, n_steps: usize, strength: f64,
                   noise: Option<&[f32]>, seed: u64) -> Result<Vec<Vec<u8>>, SdbError> {
        let mut out = vec![0u8; n * 8 * h * 8 * w * 3];
        self.check(unsafe {
            sdb_img2img(self.ctx, rgb.as_ptr(), mask.map_or(std::ptr::null(), |s| s.as_ptr()), context.as_ptr(), n as c_int,
                        l as c_int, unconditional_context.as_ptr(), lu as c_int, unconditional_guidance_scale, n_steps as c_int,
                        strength, noise.map_or(std::ptr::null(), |s| s.as_ptr()), seed, h as c_int, w as c_int,
                        std::ptr::null_mut(), out.as_mut_ptr())
        })?;
        Ok(out.chunks(8 * h * 8 * w * 3).map(|c| c.to_vec()).collect())
    }

    /// `sample_image` with a selectable sampler (DESIGN.md §7 row f6; the reference's only sampler is `Sampler::Ddim { eta: 0.0 }`,
    /// src/model/stablediffusion/mod.rs:119). `step_noise` ([T, n, 4, 64, 64], DDIM with eta > 0 only) or `None`: step i draws
    /// from the device stream keyed by `seed ^ ((i + 1) * 0x9E3779B97F4A7C15)`.
    #[allow(clippy::too_many_arguments)]
    pub fn sample_ex(&self, context: &[f32], [n, l]: [usize; 2], unconditional_context: &[f32], lu: usize,
                     unconditional_guidance_scale: f64, n_steps: usize, sampler: Sampler, init_latent: Option<&[f32]>,
                     step_noise: Option<&[f32]>, seed: u64) -> Result<Vec<Vec<u8>>, SdbError> {
        let (h, w) = (64usize, 64usize);
        let (id, eta) = match sampler {
            Sampler::Ddim { eta } => (SDB_SAMPLER_DDIM, eta),
            Sampler::DpmPp2M => (SDB_SAMPLER_DPMPP_2M, 0.0),
        };
        let mut rgb = vec![0u8; n * 8 * h * 8 * w * 3];
        self.check(unsafe {
            sdb_sample_ex(self.ctx, context.as_ptr(), n as c_int, l as c_int, unconditional_context.as_ptr(), lu as c_int,
                          unconditional_guidance_scale, n_steps as c_int, id, eta,
                          init_latent.map_or(std::ptr::null(), |s| s.as_ptr()), step_noise.map_or(std::ptr::null(), |s| s.as_ptr()),
                          seed, h as c_int, w as c_int, std::ptr::null_mut(), rgb.as_mut_ptr())
        })?;
        Ok(rgb.chunks(8 * h * 8 * w * 3).map(|c| c.to_vec()).collect())
    }

    /// Multi-GPU init: rank 0 calls `nccl_unique_id()` and ships the 128 bytes to the other ranks by any means; every rank then
    /// calls `broadcast_weights(&id, rank, world)` (one ncclBroadcast of the weight arena from rank 0) and `finalize_weights()`.
    pub fn nccl_unique_id() -> Result<[u8; 128], SdbError> {
        let mut id = [0u8; 128];
        if unsafe { sdb_nccl_unique_id(id.as_mut_ptr() as *mut c_void) } != 0 {
            return Err(SdbError("ncclGetUniqueId failed".into()));
        }
        Ok(id)
    }
    pub fn broadcast_weights(&self, id: &[u8; 128], rank: usize, world: usize) -> Result<(), SdbError> {
        self.check(unsafe { sdb_broadcast_weights(self.ctx, id.as_ptr() as *const c_void, rank as c_int, world as c_int) })
    }
}

impl Drop for StableDiffusion {
    fn drop(&mut self) {
        unsafe { sdb_destroy(self.ctx) };
    }
}
