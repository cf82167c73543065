//! Safe Rust host layer over `libgl_commit` (C ABI in `include/gl_commit.h`): the B200 commitment path behind plonky2's own
//! items.  This is what a plonky2 fork at rev 3de92d9 (the reference's pinned dependency, `/root/reference/Cargo.toml:15-19`)
//! calls from the bodies of
//!
//! * `plonky2/src/fri/oracle.rs`   · `PolynomialBatch::from_values / from_coeffs / get_lde_values / prove_openings`
//! * `plonky2/src/hash/merkle_tree.rs` · `MerkleTree::new / get / prove`
//! * `plonky2/src/fri/prover.rs`   · `fri_committed_trees / fri_proof_of_work / fri_prover_query_rounds`
//!
//! (driven by the reference at `src/p3/mod.rs:250` `builder.build::<C>()` and `:260` `data.prove(pw)`; the replacement bodies
//! are in INTEGRATION.md §3).  Field elements cross the boundary as `u64` words (`GoldilocksField` is
//! `#[repr(transparent)] struct(pub u64)`), extension elements as `[u64; 2]`.
//!
//! Error behaviour: upstream functions are infallible and `assert!`-panic on misuse.  Every wrapper returns `Result<_, Error>`;
//! `Error::Invalid` carries the upstream assert text, and `.expect_upstream()` turns it into the same panic.  There is no CPU
//! fallback: `Context::new` fails without a CUDA device.
//!
//! NOT COMPILED in this repository's image (no cargo/rustc).  The same ABI is exercised on the GPU by the C++ mirror
//! (`include/gl_plonky2.hpp`, `tests/cpp/host_mirror_test.cpp`) and the Python mirror (`plonky2.5_b200/api.py`).

pub mod ffi;

use std::ffi::CStr;
use std::os::raw::c_int;
use std::ptr;

pub type Ext = [u64; 2];
pub type HashOut = [u64; 4];

#[derive(Debug, Clone, PartialEq, Eq)]
pub enum Error {
    /// an upstream `assert!` would have fired (message = upstream text)
    Invalid(String),
    /// CUDA runtime error / no device
    Cuda(String),
    OutOfMemory(String),
    UnknownHandle(String),
    Unsupported(String),
}

impl std::fmt::Display for Error {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        match self {
            Error::Invalid(m) | Error::Cuda(m) | Error::OutOfMemory(m) | Error::UnknownHandle(m) | Error::Unsupported(m) => f.write_str(m),
        }
    }
}
impl std::error::Error for Error {}

pub trait ExpectUpstream<T> {
    /// upstream is infallible: panic with the upstream message, as `assert!` would
    fn expect_upstream(self) -> T;
}
impl<T> ExpectUpstream<T> for Result<T, Error> {
    fn expect_upstream(self) -> T {
        match self {
            Ok(v) => v,
            Err(e) => panic!("{e}"),
        }
    }
}

/// One CUDA device + stream + cached twiddle tables (`gl_ctx`).  Calls on one context are serialised by the library; use one
/// per prover thread (`Context::with_thread_default`), as `cargo test` proves from several threads at once.
pub struct Context {
    raw: *mut ffi::gl_ctx,
}
// the library takes the context's mutex on every call
// Send only: one context per prover thread is the intended use (every call serialises on the context's mutex anyway).
unsafe impl Send for Context {}

impl Context {
    pub fn new(device: i32) -> Result<Self, Error> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { ffi::gl_ctx_create(&mut raw, device as c_int) };
        if rc != ffi::GL_OK {
            let what = unsafe { CStr::from_ptr(ffi::gl_strerror(rc)) }.to_string_lossy().into_owned();
            return Err(Error::Cuda(format!("gl_ctx_create(device={device}) failed: {what} (libgl_commit has no CPU fallback)")));
        }
        Ok(Self { raw })
    }

    /// the calling thread's own context on device 0 (created on first use)
    pub fn with_thread_default<R>(f: impl FnOnce(&Context) -> R) -> R {
        thread_local! { static CTX: Context = Context::new(0).expect("no CUDA device: libgl_commit has no CPU path"); }
        CTX.with(|c| f(c))
    }

    fn check(&self, rc: c_int) -> Result<(), Error> {
        if rc == ffi::GL_OK {
            return Ok(());
        }
        let what = unsafe { CStr::from_ptr(ffi::gl_strerror(rc)) }.to_string_lossy();
        let msg = unsafe { CStr::from_ptr(ffi::gl_ctx_last_error(self.raw)) }.to_string_lossy();
        let text = format!("{what}: {msg}");
        Err(match rc {
            ffi::GL_ERR_INVALID => Error::Invalid(text),
            ffi::GL_ERR_OOM => Error::OutOfMemory(text),
            ffi::GL_ERR_HANDLE => Error::UnknownHandle(text),
            ffi::GL_ERR_UNSUPPORTED => Error::Unsupported(text),
            _ => Error::Cuda(text),
        })
    }

    /// `PoseidonPermutation::permute` on `states.len() / 12` states, in place (used by the host-side `Challenger`)
    pub fn poseidon_permute(&self, states: &mut [u64]) -> Result<(), Error> {
        assert!(states.len() % 12 == 0, "states must be a multiple of the sponge width");
        self.check(unsafe { ffi::gl_poseidon_permute(self.raw, states.as_mut_ptr(), (states.len() / 12) as u64) })
    }

    /// `PolynomialBatch::from_values` (`input_is_coeffs = false`) / `from_coeffs` (`true`): `cols[j]` is column j, all of length
    /// 2^log_n.  The batch (coefficients, LDE leaves, digests) stays in HBM behind the returned `DeviceTree`; only the cap comes back.
    pub fn commit(&self, cols: &[&[u64]], rate_bits: usize, cap_height: usize, input_is_coeffs: bool) -> Result<DeviceTree<'_>, Error> {
        let n = cols.first().map(|c| c.len()).ok_or_else(|| Error::Invalid("empty polynomial batch".into()))?;
        if cols.iter().any(|c| c.len() != n) {
            return Err(Error::Invalid("Polynomial degrees inconsistent".into()));
        }
        if n == 0 || !n.is_power_of_two() {
            return Err(Error::Invalid("polynomial length must be a power of two".into()));
        }
        if cap_height > n.trailing_zeros() as usize + rate_bits {
            // upstream's assert, checked before the cap is sized by 2^cap_height
            return Err(Error::Invalid(format!("cap_height={cap_height} should be at most log2(leaves.len())")));
        }
        let ptrs: Vec<*const u64> = cols.iter().map(|c| c.as_ptr()).collect();
        let mut cap = vec![[0u64; 4]; 1 << cap_height];
        let mut handle: ffi::gl_handle = 0;
        self.check(unsafe {
            ffi::gl_commit(
                self.raw,
                ptrs.as_ptr(),
                cols.len() as u32,
                n.trailing_zeros(),
                rate_bits as u32,
                cap_height as u32,
                input_is_coeffs as c_int,
                ptr::null_mut(),
                ptr::null_mut(),
                ptr::null_mut(),
                cap.as_mut_ptr() as *mut u64,
                &mut handle,
            )
        })?;
        DeviceTree::adopt(self, handle, cap)
    }

    /// `MerkleTree::new(leaves, cap_height)` over packed row-major leaves `[n_leaves][leaf_len]`
    pub fn merkle_new(&self, leaves: &[u64], leaf_len: usize, cap_height: usize) -> Result<DeviceTree<'_>, Error> {
        if leaf_len == 0 || leaves.len() % leaf_len != 0 {
            return Err(Error::Invalid("leaves must be n_leaves * leaf_len words".into()));
        }
        let n_leaves = leaves.len() / leaf_len;
        if cap_height >= 64 || n_leaves == 0 || (1usize << cap_height) > n_leaves {
            // upstream's assert, checked before the cap is sized by 2^cap_height
            return Err(Error::Invalid(format!("cap_height={cap_height} should be at most log2(leaves.len())")));
        }
        let mut cap = vec![[0u64; 4]; 1 << cap_height];
        let mut handle: ffi::gl_handle = 0;
        self.check(unsafe {
            ffi::gl_merkle_new(
                self.raw,
                leaves.as_ptr(),
                (leaves.len() / leaf_len) as u64,
                leaf_len as u32,
                cap_height as u32,
                ptr::null_mut(),
                cap.as_mut_ptr() as *mut u64,
                &mut handle,
            )
        })?;
        DeviceTree::adopt(self, handle, cap)
    }

    /// `fri_proof_of_work`: the SMALLEST witness for the challenger state (`sponge_state`, pending `input_buffer`), i.e. what the
    /// serial `find` of the reference build returns.  The caller then observes it and draws the response as upstream does.
    pub fn fri_pow(&self, sponge_state: &[u64; 12], input_buffer: &[u64], min_leading_zeros: u32) -> Result<u64, Error> {
        assert!(input_buffer.len() < 8, "a full input buffer would already have been absorbed");
        let mut w = 0u64;
        let buf = if input_buffer.is_empty() { ptr::null() } else { input_buffer.as_ptr() };
        self.check(unsafe { ffi::gl_fri_pow(self.raw, sponge_state.as_ptr(), buf, input_buffer.len() as u32, min_leading_zeros, &mut w) })?;
        Ok(w)
    }

    /// `fri_committed_trees` state from host arrays: `values = coeffs.coset_fft(7)` in natural order, as upstream passes them
    pub fn fri_begin(&self, coeffs: &[Ext], values: &[Ext], rate_bits: usize, cap_height: usize) -> Result<FriState<'_>, Error> {
        if coeffs.len() != values.len() || coeffs.is_empty() {
            return Err(Error::Invalid("coeffs and values must have the same length".into()));
        }
        let mut h: ffi::gl_handle = 0;
        self.check(unsafe {
            ffi::gl_fri_begin(self.raw, coeffs.as_ptr() as *const u64, values.as_ptr() as *const u64, coeffs.len() as u64, rate_bits as u32, cap_height as u32, &mut h)
        })?;
        Ok(FriState { ctx: self, handle: h, cap_height })
    }

    /// `prove_openings`, front half: start accumulating `final_poly` over batches of degree 2^log_n
    /// `Gate::eval_unfiltered_base_batch` on host rows (`rows.len() = n * num_wires`): every constraint value, uncombined.
    /// `kind` is one of the gate constants of `ffi` (`ffi::GL_GATE_POSEIDON2`, `ffi::GL_GATE_U32_ARITHMETIC`, ...: the reference's Poseidon2Gate and u32 / b32 gates), `param` as documented in the header.
    pub fn evaluate_gate_constraints(&self, kind: i32, param: u32, rows: &[u64]) -> Result<Vec<u64>, Error> {
        let (nw, nc) = unsafe { (ffi::gl_gate_num_wires(kind as c_int, param), ffi::gl_gate_num_constraints(kind as c_int, param)) };
        if nw <= 0 || nc <= 0 || rows.len() % nw as usize != 0 {
            return Err(Error::Invalid("unknown gate kind / parameter, or rows is not n * num_wires words".into()));
        }
        let n = rows.len() / nw as usize;
        let mut out = vec![0u64; n * nc as usize];
        self.check(unsafe { ffi::gl_gate_eval_rows(self.raw, kind as c_int, param, rows.as_ptr(), n as u64, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// the gate part of `plonk/prover.rs · compute_quotient_polys` over the resident LDE rows of the wires commit
    pub fn quotient_begin<'c>(&'c self, wires: &DeviceTree<'c>, num_challenges: usize) -> Result<Quotient<'c>, Error> {
        let mut h: ffi::gl_handle = 0;
        self.check(unsafe { ffi::gl_quotient_begin(self.raw, wires.handle, num_challenges as u32, &mut h) })?;
        Ok(Quotient { ctx: self, handle: h, num_challenges })
    }

    /// `plonk/prover.rs · all_wires_permutation_partial_products` in `prove()`'s column order (the Z of every challenge first);
    /// returns `num_challenges * ceil(n_routed / degree)` columns of `N` values, flattened.
    pub fn partial_products_and_zs(&self, wires: &[&[u64]], sigmas: &[&[u64]], k_is: &[u64], betas: &[u64], gammas: &[u64],
                                   degree: usize) -> Result<Vec<u64>, Error> {
        let n = wires.first().map(|c| c.len()).ok_or_else(|| Error::Invalid("no routed wires".into()))?;
        if !n.is_power_of_two() || wires.len() != sigmas.len() || wires.len() != k_is.len() || betas.len() != gammas.len() || betas.is_empty()
            || degree == 0 || wires.iter().chain(sigmas.iter()).any(|c| c.len() != n)
        {
            return Err(Error::Invalid("partial_products_and_zs: inconsistent shapes".into()));
        }
        let wp: Vec<*const u64> = wires.iter().map(|c| c.as_ptr()).collect();
        let sp: Vec<*const u64> = sigmas.iter().map(|c| c.as_ptr()).collect();
        let n_chunks = (wires.len() + degree - 1) / degree;
        let mut out = vec![0u64; betas.len() * n_chunks * n];
        self.check(unsafe {
            ffi::gl_partial_products(self.raw, wp.as_ptr(), sp.as_ptr(), wires.len() as u32, n.trailing_zeros(), k_is.as_ptr(), betas.as_ptr(),
                                     gammas.as_ptr(), betas.len() as u32, degree as u32, out.as_mut_ptr())
        })?;
        Ok(out)
    }

    /// `Poseidon2Generator::run_once` for `inputs.len() / 13` gate rows (12 state inputs + swap flag each) -> 135 wires per row
    pub fn poseidon2_gate_witness(&self, inputs: &[u64]) -> Result<Vec<u64>, Error> {
        if inputs.len() % 13 != 0 {
            return Err(Error::Invalid("inputs must be n * 13 words".into()));
        }
        let n = inputs.len() / 13;
        let mut out = vec![0u64; n * 135];
        self.check(unsafe { ffi::gl_poseidon2_gate_witness(self.raw, inputs.as_ptr(), n as u64, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// plonky2 `gates/poseidon.rs · PoseidonGenerator::run_once` for `inputs.len() / 13` PoseidonGate rows (12 state inputs + swap flag
    /// each) -> 135 wires per row
    pub fn poseidon_gate_witness(&self, inputs: &[u64]) -> Result<Vec<u64>, Error> {
        if inputs.len() % 13 != 0 {
            return Err(Error::Invalid("inputs must be n * 13 words".into()));
        }
        let n = inputs.len() / 13;
        let mut out = vec![0u64; n * 135];
        self.check(unsafe { ffi::gl_poseidon_gate_witness(self.raw, inputs.as_ptr(), n as u64, out.as_mut_ptr()) })?;
        Ok(out)
    }

    pub fn openings_begin(&self, log_n: usize) -> Result<Openings<'_>, Error> {
        let mut h: ffi::gl_handle = 0;
        self.check(unsafe { ffi::gl_openings_begin(self.raw, log_n as u32, &mut h) })?;
        Ok(Openings { ctx: self, handle: h })
    }
}

/// `PolynomialBatch::from_values / from_coeffs` on several GPUs from this one process (`gl_commit_multi`): one context per
/// device.  Returns the cap of the whole batch and one shard tree per context; leaf row `i` lives in
/// `shards[i / rows_per_shard]` at local index `i % rows_per_shard`, and `prove` there is `MerkleTree::prove(i)`.
pub fn commit_multi<'c>(
    ctxs: &[&'c Context],
    cols: &[&[u64]],
    rate_bits: usize,
    cap_height: usize,
    input_is_coeffs: bool,
) -> Result<(Vec<HashOut>, Vec<DeviceTree<'c>>), Error> {
    let first = *ctxs.first().ok_or_else(|| Error::Invalid("no contexts".into()))?;
    let n = cols.first().map(|c| c.len()).ok_or_else(|| Error::Invalid("empty polynomial batch".into()))?;
    if cols.iter().any(|c| c.len() != n) {
        return Err(Error::Invalid("Polynomial degrees inconsistent".into()));
    }
    if n == 0 || !n.is_power_of_two() {
        return Err(Error::Invalid("polynomial length must be a power of two".into()));
    }
    if cap_height > 40 {
        return Err(Error::Invalid(format!("cap_height={cap_height} should be at most log2(leaves.len())")));
    }
    let raw: Vec<*mut ffi::gl_ctx> = ctxs.iter().map(|c| c.raw).collect();
    let ptrs: Vec<*const u64> = cols.iter().map(|c| c.as_ptr()).collect();
    let mut cap = vec![[0u64; 4]; 1 << cap_height];
    let mut handles = vec![0 as ffi::gl_handle; ctxs.len()];
    first.check(unsafe {
        ffi::gl_commit_multi(
            raw.as_ptr(),
            raw.len() as u32,
            ptrs.as_ptr(),
            cols.len() as u32,
            n.trailing_zeros(),
            rate_bits as u32,
            cap_height as u32,
            input_is_coeffs as c_int,
            cap.as_mut_ptr() as *mut u64,
            handles.as_mut_ptr(),
        )
    })?;
    let per = cap.len() / ctxs.len();
    let mut shards = Vec::with_capacity(ctxs.len());
    for (g, (&ctx, &h)) in ctxs.iter().zip(handles.iter()).enumerate() {
        shards.push(DeviceTree::adopt(ctx, h, cap[g * per..(g + 1) * per].to_vec())?);
    }
    Ok((cap, shards))
}

impl Drop for Context {
    fn drop(&mut self) {
        unsafe { ffi::gl_ctx_destroy(self.raw) }
    }
}

/// A device-resident `MerkleTree` (and, for commits, the `PolynomialBatch` around it): leaves `[n_leaves][leaf_len]` in plonky2's
/// leaf order (row i = LDE point `reverse_bits(i)`), digests in upstream's interleaved layout, coefficients `[leaf_len][N]`.
pub struct DeviceTree<'c> {
    ctx: &'c Context,
    handle: ffi::gl_handle,
    pub cap: Vec<HashOut>,
    pub info: ffi::gl_tree_info_t,
}

impl<'c> DeviceTree<'c> {
    fn adopt(ctx: &'c Context, handle: ffi::gl_handle, cap: Vec<HashOut>) -> Result<Self, Error> {
        let mut info = ffi::gl_tree_info_t::default();
        ctx.check(unsafe { ffi::gl_tree_info(ctx.raw, handle, &mut info) })?;
        Ok(Self { ctx, handle, cap, info })
    }
    pub fn handle(&self) -> u64 {
        self.handle
    }
    pub fn depth(&self) -> usize {
        self.info.n_leaves.trailing_zeros() as usize - self.info.cap_height as usize
    }
    /// `MerkleTree::get(i)`
    pub fn get(&self, leaf_index: usize) -> Result<Vec<u64>, Error> {
        let mut row = vec![0u64; self.info.leaf_len as usize];
        self.ctx.check(unsafe { ffi::gl_tree_get(self.ctx.raw, self.handle, leaf_index as u64, row.as_mut_ptr()) })?;
        Ok(row)
    }
    /// `MerkleTree::prove(i)`: `MerkleProof::siblings`, bottom-up
    pub fn prove(&self, leaf_index: usize) -> Result<Vec<HashOut>, Error> {
        let mut sib = vec![[0u64; 4]; self.depth()];
        let p = if sib.is_empty() { ptr::null_mut() } else { sib.as_mut_ptr() as *mut u64 };
        self.ctx.check(unsafe { ffi::gl_tree_prove(self.ctx.raw, self.handle, leaf_index as u64, p) })?;
        Ok(sib)
    }
    /// `(get(i), prove(i))` for all indices in one device round trip (the FRI query rounds open 28 indices per tree)
    pub fn open_batch(&self, indices: &[u64]) -> Result<Vec<(Vec<u64>, Vec<HashOut>)>, Error> {
        let (n, ll, d) = (indices.len(), self.info.leaf_len as usize, self.depth());
        let mut rows = vec![0u64; n * ll];
        let mut sib = vec![[0u64; 4]; n * d];
        let idx = if n == 0 { ptr::null() } else { indices.as_ptr() };
        let rp = if rows.is_empty() { ptr::null_mut() } else { rows.as_mut_ptr() };
        let sp = if sib.is_empty() { ptr::null_mut() } else { sib.as_mut_ptr() as *mut u64 };
        self.ctx.check(unsafe { ffi::gl_tree_open_batch(self.ctx.raw, self.handle, idx, n as u32, rp, sp) })?;
        Ok((0..n).map(|q| (rows[q * ll..(q + 1) * ll].to_vec(), sib[q * d..(q + 1) * d].to_vec())).collect())
    }
    /// `PolynomialBatch::get_lde_values(index, step)`
    pub fn get_lde_values(&self, index: usize, step: usize) -> Result<Vec<u64>, Error> {
        let mut row = vec![0u64; self.info.leaf_len as usize];
        self.ctx.check(unsafe { ffi::gl_tree_get_lde_values(self.ctx.raw, self.handle, index as u64, step as u64, row.as_mut_ptr()) })?;
        Ok(row)
    }
    fn read(&self, part: c_int, words: usize) -> Result<Vec<u64>, Error> {
        let mut out = vec![0u64; words.max(1)];
        self.ctx.check(unsafe { ffi::gl_tree_read(self.ctx.raw, self.handle, part, out.as_mut_ptr()) })?;
        out.truncate(words);
        Ok(out)
    }
    /// `PolynomialBatch::polynomials`, column-major `[leaf_len][N]`, canonical
    pub fn coeffs(&self) -> Result<Vec<u64>, Error> {
        self.read(ffi::GL_PART_COEFFS, (self.info.leaf_len as usize) << self.info.degree_log)
    }
    /// `MerkleTree::leaves`, packed row-major
    pub fn leaves(&self) -> Result<Vec<u64>, Error> {
        self.read(ffi::GL_PART_LEAVES, self.info.n_leaves as usize * self.info.leaf_len as usize)
    }
    /// `MerkleTree::digests`, 4 words per hash
    pub fn digests(&self) -> Result<Vec<u64>, Error> {
        self.read(ffi::GL_PART_DIGESTS, 8 * (self.info.n_leaves as usize - (1usize << self.info.cap_height)))
    }
    /// `OpeningSet::new`'s `eval_commitment`: every polynomial of the batch at each of 1 or 2 extension points,
    /// `out[p][j] = polynomials[j].to_extension().eval(points[p])`; the coefficients stay on the device
    pub fn eval_at(&self, points: &[Ext]) -> Result<Vec<Vec<Ext>>, Error> {
        let ll = self.info.leaf_len as usize;
        let mut out = vec![[0u64; 2]; points.len() * ll];
        let pp = if points.is_empty() { ptr::null() } else { points.as_ptr() as *const u64 };
        let op = if out.is_empty() { ptr::null_mut() } else { out.as_mut_ptr() as *mut u64 };
        self.ctx.check(unsafe { ffi::gl_batch_eval(self.ctx.raw, self.handle, pp, points.len() as u32, op) })?;
        Ok(out.chunks(ll.max(1)).map(|c| c.to_vec()).collect())
    }
}

impl Drop for DeviceTree<'_> {
    fn drop(&mut self) {
        unsafe { ffi::gl_tree_free(self.ctx.raw, self.handle) };
    }
}

/// The device-resident state of `fri_committed_trees`; the Fiat–Shamir challenger stays upstream code on the host:
/// per layer `commit_layer` → observe the cap, draw beta → `fold(beta)`; then `final_poly`.
pub struct FriState<'c> {
    ctx: &'c Context,
    handle: ffi::gl_handle,
    cap_height: usize,
}

impl<'c> FriState<'c> {
    /// `reverse_index_bits_in_place(values)`; leaves = chunks of 2^arity_bits, flattened; `MerkleTree::new(leaves, cap_height)`
    pub fn commit_layer(&mut self, arity_bits: usize) -> Result<DeviceTree<'c>, Error> {
        let mut cap = vec![[0u64; 4]; 1 << self.cap_height];
        let mut th: ffi::gl_handle = 0;
        self.ctx.check(unsafe {
            ffi::gl_fri_commit_layer(self.ctx.raw, self.handle, arity_bits as u32, ptr::null_mut(), ptr::null_mut(), cap.as_mut_ptr() as *mut u64, &mut th)
        })?;
        DeviceTree::adopt(self.ctx, th, cap)
    }
    /// coeffs ← `reduce_with_powers` over chunks; shift ← shift^arity; values ← `coset_fft(coeffs, shift)`
    pub fn fold(&mut self, beta: Ext) -> Result<(), Error> {
        self.ctx.check(unsafe { ffi::gl_fri_fold(self.ctx.raw, self.handle, beta.as_ptr()) })
    }
    /// the coefficients truncated to `len >> rate_bits` (`final_poly`)
    pub fn final_poly(&self) -> Result<Vec<Ext>, Error> {
        let mut n = 0u64;
        self.ctx.check(unsafe { ffi::gl_fri_final_poly(self.ctx.raw, self.handle, ptr::null_mut(), &mut n) })?;
        let mut out = vec![[0u64; 2]; n as usize];
        if n > 0 {
            self.ctx.check(unsafe { ffi::gl_fri_final_poly(self.ctx.raw, self.handle, out.as_mut_ptr() as *mut u64, &mut n) })?;
        }
        Ok(out)
    }
    /// number of extension elements of the current codeword (`lde_polynomial_values.len()` before the first fold)
    pub fn len(&self) -> Result<usize, Error> {
        let mut n = 0u64;
        self.ctx.check(unsafe { ffi::gl_fri_read(self.ctx.raw, self.handle, ptr::null_mut(), ptr::null_mut(), &mut n) })?;
        Ok(n as usize)
    }
}

impl Drop for FriState<'_> {
    fn drop(&mut self) {
        unsafe { ffi::gl_fri_end(self.ctx.raw, self.handle) };
    }
}

/// `PolynomialBatch::prove_openings`, front half, on the coefficient matrices the commits left in HBM
pub struct Openings<'c> {
    ctx: &'c Context,
    handle: ffi::gl_handle,
}

impl<'c> Openings<'c> {
    /// one `FriBatchInfo { point, polynomials }`: `reduce_polys_base` (powers of alpha restart at 1), `divide_by_linear`,
    /// `final_poly = final_poly * alpha^len + quotient`.  `polys[j] = (batch, polynomial_index)`.
    pub fn add_batch(&mut self, polys: &[(&DeviceTree<'_>, usize)], alpha: Ext, point: Ext) -> Result<(), Error> {
        let hs: Vec<ffi::gl_handle> = polys.iter().map(|(t, _)| t.handle).collect();
        let cs: Vec<u32> = polys.iter().map(|(_, i)| *i as u32).collect();
        let (hp, cp) = if hs.is_empty() { (ptr::null(), ptr::null()) } else { (hs.as_ptr(), cs.as_ptr()) };
        self.ctx.check(unsafe { ffi::gl_openings_add_batch(self.ctx.raw, self.handle, hp, cp, hs.len() as u32, alpha.as_ptr(), point.as_ptr(), ptr::null_mut()) })
    }
    /// `final_poly.lde(rate_bits)` and `coset_fft(7)`, handed to the commit phase without leaving the device
    pub fn into_fri(self, rate_bits: usize, cap_height: usize) -> Result<FriState<'c>, Error> {
        let mut fh: ffi::gl_handle = 0;
        self.ctx.check(unsafe { ffi::gl_openings_lde(self.ctx.raw, self.handle, rate_bits as u32, cap_height as u32, &mut fh) })?;
        Ok(FriState { ctx: self.ctx, handle: fh, cap_height })
    }
}

impl Drop for Openings<'_> {
    fn drop(&mut self) {
        unsafe { ffi::gl_openings_end(self.ctx.raw, self.handle) };
    }
}

/// `gates/selectors.rs · SelectorsInfo`: gate i is filtered by selector column `selector_indices[i]`, whose gate range is
/// `groups[selector_indices[i]]`
pub struct SelectorsInfo {
    pub selector_indices: Vec<usize>,
    pub groups: Vec<std::ops::Range<usize>>,
}

impl SelectorsInfo {
    pub fn num_selectors(&self) -> usize {
        self.groups.len()
    }
}

/// Pinned host memory for outputs that must be materialised on the host (INTEGRATION.md "Host memory for copy-back")
/// accumulator of `sum_i alpha_k^(offset + i) * constraint_i` over every LDE row of a wires commit (`gl_quotient_*`)
pub struct Quotient<'c> {
    ctx: &'c Context,
    handle: ffi::gl_handle,
    num_challenges: usize,
}

impl<'c> Quotient<'c> {
    pub fn add_gate(&mut self, kind: i32, param: u32, alphas: &[u64], constraint_offset: usize, filter: Option<(&DeviceTree<'c>, usize)>) -> Result<(), Error> {
        assert_eq!(alphas.len(), self.num_challenges, "one alpha per challenge");
        let (fb, fc) = filter.map(|(t, c)| (t.handle, c as u32)).unwrap_or((0, 0));
        self.ctx.check(unsafe { ffi::gl_quotient_add_gate(self.ctx.raw, self.handle, kind as c_int, param, alphas.as_ptr(), constraint_offset as u32, fb, fc) })
    }

    /// `plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch` over the LDE rows: `gates[i] = (kind, param)` of
    /// `CommonCircuitData::gates`, `selectors_info` its `SelectorsInfo`; each gate's constraints times `compute_filter` of its selector
    /// column in `constants_sigmas` (commit #0), constants read from the columns after the selectors
    #[allow(clippy::too_many_arguments)]
    pub fn add_gates(&mut self, gates: &[(i32, u32)], selectors_info: &SelectorsInfo, num_lookup_selectors: usize, constants_sigmas: &DeviceTree<'c>,
                     num_constants: usize, public_inputs_hash: &[u64; 4], alphas: &[u64], constraint_offset: usize) -> Result<(), Error> {
        assert_eq!(alphas.len(), self.num_challenges, "one alpha per challenge");
        assert_eq!(selectors_info.selector_indices.len(), gates.len(), "one selector index per gate");
        let kinds: Vec<c_int> = gates.iter().map(|g| g.0 as c_int).collect();
        let params: Vec<u32> = gates.iter().map(|g| g.1).collect();
        let sel: Vec<u32> = selectors_info.selector_indices.iter().map(|&i| i as u32).collect();
        let groups: Vec<u32> = selectors_info.groups.iter().flat_map(|r| [r.start as u32, r.end as u32]).collect();
        self.ctx.check(unsafe {
            ffi::gl_quotient_add_gates(self.ctx.raw, self.handle, kinds.as_ptr(), params.as_ptr(), gates.len() as u32, sel.as_ptr(), groups.as_ptr(),
                                       selectors_info.num_selectors() as u32, num_lookup_selectors as u32, constants_sigmas.handle,
                                       num_constants as u32, public_inputs_hash.as_ptr(), alphas.as_ptr(), constraint_offset as u32)
        })
    }

    /// the permutation-argument terms of `eval_vanishing_poly_base_batch` (`vanishing_terms[0 .. n_ch * (1 + n_chunks))`)
    #[allow(clippy::too_many_arguments)]
    pub fn add_permutation(&mut self, sigmas: &DeviceTree<'c>, sigma_col0: usize, zs_partial_products: &DeviceTree<'c>, n_routed: usize, degree: usize,
                           k_is: &[u64], betas: &[u64], gammas: &[u64], alphas: &[u64]) -> Result<(), Error> {
        assert!(k_is.len() == n_routed && betas.len() == self.num_challenges && gammas.len() == self.num_challenges && alphas.len() == self.num_challenges);
        self.ctx.check(unsafe {
            ffi::gl_quotient_add_permutation(self.ctx.raw, self.handle, sigmas.handle, sigma_col0 as u32, zs_partial_products.handle, n_routed as u32,
                                             degree as u32, k_is.as_ptr(), betas.as_ptr(), gammas.as_ptr(), alphas.as_ptr())
        })
    }

    /// divide by Z_H on the coset, coset_ifft, chunks(degree), `PolynomialBatch::from_coeffs`: the quotient commitment
    pub fn commit(&self, cap_height: usize) -> Result<DeviceTree<'c>, Error> {
        if cap_height > 31 {
            return Err(Error::Invalid(format!("cap_height={cap_height} should be at most log2(leaves.len())")));
        }
        let mut cap = vec![[0u64; 4]; 1 << cap_height];
        let mut h: ffi::gl_handle = 0;
        self.ctx.check(unsafe { ffi::gl_quotient_commit(self.ctx.raw, self.handle, cap_height as u32, cap.as_mut_ptr() as *mut u64, &mut h) })?;
        DeviceTree::adopt(self.ctx, h, cap)
    }
}

impl Drop for Quotient<'_> {
    fn drop(&mut self) {
        unsafe { ffi::gl_quotient_end(self.ctx.raw, self.handle) };
    }
}

pub struct PinnedBuf {
    ptr: *mut u64,
    words: usize,
}

impl PinnedBuf {
    pub fn new(words: usize) -> Option<Self> {
        let p = unsafe { ffi::gl_host_alloc(words * 8) } as *mut u64;
        if p.is_null() {
            None
        } else {
            Some(Self { ptr: p, words })
        }
    }
    pub fn as_slice(&self) -> &[u64] {
        unsafe { std::slice::from_raw_parts(self.ptr, self.words) }
    }
    pub fn as_mut_slice(&mut self) -> &mut [u64] {
        unsafe { std::slice::from_raw_parts_mut(self.ptr, self.words) }
    }
}

impl Drop for PinnedBuf {
    fn drop(&mut self) {
        unsafe { ffi::gl_host_free(self.ptr as *mut std::os::raw::c_void) }
    }
}
