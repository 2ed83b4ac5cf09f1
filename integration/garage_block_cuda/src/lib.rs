//! Safe wrapper with Garage's conventions (see INTEGRATION.md section 2).  NOT compiled here.
pub mod batch;   // the batching front-end (row f1): EcBatcher::encode / ::reconstruct are what BlockManager calls
pub mod placement;   // row f4: shard-aware nodes_of / write sets / read plan (pure Rust, belongs in garage_rpc)
pub mod sys;

use bytes::Bytes;
use garage_util::data::Hash;
use garage_util::error::Error;

pub struct ErasureCoder { pub(crate) ctx: *mut sys::garage_ec_ctx, pub k: usize, pub m: usize }
unsafe impl Send for ErasureCoder {}   // the C context is internally synchronised
unsafe impl Sync for ErasureCoder {}

pub(crate) fn check(ctx: *const sys::garage_ec_ctx, rc: i32) -> Result<(), Error> {
    if rc == sys::GARAGE_EC_OK { return Ok(()); }
    let msg = unsafe { std::ffi::CStr::from_ptr(sys::garage_ec_strerror(rc)) }.to_string_lossy();
    let det = unsafe { std::ffi::CStr::from_ptr(sys::garage_ec_last_error(ctx)) }.to_string_lossy();
    Err(Error::Message(format!("garage_ec: {} {}", msg, det)))
}

impl ErasureCoder {
    pub fn new(cuda_device: i32, k: usize, m: usize) -> Result<Self, Error> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { sys::garage_ec_create(&mut ctx, cuda_device, k as i32, m as i32, sys::GARAGE_EC_VANDERMONDE) };
        check(std::ptr::null(), rc)?;       // NODEVICE => node refuses to start in EC mode: no CPU fallback
        Ok(Self { ctx, k, m })
    }
    /// HOST-mode calls sleep on an event instead of spinning in the driver: for the batch dispatchers,
    /// which otherwise pin one CPU each while their batch is on the GPU.
    pub fn set_wait_blocking(&self, blocking: bool) {
        unsafe { sys::garage_ec_set_wait_mode(self.ctx, blocking as i32) };
    }
    pub fn shard_len(&self, block_len: usize) -> usize {
        unsafe { sys::garage_ec_shard_len(block_len as u32, self.k as i32) as usize }
    }

    /// Parity shards of a batch of blocks.  Data shard j of block s is the slice
    /// blocks[s][j*L..(j+1)*L] (zero padded), so only parity crosses PCIe back.
    pub fn encode_blocks(&self, blocks: &[Bytes]) -> Result<Vec<Vec<Bytes>>, Error> {
        let max = blocks.iter().map(|b| b.len()).max().unwrap_or(0);
        let stride = unsafe { sys::garage_ec_stride_for(self.shard_len(max) as u32) };
        let ptrs: Vec<*const u8> = blocks.iter().map(|b| b.as_ptr()).collect();
        let lens: Vec<u32> = blocks.iter().map(|b| b.len() as u32).collect();
        let mut parity = vec![0u8; blocks.len() * self.m * stride];
        let rc = unsafe { sys::garage_ec_encode_blocks(self.ctx, ptrs.as_ptr(), lens.as_ptr(), blocks.len(),
                                                       parity.as_mut_ptr(), stride) };
        check(self.ctx, rc)?;
        let parity = Bytes::from(parity);
        Ok(blocks.iter().enumerate().map(|(s, b)| {
            let l = self.shard_len(b.len());
            (0..self.m).map(|i| parity.slice((s * self.m + i) * stride..(s * self.m + i) * stride + l)).collect()
        }).collect())
    }

    /// GET / resync, ONE stripe per call: kept for tools and tests.  The block manager goes through
    /// batch::EcBatcher::reconstruct instead (one FFI call per stripe is the slowest way to drive the GPU).
    /// `shards[i]` is Some(bytes) for every shard that arrived.  Rebuilds the
    /// shards selected by `want` (data shards for GET, this node's index for resync).
    pub fn reconstruct(&self, hash: &Hash, block_len: usize, shards: &mut [Option<Vec<u8>>], want: &[bool])
        -> Result<(), Error>
    {
        let tot = self.k + self.m;
        let l = self.shard_len(block_len);
        let stride = unsafe { sys::garage_ec_stride_for(l as u32) };
        // the C ABI wants 16-byte aligned bases: glibc's allocator gives that for a Vec<u8> of this size;
        // production code takes these buffers from garage_ec_host_alloc (pinned, page aligned)
        let mut buf = vec![0u8; tot * stride];
        let mut present = vec![0u8; tot];
        for (i, s) in shards.iter().enumerate() {
            if let Some(s) = s { buf[i * stride..i * stride + l].copy_from_slice(&s[..l]); present[i] = 1; }
        }
        let want_u8: Vec<u8> = want.iter().map(|w| *w as u8).collect();
        let (mut status, lens) = ([0i32; 1], [l as u32; 1]);
        let rc = unsafe { sys::garage_ec_reconstruct(self.ctx, buf.as_mut_ptr(), present.as_ptr(), want_u8.as_ptr(),
                          status.as_mut_ptr(), lens.as_ptr(), stride, 1, sys::GARAGE_EC_MEM_HOST, std::ptr::null_mut()) };
        if rc == sys::GARAGE_EC_E_UNRECOVERABLE { return Err(Error::MissingBlock(*hash)); }
        check(self.ctx, rc)?;
        for i in 0..tot {
            if present[i] == 0 && want[i] { shards[i] = Some(buf[i * stride..i * stride + l].to_vec()); }
        }
        Ok(())
    }

    /// GET whose block failed DataBlock::verify (src/block/block.rs:69-83) although every shard passed its
    /// own tag: locate and repair the wrong shards of ONE stripe from the parity alone.  `shards[i]` is
    /// Some(bytes) for every shard that arrived; on success the absent ones are filled in, the wrong ones
    /// rewritten, and the indices of the rewritten shards are returned (quarantine them, queue resync).
    /// Err(CorruptData) when some column has more wrong shards than the parity can locate: fall back to
    /// the tags / a leave-one-out search.  The block hash stays the final check.
    pub fn correct(&self, hash: &Hash, block_len: usize, shards: &mut [Option<Vec<u8>>]) -> Result<Vec<usize>, Error> {
        let tot = self.k + self.m;
        let l = self.shard_len(block_len);
        let stride = unsafe { sys::garage_ec_stride_for(l as u32) };
        let mut buf = vec![0u8; tot * stride];
        let mut present = vec![0u8; tot];
        for (i, s) in shards.iter().enumerate() {
            if let Some(s) = s { buf[i * stride..i * stride + l].copy_from_slice(&s[..l]); present[i] = 1; }
        }
        let (mut status, mut fixed, lens) = ([0i32; 1], vec![0u8; tot], [l as u32; 1]);
        let rc = unsafe { sys::garage_ec_correct(self.ctx, buf.as_mut_ptr(), present.as_ptr(), status.as_mut_ptr(),
                          fixed.as_mut_ptr(), lens.as_ptr(), stride, 1, sys::GARAGE_EC_MEM_HOST, std::ptr::null_mut()) };
        if rc == sys::GARAGE_EC_E_UNRECOVERABLE { return Err(Error::MissingBlock(*hash)); }
        if rc == sys::GARAGE_EC_E_UNCORRECTABLE { return Err(Error::CorruptData(*hash)); }
        check(self.ctx, rc)?;
        for i in 0..tot {
            if present[i] == 0 || fixed[i] != 0 { shards[i] = Some(buf[i * stride..i * stride + l].to_vec()); }
        }
        Ok((0..tot).filter(|&i| fixed[i] != 0).collect())
    }

    /// Scrub: bit i of the result set = stored parity row i disagrees with the data shards.
    pub fn verify(&self, shards_layout: &[u8], shard_len: &[u32], stride: usize) -> Result<Vec<u32>, Error> {
        let n = shard_len.len();
        let mut mm = vec![0u32; n];
        let rc = unsafe { sys::garage_ec_verify(self.ctx, shards_layout.as_ptr(), mm.as_mut_ptr(), shard_len.as_ptr(),
                          stride, n, sys::GARAGE_EC_MEM_HOST, std::ptr::null_mut()) };
        check(self.ctx, rc)?;
        Ok(mm)
    }
}
impl Drop for ErasureCoder { fn drop(&mut self) { unsafe { sys::garage_ec_destroy(self.ctx) } } }
