//! gpu_index.rs -- drop-in for `usearch::ffi::{new_index, Index, IndexOptions, ...}` backed by
//! libdawn_b200 (include/dawn_index.h).  UNCOMPILED IN THIS REPO (no Rust toolchain in the image).
//!
//! `src/search/search_provider.rs` changes exactly one line:
//!     -use usearch::ffi::{new_index, Index, IndexOptions, MetricKind, ScalarKind};
//!     +use crate::index::gpu_index::{new_index, Index, IndexOptions, MetricKind, ScalarKind};
//! Every method keeps the name, argument meaning and `Result` behaviour of the cxx bridge the
//! reference calls at search_provider.rs:102,115,117,133,149,178,214,221,246,280-284.
use std::ffi::{c_char, c_int, c_void, CStr, CString};

#[repr(C)]
struct DawnOptions { dimensions: u32, metric: u32, scalar: u32, device: i32, capacity: u64, flags: u32, reserved: u32 }

extern "C" {
    fn dawn_last_error() -> *const c_char;
    fn dawn_index_create(opts: *const DawnOptions, out: *mut *mut c_void) -> c_int;
    fn dawn_index_free(idx: *mut c_void);
    fn dawn_index_reserve(idx: *mut c_void, n: usize) -> c_int;
    fn dawn_index_add(idx: *mut c_void, label: u64, v: *const f32) -> c_int;
    fn dawn_index_add_batch(idx: *mut c_void, labels: *const u64, v: *const f32, n: usize) -> c_int;
    fn dawn_index_remove(idx: *mut c_void, label: u64, removed: *mut usize) -> c_int;
    fn dawn_index_remove_batch(idx: *mut c_void, labels: *const u64, n: usize, removed: *mut usize) -> c_int;
    fn dawn_index_search(idx: *mut c_void, q: *const f32, k: usize, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_index_search_batch(idx: *mut c_void, q: *const f32, batch: usize, k: usize, labels: *mut u64, dist: *mut f32, counts: *mut usize) -> c_int;
    fn dawn_index_size(idx: *const c_void) -> usize;
    fn dawn_index_capacity(idx: *const c_void) -> usize;
    fn dawn_index_dimensions(idx: *const c_void) -> usize;
    fn dawn_index_save(idx: *mut c_void, path: *const c_char) -> c_int;
    fn dawn_index_load(idx: *mut c_void, path: *const c_char) -> c_int;
    // callers and formats either side of the path (SURVEY 8f)
    fn dawn_index_get(idx: *mut c_void, label: u64, out384: *mut f32) -> c_int;
    fn dawn_index_get_i24(idx: *mut c_void, label: u64, out1152: *mut u8) -> c_int;
    fn dawn_index_search_limit(idx: *mut c_void, q: *const f32, k: usize, distance_limit: f32, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_index_search_i24(idx: *mut c_void, q1152: *const u8, k: usize, has_limit: c_int, distance_limit: f32, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_batcher_create(idx: *mut c_void, max_batch: usize, max_wait_us: u32, out: *mut *mut c_void) -> c_int;
    fn dawn_batcher_create_multi(m: *mut c_void, max_batch: usize, max_wait_us: u32, out: *mut *mut c_void) -> c_int;
    fn dawn_batcher_search(b: *mut c_void, q: *const f32, k: usize, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_batcher_free(b: *mut c_void);
    fn dawn_index_verify(idx: *mut c_void, bad_rows: *mut usize, min_norm: *mut f32, max_norm: *mut f32) -> c_int;
    fn dawn_index_set_option(idx: *mut c_void, key: *const c_char, value: i64) -> c_int;
    fn dawn_multi_set_option(m: *mut c_void, key: *const c_char, value: i64) -> c_int;
    // several GPUs, one process: shards + one NCCL all-gather + device merge inside the library
    fn dawn_multi_create(devices: *const c_int, n_devices: usize, scalar: u32, out: *mut *mut c_void) -> c_int;
    fn dawn_multi_free(m: *mut c_void);
    fn dawn_multi_reserve(m: *mut c_void, n_total: usize) -> c_int;
    fn dawn_multi_add(m: *mut c_void, label: u64, v: *const f32) -> c_int;
    fn dawn_multi_add_batch(m: *mut c_void, labels: *const u64, v: *const f32, n: usize) -> c_int;
    fn dawn_multi_remove(m: *mut c_void, label: u64, removed: *mut usize) -> c_int;
    fn dawn_multi_remove_batch(m: *mut c_void, labels: *const u64, n: usize, removed: *mut usize) -> c_int;
    fn dawn_multi_search(m: *mut c_void, q: *const f32, k: usize, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_multi_search_batch(m: *mut c_void, q: *const f32, batch: usize, k: usize, labels: *mut u64, dist: *mut f32, counts: *mut usize) -> c_int;
    fn dawn_multi_search_limit(m: *mut c_void, q: *const f32, k: usize, limit: f32, labels: *mut u64, dist: *mut f32, count: *mut usize) -> c_int;
    fn dawn_multi_size(m: *const c_void) -> usize;
    fn dawn_multi_capacity(m: *const c_void) -> usize;
    fn dawn_multi_shards(m: *const c_void) -> usize;
    fn dawn_multi_last_error() -> *const c_char;
}

#[derive(Clone, Copy)] pub enum MetricKind { IP }
#[derive(Clone, Copy)] pub enum ScalarKind { F32, F16, F8 }

pub struct IndexOptions {          // same fields as usearch::ffi::IndexOptions (search_provider.rs:35-42)
    pub dimensions: usize, pub metric: MetricKind, pub quantization: ScalarKind,
    pub connectivity: usize, pub expansion_add: usize, pub expansion_search: usize,
}

pub struct Matches { pub labels: Vec<u64>, pub distances: Vec<f32> }   // search_provider.rs:221

pub struct Index { h: *mut c_void }
unsafe impl Send for Index {}      // a handle may be used from any thread
unsafe impl Sync for Index {}      // search* / get are re-entrant, add* / reserve / save / load are serialised inside the library

fn err() -> anyhow::Error {
    anyhow::anyhow!(unsafe { CStr::from_ptr(dawn_last_error()) }.to_string_lossy().into_owned())
}
fn ck(rc: c_int) -> anyhow::Result<()> { if rc == 0 { Ok(()) } else { Err(err()) } }

// usearch ScalarKind -> DAWN_SCALAR_*: F32 keeps the original f32 rows beside the fp16 selection copy, so distances are
// those of an exact f32 brute force over the vectors as given (what the reference's ScalarKind::F32 index stores,
// search_provider.rs:38); F16 = fp16 rows only (768 B / page); F8 = int8 + per-vector scale (388 B / page).
fn scalar_code(q: ScalarKind) -> u32 { match q { ScalarKind::F16 => 0, ScalarKind::F8 => 1, ScalarKind::F32 => 2 } }

pub fn new_index(o: &IndexOptions) -> anyhow::Result<Box<Index>> {       // search_provider.rs:102
    new_index_on(o, 0)
}
/// `new_index` on a chosen CUDA device (the reference has no such knob: USearch runs on the CPU).
pub fn new_index_on(o: &IndexOptions, device: i32) -> anyhow::Result<Box<Index>> {
    let opts = DawnOptions { dimensions: o.dimensions as u32, metric: 0, scalar: scalar_code(o.quantization), device, capacity: 0, flags: 0, reserved: 0 };
    let mut h = std::ptr::null_mut();
    ck(unsafe { dawn_index_create(&opts, &mut h) })?;
    Ok(Box::new(Index { h }))
}

impl Index {
    pub fn reserve(&self, capacity: usize) -> anyhow::Result<()> { ck(unsafe { dawn_index_reserve(self.h, capacity) }) }      // :133,282
    pub fn add(&self, label: u64, vector: &[f32]) -> anyhow::Result<()> {                                                     // :149,284
        anyhow::ensure!(vector.len() == 384, "vector must have 384 dimensions");
        ck(unsafe { dawn_index_add(self.h, label, vector.as_ptr()) })
    }
    pub fn add_batch(&self, labels: &[u64], vectors: &[f32]) -> anyhow::Result<()> {      // bulk rebuild (fill_index_from_db, :127-153)
        anyhow::ensure!(vectors.len() == labels.len() * 384, "vectors must be labels.len() x 384");
        ck(unsafe { dawn_index_add_batch(self.h, labels.as_ptr(), vectors.as_ptr(), labels.len()) })
    }
    /// Drops every stored vector with `label` (a page that was deleted); returns how many were removed.  A re-crawled or
    /// re-embedded page is `remove(id)` then `add(id, &v)`.
    pub fn remove(&self, label: u64) -> anyhow::Result<usize> {
        let mut n = 0usize;
        ck(unsafe { dawn_index_remove(self.h, label, &mut n) })?;
        Ok(n)
    }
    pub fn remove_batch(&self, labels: &[u64]) -> anyhow::Result<usize> {
        let mut n = 0usize;
        ck(unsafe { dawn_index_remove_batch(self.h, labels.as_ptr(), labels.len(), &mut n) })?;
        Ok(n)
    }
    pub fn search(&self, query: &[f32], count: usize) -> anyhow::Result<Matches> {                                            // :214
        anyhow::ensure!(query.len() == 384, "query must have 384 dimensions");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        ck(unsafe { dawn_index_search(self.h, query.as_ptr(), count, labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
    pub fn search_batch(&self, queries: &[f32], count: usize) -> anyhow::Result<Vec<Matches>> {   // for a batching front-end (SURVEY 8f-1)
        let b = queries.len() / 384;
        let (mut labels, mut distances, mut counts) = (vec![0u64; b * count], vec![0f32; b * count], vec![0usize; b]);
        ck(unsafe { dawn_index_search_batch(self.h, queries.as_ptr(), b, count, labels.as_mut_ptr(), distances.as_mut_ptr(), counts.as_mut_ptr()) })?;
        Ok((0..b).map(|i| Matches { labels: labels[i * count..i * count + counts[i]].to_vec(),
                                    distances: distances[i * count..i * count + counts[i]].to_vec() }).collect())
    }
    /// `UdpPacket::Search { distance_limit, .. }` (src/net/udp_packets.rs:29-39): hits with `distance >= limit` are not
    /// returned (src/net/udp_service.rs:196-199); the limit is pushed down into the scan kernels.
    pub fn search_limit(&self, query: &[f32], count: usize, distance_limit: Option<f32>) -> anyhow::Result<Matches> {
        anyhow::ensure!(query.len() == 384, "query must have 384 dimensions");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        ck(unsafe { dawn_index_search_limit(self.h, query.as_ptr(), count, distance_limit.unwrap_or(f32::NAN),
                                            labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
    /// The peer side of a remote search: the 1152-byte i24 embedding straight off the wire (src/search/vector.rs:48-87).
    pub fn search_i24(&self, wire: &[u8], count: usize, distance_limit: Option<f32>) -> anyhow::Result<Matches> {
        anyhow::ensure!(wire.len() == 1152, "i24 embedding must be 1152 bytes");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        ck(unsafe { dawn_index_search_i24(self.h, wire.as_ptr(), count, distance_limit.is_some() as c_int, distance_limit.unwrap_or(0.0),
                                          labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
    /// `embedding_for_page` (search_provider.rs:183-195) served from the device corpus (the stored, fp16-rounded vector).
    pub fn get(&self, label: u64) -> anyhow::Result<Vec<f32>> {
        let mut v = vec![0f32; 384];
        ck(unsafe { dawn_index_get(self.h, label, v.as_mut_ptr()) })?;
        Ok(v)
    }
    /// `GetEmbedding` over UDP (udp_service.rs:254-276): the stored vector in wire format.
    pub fn get_i24(&self, label: u64) -> anyhow::Result<Vec<u8>> {
        let mut v = vec![0u8; 1152];
        ck(unsafe { dawn_index_get_i24(self.h, label, v.as_mut_ptr()) })?;
        Ok(v)
    }
    pub fn size(&self) -> usize { unsafe { dawn_index_size(self.h) } }                 // :246,280
    pub fn capacity(&self) -> usize { unsafe { dawn_index_capacity(self.h) } }         // :280
    pub fn dimensions(&self) -> usize { unsafe { dawn_index_dimensions(self.h) } }
    pub fn save(&self, path: &str) -> anyhow::Result<()> { let p = CString::new(path)?; ck(unsafe { dawn_index_save(self.h, p.as_ptr()) }) }   // :117,178
    pub fn load(&self, path: &str) -> anyhow::Result<()> { let p = CString::new(path)?; ck(unsafe { dawn_index_load(self.h, p.as_ptr()) }) }   // :115
    pub fn view(&self, path: &str) -> anyhow::Result<()> { self.load(path) }          // examples_old/search_usearch.rs:47
}

impl Index {
    /// `SearchProvider::verify` (search_provider.rs:289-327) over the device corpus: (rows failing the norm gate, min |v|, max |v|).
    pub fn verify(&self) -> anyhow::Result<(usize, f32, f32)> {
        let (mut bad, mut lo, mut hi) = (0usize, 0f32, 0f32);
        ck(unsafe { dawn_index_verify(self.h, &mut bad, &mut lo, &mut hi) })?;
        Ok((bad, lo, hi))
    }
    /// Tuning knobs of the library (include/dawn_index.h).  The one a deployment may want: `set_option("shadow_i8", 1)` --
    /// the fp16 corpus also keeps an int8 copy of itself (+388 B per page) that is only used to FILTER on the int8 tensor
    /// cores; every candidate is re-scored on the fp16 rows, so results do not change, batches run ~1.7x faster and a single
    /// query over a big corpus takes half the time.
    pub fn set_option(&self, key: &str, value: i64) -> anyhow::Result<()> {
        let k = std::ffi::CString::new(key)?;
        ck(unsafe { dawn_index_set_option(self.h, k.as_ptr(), value) })
    }
}

impl Drop for Index { fn drop(&mut self) { unsafe { dawn_index_free(self.h) } } }

/// The corpus sharded over several B200s of one box, owned by THIS process (the reference binary is one process,
/// src/bin/dawnsearch.rs:59-128).  Same method names as `Index`, so `SearchProvider` can hold either.  Every search is:
/// local exact top-k on each GPU -> one NCCL all-gather of k (label, distance) pairs per query -> device merge; the
/// on-box analogue of `search_remote` (src/search/search_service.rs:201-277).
pub struct MultiIndex { m: *mut c_void }
unsafe impl Send for MultiIndex {}
fn merr() -> anyhow::Error {
    anyhow::anyhow!(unsafe { CStr::from_ptr(dawn_multi_last_error()) }.to_string_lossy().into_owned())
}
fn mck(rc: c_int) -> anyhow::Result<()> { if rc == 0 { Ok(()) } else { Err(merr()) } }
impl MultiIndex {
    pub fn new(devices: &[i32], quantization: ScalarKind) -> anyhow::Result<MultiIndex> {
        let mut m = std::ptr::null_mut();
        mck(unsafe { dawn_multi_create(devices.as_ptr(), devices.len(), scalar_code(quantization), &mut m) })?;
        Ok(MultiIndex { m })
    }
    pub fn reserve(&self, capacity: usize) -> anyhow::Result<()> { mck(unsafe { dawn_multi_reserve(self.m, capacity) }) }
    pub fn add(&self, label: u64, vector: &[f32]) -> anyhow::Result<()> {
        anyhow::ensure!(vector.len() == 384, "vector must have 384 dimensions");
        mck(unsafe { dawn_multi_add(self.m, label, vector.as_ptr()) })
    }
    pub fn add_batch(&self, labels: &[u64], vectors: &[f32]) -> anyhow::Result<()> {
        anyhow::ensure!(vectors.len() == labels.len() * 384, "vectors must be labels.len() x 384");
        mck(unsafe { dawn_multi_add_batch(self.m, labels.as_ptr(), vectors.as_ptr(), labels.len()) })
    }
    /// Drops the label's vectors on every shard; returns how many were removed in all.
    pub fn remove(&self, label: u64) -> anyhow::Result<usize> {
        let mut n = 0usize;
        mck(unsafe { dawn_multi_remove(self.m, label, &mut n) })?;
        Ok(n)
    }
    pub fn remove_batch(&self, labels: &[u64]) -> anyhow::Result<usize> {
        let mut n = 0usize;
        mck(unsafe { dawn_multi_remove_batch(self.m, labels.as_ptr(), labels.len(), &mut n) })?;
        Ok(n)
    }
    pub fn search(&self, query: &[f32], count: usize) -> anyhow::Result<Matches> {
        anyhow::ensure!(query.len() == 384, "query must have 384 dimensions");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        mck(unsafe { dawn_multi_search(self.m, query.as_ptr(), count, labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
    /// `UdpPacket::Search.distance_limit` (src/net/udp_packets.rs:29-39): every shard applies it before the exchange.
    pub fn search_limit(&self, query: &[f32], count: usize, distance_limit: f32) -> anyhow::Result<Matches> {
        anyhow::ensure!(query.len() == 384, "query must have 384 dimensions");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        mck(unsafe { dawn_multi_search_limit(self.m, query.as_ptr(), count, distance_limit, labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
    pub fn search_batch(&self, queries: &[f32], count: usize) -> anyhow::Result<Vec<Matches>> {
        let b = queries.len() / 384;
        let (mut labels, mut distances, mut counts) = (vec![0u64; b * count], vec![0f32; b * count], vec![0usize; b]);
        mck(unsafe { dawn_multi_search_batch(self.m, queries.as_ptr(), b, count, labels.as_mut_ptr(), distances.as_mut_ptr(), counts.as_mut_ptr()) })?;
        Ok((0..b).map(|i| Matches { labels: labels[i * count..i * count + counts[i]].to_vec(),
                                    distances: distances[i * count..i * count + counts[i]].to_vec() }).collect())
    }
    /// Forwarded to every shard (e.g. `"shadow_i8"`); `"exchange"`: 0 auto, 1 peer copies, 2 NCCL.
    pub fn set_option(&self, key: &str, value: i64) -> anyhow::Result<()> {
        let k = std::ffi::CString::new(key)?;
        mck(unsafe { dawn_multi_set_option(self.m, k.as_ptr(), value) })
    }
    pub fn size(&self) -> usize { unsafe { dawn_multi_size(self.m) } }
    pub fn capacity(&self) -> usize { unsafe { dawn_multi_capacity(self.m) } }
    pub fn shards(&self) -> usize { unsafe { dawn_multi_shards(self.m) } }
}
impl Drop for MultiIndex { fn drop(&mut self) { unsafe { dawn_multi_free(self.m) } } }

/// Micro-batching front for `SearchService` (src/search/search_service.rs:55-104): any number of threads call
/// `search` with one query each; the library answers them in batches (what arrived while the previous batch was on the
/// GPU; a lone caller never waits), which is what feeds the tensor-core path.  The batcher borrows the index: drop it
/// before the index.
pub struct Batcher { b: *mut c_void }
unsafe impl Send for Batcher {}
unsafe impl Sync for Batcher {}
impl Batcher {
    pub fn new(index: &Index, max_batch: usize, max_wait_us: u32) -> anyhow::Result<Batcher> {
        let mut b = std::ptr::null_mut();
        ck(unsafe { dawn_batcher_create(index.h, max_batch, max_wait_us, &mut b) })?;
        Ok(Batcher { b })
    }
    /// The same front over the one-process multi-GPU handle.
    pub fn new_multi(index: &MultiIndex, max_batch: usize, max_wait_us: u32) -> anyhow::Result<Batcher> {
        let mut b = std::ptr::null_mut();
        ck(unsafe { dawn_batcher_create_multi(index.m, max_batch, max_wait_us, &mut b) })?;
        Ok(Batcher { b })
    }
    pub fn search(&self, query: &[f32], count: usize) -> anyhow::Result<Matches> {
        anyhow::ensure!(query.len() == 384, "query must have 384 dimensions");
        let (mut labels, mut distances, mut n) = (vec![0u64; count], vec![0f32; count], 0usize);
        ck(unsafe { dawn_batcher_search(self.b, query.as_ptr(), count, labels.as_mut_ptr(), distances.as_mut_ptr(), &mut n) })?;
        labels.truncate(n); distances.truncate(n);
        Ok(Matches { labels, distances })
    }
}
impl Drop for Batcher { fn drop(&mut self) { unsafe { dawn_batcher_free(self.b) } } }
