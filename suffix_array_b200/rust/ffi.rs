//! `extern "C"` declarations of include/sab200.h (libsab200.so).  NOT COMPILED HERE (no Rust toolchain).
#![allow(dead_code)]
use std::ffi::CStr;
use std::os::raw::c_char;

#[repr(C)]
pub struct Sab200Index {
    _private: [u8; 0],
}

#[link(name = "sab200")]
extern "C" {
    pub fn sab200_saca(s: *const u8, n: u64, sa: *mut u32, ngpus: i32) -> i32;
    pub fn sab200_enable_buckets(s: *const u8, n: u64, bkt: *mut u32) -> i32;
    pub fn sab200_check(s: *const u8, n: u64, sa: *const u32, sa_len: u64) -> i32;
    pub fn sab200_index_create(s: *const u8, n: u64, sa: *const u32, sa_len: u64, bkt_or_null: *const u32, ngpus: i32) -> *mut Sab200Index;
    pub fn sab200_index_destroy(ix: *mut Sab200Index);
    pub fn sab200_search_all_batch(ix: *mut Sab200Index, pats: *const u8, offs: *const u64, np: u64, lo: *mut u32, hi: *mut u32) -> i32;
    pub fn sab200_contains_batch(ix: *mut Sab200Index, pats: *const u8, offs: *const u64, np: u64, out: *mut u8) -> i32;
    pub fn sab200_search_lcp_batch(ix: *mut Sab200Index, pats: *const u8, offs: *const u64, np: u64, start: *mut u32, end: *mut u32) -> i32;
    // matching statistics: len / lo / hi hold offs[nq] entries each, indexed by the absolute offset in qs (include/sab200.h)
    pub fn sab200_matching_statistics_batch(ix: *mut Sab200Index, qs: *const u8, offs: *const u64, nq: u64, len: *mut u32, lo: *mut u32, hi: *mut u32) -> i32;
    pub fn sab200_matching_statistics_batch_device(ix: *mut Sab200Index, d_qs: *const u8, d_offs: *const u64, nq: u64, d_len: *mut u32, d_lo: *mut u32, d_hi: *mut u32) -> i32;
    // feature "pack": GPU forms of PackedSuffixArray::from_sa + dump_bytes / load_bytes + into_sa (src/packed_sa.rs)
    pub fn sab200_pack_bound(sa_len: u64) -> u64;
    pub fn sab200_pack(sa: *const u32, sa_len: u64, out: *mut u8, out_cap: u64, out_len: *mut u64) -> i32;
    pub fn sab200_unpack(bytes: *const u8, nbytes: u64, sa: *mut u32, sa_cap: u64, sa_len: *mut u64) -> i32;
    // Burrows-Wheeler transform (libdivsufsort's divbwt / inverse_bw_transform layout; include/sab200.h)
    pub fn sab200_bwt(s: *const u8, n: u64, bwt: *mut u8, primary: *mut u64) -> i32;
    pub fn sab200_inverse_bwt(bwt: *const u8, n: u64, primary: u64, s: *mut u8) -> i32;
    pub fn sab200_bwt_device(d_s: *const u8, n: u64, d_bwt: *mut u8, primary: *mut u64, device: i32) -> i32;
    pub fn sab200_inverse_bwt_device(d_bwt: *const u8, n: u64, primary: u64, d_s: *mut u8, device: i32) -> i32;
    // LZ77 factorization: z factors (pos, len), len = 0 a literal; *z is reported even when cap < z (include/sab200.h)
    pub fn sab200_lz77(s: *const u8, n: u64, pos: *mut u32, len: *mut u32, cap: u64, z: *mut u64) -> i32;
    pub fn sab200_lz77_decode(pos: *const u32, len: *const u32, z: u64, n: u64, s: *mut u8) -> i32;
    pub fn sab200_lz77_device(d_s: *const u8, n: u64, d_pos: *mut u32, d_len: *mut u32, cap: u64, z: *mut u64, device: i32) -> i32;
    pub fn sab200_lz77_decode_device(d_pos: *const u32, d_len: *const u32, z: u64, n: u64, d_s: *mut u8, device: i32) -> i32;
    pub fn sab200_device_count() -> i32;
    pub fn sab200_last_error() -> *const c_char;
    pub fn sab200_shutdown();
}

pub fn last_error() -> String {
    unsafe { CStr::from_ptr(sab200_last_error()).to_string_lossy().into_owned() }
}
