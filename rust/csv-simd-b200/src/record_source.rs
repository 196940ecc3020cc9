//! Batched lookups next to csv-simd's scalar `RecordSource::seek_record` / `seek_field`
//! (src/record_source.rs:70-140, unchanged: two reads of the host index each).
use crate::gpu::Context;
use crate::{check, sys, StructureError};
use std::ptr;

/// A device-resident copy of a tape: the bytes, the index and the `TapeCore::init` metadata (src/tape.rs:315-347).
pub struct DeviceTape<'a> {
    gpu: &'a Context,
    idx: *mut sys::csvb200_index,
    pub record_cnt: u32,
    pub jump: u64,
}

impl<'a> DeviceTape<'a> {
    /// `field_cnt` and `crlf` come from `Header::new` (src/tape.rs:226-273), which stays host code.
    pub fn new(gpu: &'a Context, bytes: &[u8], field_cnt: u32, crlf: bool) -> Result<Self, StructureError> {
        let mut idx = ptr::null_mut();
        check(unsafe {
            sys::csvb200_index_build(gpu.raw(), bytes.as_ptr(), bytes.len(),
                                     sys::CSVB200_BUILD_KEEP_BYTES | sys::CSVB200_BUILD_STRICT_MIN64, &mut idx)
        }, || gpu.last_error())?;
        let (mut record_cnt, mut jump) = (0u32, 0u64);
        let rc = unsafe { sys::csvb200_tape_init(idx, field_cnt, crlf as i32, &mut record_cnt, &mut jump) };
        if rc != sys::CSVB200_OK {
            unsafe { sys::csvb200_index_free(idx) };
            check(rc, || gpu.last_error())?;     // InvalidCsvFormat when (len - 1) % jump != 0 (src/tape.rs:327,342-344)
        }
        Ok(DeviceTape { gpu, idx, record_cnt, jump })
    }
}

impl Drop for DeviceTape<'_> {
    fn drop(&mut self) {
        unsafe { sys::csvb200_index_free(self.idx) }
    }
}

pub trait BatchedSeeks {
    /// `(start, end)` byte ranges of many `(record, field)` pairs; `None` exactly where `seek_field` returns `Ok(None)`.
    fn seek_fields(&self, rec: &[u32], fld: &[u32]) -> Result<Vec<Option<(usize, usize)>>, StructureError>;
    fn seek_records(&self, rec: &[u32]) -> Result<Vec<Option<(usize, usize)>>, StructureError>;
    /// The values behind `seek_fields`: field `fld[q]` of record `rec[q]`, trimmed / unquoted by `flags`
    /// (`sys::CSVB200_FIELD_*`), packed on the GPU.
    fn field_values(&self, rec: &[u32], fld: &[u32], flags: u32) -> Result<Values, StructureError>;
    /// The record text behind `seek_records`.
    fn record_values(&self, rec: &[u32]) -> Result<Values, StructureError>;
}

/// Packed values of a batch: value `q` is `bytes[offsets[q]..offsets[q + 1]]`.
pub struct Values {
    pub offsets: Vec<u64>,
    pub bytes: Vec<u8>,
    /// bit `q % 64` of word `q / 64`: the lookup found a range
    pub found: Vec<u64>,
}

impl Values {
    /// `None` exactly where `seek_field` / `seek_record` return `Ok(None)`.
    pub fn get(&self, q: usize) -> Option<&[u8]> {
        if (self.found[q / 64] >> (q % 64)) & 1 == 0 {
            return None;
        }
        Some(&self.bytes[self.offsets[q] as usize..self.offsets[q + 1] as usize])
    }
    pub fn len(&self) -> usize {
        self.offsets.len() - 1
    }
    pub fn is_empty(&self) -> bool {
        self.len() == 0
    }
}

fn ranges(out: Vec<sys::csvb200_range>) -> Vec<Option<(usize, usize)>> {
    out.iter().map(|r| if r.start == u64::MAX { None } else { Some((r.start as usize, r.end as usize)) }).collect()
}

impl BatchedSeeks for DeviceTape<'_> {
    fn seek_fields(&self, rec: &[u32], fld: &[u32]) -> Result<Vec<Option<(usize, usize)>>, StructureError> {
        assert_eq!(rec.len(), fld.len());
        let mut out = vec![sys::csvb200_range::default(); rec.len()];
        check(unsafe { sys::csvb200_seek_fields(self.idx, rec.as_ptr(), fld.as_ptr(), rec.len(), out.as_mut_ptr()) },
              || self.gpu.last_error())?;
        Ok(ranges(out))
    }
    fn seek_records(&self, rec: &[u32]) -> Result<Vec<Option<(usize, usize)>>, StructureError> {
        let mut out = vec![sys::csvb200_range::default(); rec.len()];
        check(unsafe { sys::csvb200_seek_records(self.idx, rec.as_ptr(), rec.len(), out.as_mut_ptr()) },
              || self.gpu.last_error())?;
        Ok(ranges(out))
    }
    fn field_values(&self, rec: &[u32], fld: &[u32], flags: u32) -> Result<Values, StructureError> {
        assert_eq!(rec.len(), fld.len());
        self.values(rec, fld.as_ptr(), flags)
    }
    fn record_values(&self, rec: &[u32]) -> Result<Values, StructureError> {
        self.values(rec, ptr::null(), 0)
    }
}

impl DeviceTape<'_> {
    // csvb200_seek_values twice: the first call sizes the bytes (CSVB200_ERR_CAPACITY), the second fills them
    fn values(&self, rec: &[u32], fld: *const u32, flags: u32) -> Result<Values, StructureError> {
        let nq = rec.len();
        let mut v = Values { offsets: vec![0; nq + 1], bytes: Vec::new(), found: vec![0; (nq + 63) / 64 + 1] };
        let mut total = 0usize;
        let rc = unsafe {
            sys::csvb200_seek_values(self.idx, rec.as_ptr(), fld, nq, flags, v.offsets.as_mut_ptr(), ptr::null_mut(), 0,
                                     &mut total, v.found.as_mut_ptr())
        };
        if rc != sys::CSVB200_ERR_CAPACITY {
            check(rc, || self.gpu.last_error())?;
        }
        v.bytes = vec![0; total];
        if total > 0 {
            check(unsafe {
                sys::csvb200_seek_values(self.idx, rec.as_ptr(), fld, nq, flags, v.offsets.as_mut_ptr(), v.bytes.as_mut_ptr(),
                                         total, &mut total, v.found.as_mut_ptr())
            }, || self.gpu.last_error())?;
        }
        Ok(v)
    }
}
