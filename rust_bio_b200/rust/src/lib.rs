//! `bio_b200::alignment::pairwise` -- the rust-bio 4.0.1 pairwise API on a B200.
//!
//! NOT COMPILED IN THIS REPOSITORY'S BUILD IMAGE (no Rust toolchain there).  It is the binding a
//! maintainer adds next to `bio`: same type and method names as
//! `bio::alignment::pairwise::{MIN_SCORE, MatchFunc, MatchParams, Scoring, Aligner}`
//! (rust-bio src/alignment/pairwise/mod.rs:174-1015) plus `*_batch` methods; every method goes
//! through the C ABI of `include/b200align.h` -- there is no CPU implementation behind it.
//!
//! ```ignore
//! // before:  use bio::alignment::pairwise::*;
//! use bio_b200::alignment::pairwise::*;
//! let score = |a: u8, b: u8| if a == b { 1i32 } else { -1i32 };
//! let mut aligner = Aligner::with_capacity(150, 150, -5, -1, &score);
//! let alns = aligner.local_batch(&pairs);          // Vec<bio_types::alignment::Alignment>
//! let one = aligner.local(x, y);                   // a batch of one
//! ```
#![allow(non_camel_case_types, non_snake_case)]

pub mod alignment {
    pub use bio_types::alignment::{Alignment, AlignmentMode, AlignmentOperation};

    pub mod pairwise {
        use super::{Alignment, AlignmentMode, AlignmentOperation};
        use std::ffi::CStr;
        use std::os::raw::{c_char, c_void};

        /// mod.rs:174
        pub const MIN_SCORE: i32 = -858_993_459;

        // ---------------------------------------------------------------- FFI (include/b200align.h)
        #[repr(C)]
        struct b2a_scoring {
            gap_open: i32,
            gap_extend: i32,
            xclip_prefix: i32,
            xclip_suffix: i32,
            yclip_prefix: i32,
            yclip_suffix: i32,
            match_score: i32,
            mismatch_score: i32,
            has_match_scores: i32,
            table: *const i32,
            alphabet: *const u8,
            alphabet_len: u32,
        }
        #[repr(C)]
        struct b2a_pairs {
            seq_blob: *const u8,
            x_off: *const u64,
            x_len: *const u32,
            y_off: *const u64,
            y_len: *const u32,
            blob_bytes: u64,
            n_pairs: u64,
        }
        #[repr(C)]
        struct b2a_results {
            score: *mut i32,
            xstart: *mut u32,
            xend: *mut u32,
            ystart: *mut u32,
            yend: *mut u32,
            ops_off: *mut u64,
            ops: *mut u8,
            ops_capacity: u64,
            clip_len: *mut u32,
            status: *mut u32, // per-pair B2A_PAIR_* codes; null = a failing pair fails the batch (-> panic, like the reference)
        }
        #[repr(C)]
        struct b2a_score_results {
            score: *mut i32,
            xend: *mut u32,
            yend: *mut u32,
            status: *mut u32,
        }
        #[link(name = "b200align")]
        extern "C" {
            fn b2a_score_batch(
                e: *mut c_void,
                mode: i32,
                scoring: *const b2a_scoring,
                pairs: *const b2a_pairs,
                results: *mut b2a_score_results,
                stats: *mut c_void,
            ) -> i32;
            fn b2a_engine_create(out: *mut *mut c_void, device_id: i32) -> i32;
            // every visible GPU from this one process (include/b200align.h: b2a_multi_*)
            fn b2a_multi_create(out: *mut *mut c_void, device_ids: *const i32, n_devices: i32) -> i32;
            fn b2a_multi_destroy(m: *mut c_void) -> i32;
            fn b2a_multi_last_error(m: *const c_void) -> *const c_char;
            fn b2a_multi_align_batch(
                m: *mut c_void,
                mode: i32,
                scoring: *const b2a_scoring,
                pairs: *const b2a_pairs,
                results: *mut b2a_results,
                stats: *mut c_void,
            ) -> i32;
            fn b2a_engine_destroy(e: *mut c_void) -> i32;
            fn b2a_last_error(e: *const c_void) -> *const c_char;
            fn b2a_align_batch(
                e: *mut c_void,
                mode: i32,
                scoring: *const b2a_scoring,
                pairs: *const b2a_pairs,
                results: *mut b2a_results,
                stats: *mut c_void,
            ) -> i32;
            fn b2a_align_batch_banded(
                e: *mut c_void,
                mode: i32,
                scoring: *const b2a_scoring,
                k: u32,
                w: u32,
                pairs: *const b2a_pairs,
                results: *mut b2a_results,
                stats: *mut c_void,
            ) -> i32;
            fn b2a_align_batch_banded_hinted(
                e: *mut c_void,
                mode: i32,
                scoring: *const b2a_scoring,
                k: u32,
                w: u32,
                pairs: *const b2a_pairs,
                hints: *const b2a_band_hints,
                results: *mut b2a_results,
                stats: *mut c_void,
            ) -> i32;
        }
        #[repr(C)]
        struct b2a_band_hints {
            match_off: *const u64,
            match_xy: *const u32,
            path_off: *const u64,
            path_idx: *const u32,
            allowed_mismatches: i32,
            use_lcskpp_union: i32,
        }

        /// What a banded call adds to `Aligner::batch`: k, w and (banded.rs:294-401) the caller's band inputs.
        pub(crate) struct BandedCall<'a> {
            pub k: u32,
            pub w: u32,
            pub matches: Option<&'a [&'a [(u32, u32)]]>,
            pub paths: Option<&'a [&'a [usize]]>,
            pub allowed_mismatches: Option<usize>,
            pub use_lcskpp_union: bool,
        }

        // ---------------------------------------------------------------- scoring, mod.rs:177-429
        pub trait MatchFunc {
            fn score(&self, a: u8, b: u8) -> i32;
        }

        #[derive(Default, Copy, Clone, Eq, PartialEq, Ord, PartialOrd, Hash, Debug)]
        pub struct MatchParams {
            pub match_score: i32,
            pub mismatch_score: i32,
        }
        impl MatchParams {
            pub fn new(match_score: i32, mismatch_score: i32) -> Self {
                assert!(match_score >= 0, "match_score can't be negative");
                assert!(mismatch_score <= 0, "mismatch_score can't be positive");
                MatchParams { match_score, mismatch_score }
            }
        }
        impl MatchFunc for MatchParams {
            fn score(&self, a: u8, b: u8) -> i32 {
                if a == b { self.match_score } else { self.mismatch_score }
            }
        }
        impl<F> MatchFunc for F
        where
            F: Fn(u8, u8) -> i32,
        {
            fn score(&self, a: u8, b: u8) -> i32 {
                (self)(a, b)
            }
        }

        #[derive(Default, Copy, Clone, Eq, PartialEq, Ord, PartialOrd, Hash, Debug)]
        pub struct Scoring<F: MatchFunc> {
            pub gap_open: i32,
            pub gap_extend: i32,
            pub match_fn: F,
            pub match_scores: Option<(i32, i32)>,
            pub xclip_prefix: i32,
            pub xclip_suffix: i32,
            pub yclip_prefix: i32,
            pub yclip_suffix: i32,
        }
        impl Scoring<MatchParams> {
            pub fn from_scores(gap_open: i32, gap_extend: i32, match_score: i32, mismatch_score: i32) -> Self {
                assert!(gap_open <= 0, "gap_open can't be positive");
                assert!(gap_extend <= 0, "gap_extend can't be positive");
                Scoring {
                    gap_open,
                    gap_extend,
                    match_fn: MatchParams::new(match_score, mismatch_score),
                    match_scores: Some((match_score, mismatch_score)),
                    xclip_prefix: MIN_SCORE,
                    xclip_suffix: MIN_SCORE,
                    yclip_prefix: MIN_SCORE,
                    yclip_suffix: MIN_SCORE,
                }
            }
        }
        impl<F: MatchFunc> Scoring<F> {
            pub fn new(gap_open: i32, gap_extend: i32, match_fn: F) -> Self {
                assert!(gap_open <= 0, "gap_open can't be positive");
                assert!(gap_extend <= 0, "gap_extend can't be positive");
                Scoring {
                    gap_open,
                    gap_extend,
                    match_fn,
                    match_scores: None,
                    xclip_prefix: MIN_SCORE,
                    xclip_suffix: MIN_SCORE,
                    yclip_prefix: MIN_SCORE,
                    yclip_suffix: MIN_SCORE,
                }
            }
            pub fn xclip(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.xclip_prefix = penalty;
                self.xclip_suffix = penalty;
                self
            }
            pub fn xclip_prefix(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.xclip_prefix = penalty;
                self
            }
            pub fn xclip_suffix(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.xclip_suffix = penalty;
                self
            }
            pub fn yclip(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.yclip_prefix = penalty;
                self.yclip_suffix = penalty;
                self
            }
            pub fn yclip_prefix(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.yclip_prefix = penalty;
                self
            }
            pub fn yclip_suffix(mut self, penalty: i32) -> Self {
                assert!(penalty <= 0, "Clipping penalty can't be positive");
                self.yclip_suffix = penalty;
                self
            }
        }

        // ---------------------------------------------------------------- Aligner, mod.rs:472-1015
        /// Holds the scoring and an engine handle (one CUDA device) instead of host scratch vectors.
        /// Not `Clone`/`Serialize` (documented API deviation, SURVEY section 5).
        pub struct Aligner<F: MatchFunc> {
            scoring: Scoring<F>,
            engine: *mut c_void,
            /// non-null after `on_all_gpus()`: `*_batch` calls are split over every visible GPU (one ncclAllGather
            /// reassembles them); the banded entry points stay on `engine`'s device
            multi: *mut c_void,
        }
        unsafe impl<F: MatchFunc + Send> Send for Aligner<F> {}

        impl<F: MatchFunc> Drop for Aligner<F> {
            fn drop(&mut self) {
                unsafe {
                    if !self.multi.is_null() {
                        b2a_multi_destroy(self.multi);
                    }
                    b2a_engine_destroy(self.engine)
                };
            }
        }

        const DEFAULT_ALIGNER_CAPACITY: usize = 200;

        impl<F: MatchFunc> Aligner<F> {
            pub fn new(gap_open: i32, gap_extend: i32, match_fn: F) -> Self {
                Aligner::with_capacity(DEFAULT_ALIGNER_CAPACITY, DEFAULT_ALIGNER_CAPACITY, gap_open, gap_extend, match_fn)
            }
            pub fn with_capacity(_m: usize, _n: usize, gap_open: i32, gap_extend: i32, match_fn: F) -> Self {
                assert!(gap_open <= 0, "gap_open can't be positive");
                assert!(gap_extend <= 0, "gap_extend can't be positive");
                Self::make(Scoring::new(gap_open, gap_extend, match_fn))
            }
            pub fn with_scoring(scoring: Scoring<F>) -> Self {
                Aligner::with_capacity_and_scoring(DEFAULT_ALIGNER_CAPACITY, DEFAULT_ALIGNER_CAPACITY, scoring)
            }
            pub fn with_capacity_and_scoring(_m: usize, _n: usize, scoring: Scoring<F>) -> Self {
                assert!(scoring.gap_open <= 0, "gap_open can't be positive");
                assert!(scoring.gap_extend <= 0, "gap_extend can't be positive");
                assert!(scoring.xclip_prefix <= 0, "Clipping penalty (x prefix) can't be positive");
                assert!(scoring.xclip_suffix <= 0, "Clipping penalty (x suffix) can't be positive");
                assert!(scoring.yclip_prefix <= 0, "Clipping penalty (y prefix) can't be positive");
                assert!(scoring.yclip_suffix <= 0, "Clipping penalty (y suffix) can't be positive");
                Self::make(scoring)
            }
            fn make(scoring: Scoring<F>) -> Self {
                let mut engine: *mut c_void = std::ptr::null_mut();
                let device = std::env::var("B2A_DEVICE").ok().and_then(|v| v.parse().ok()).unwrap_or(0);
                let rc = unsafe { b2a_engine_create(&mut engine, device) };
                assert!(rc == 0, "b200align: no usable sm_100 device (rc = {}); there is no CPU fallback", rc);
                Aligner { scoring, engine, multi: std::ptr::null_mut() }
            }

            /// Use every visible B200 for the `*_batch` methods (not part of rust-bio's API: its Aligner is a
            /// single-threaded CPU object).  Panics if the devices cannot be opened.
            pub fn on_all_gpus(mut self) -> Self {
                let mut m: *mut c_void = std::ptr::null_mut();
                let rc = unsafe { b2a_multi_create(&mut m, std::ptr::null(), 0) };
                assert!(rc == 0, "b200align: cannot open every visible device (rc = {})", rc);
                self.multi = m;
                self
            }

            /// Aligner::custom / global / semiglobal / local over a batch (mode = B2A_MODE_*).
            pub(crate) fn batch(&mut self, mode: i32, banded: Option<BandedCall>, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> {
                let n = pairs.len();
                // 16-byte aligned slots, x then y per pair
                let mut x_off = Vec::with_capacity(n);
                let mut y_off = Vec::with_capacity(n);
                let mut x_len = Vec::with_capacity(n);
                let mut y_len = Vec::with_capacity(n);
                let mut blob: Vec<u8> = Vec::new();
                let mut present = [false; 256];
                for (x, y) in pairs {
                    for s in [x, y] {
                        while blob.len() % 16 != 0 {
                            blob.push(0);
                        }
                        if std::ptr::eq(*s, *x) { x_off.push(blob.len() as u64) } else { y_off.push(blob.len() as u64) }
                        blob.extend_from_slice(s);
                        for &b in s.iter() {
                            present[b as usize] = true;
                        }
                    }
                    x_len.push(x.len() as u32);
                    y_len.push(y.len() as u32);
                }
                // tabulate the MatchFunc over the symbols present (mod.rs:221-228 allows any closure)
                let alphabet: Vec<u8> = (0..=255u8).filter(|b| present[*b as usize]).collect();
                let mut table = vec![0i32; 256 * 256];
                for &a in &alphabet {
                    for &b in &alphabet {
                        table[a as usize * 256 + b as usize] = self.scoring.match_fn.score(a, b);
                    }
                }
                let (ms, mm) = self.scoring.match_scores.unwrap_or((0, 0));
                let cs = b2a_scoring {
                    gap_open: self.scoring.gap_open,
                    gap_extend: self.scoring.gap_extend,
                    xclip_prefix: self.scoring.xclip_prefix,
                    xclip_suffix: self.scoring.xclip_suffix,
                    yclip_prefix: self.scoring.yclip_prefix,
                    yclip_suffix: self.scoring.yclip_suffix,
                    match_score: ms,
                    mismatch_score: mm,
                    has_match_scores: self.scoring.match_scores.is_some() as i32,
                    table: table.as_ptr(),
                    alphabet: alphabet.as_ptr(),
                    alphabet_len: alphabet.len() as u32,
                };
                let cp = b2a_pairs {
                    seq_blob: blob.as_ptr(),
                    x_off: x_off.as_ptr(),
                    x_len: x_len.as_ptr(),
                    y_off: y_off.as_ptr(),
                    y_len: y_len.as_ptr(),
                    blob_bytes: blob.len() as u64,
                    n_pairs: n as u64,
                };
                let cap: u64 = pairs.iter().map(|(x, y)| (x.len() + y.len() + 4) as u64).sum();
                let mut score = vec![0i32; n];
                let (mut xs, mut xe, mut ys, mut ye) = (vec![0u32; n], vec![0u32; n], vec![0u32; n], vec![0u32; n]);
                let mut ops_off = vec![0u64; n + 1];
                let mut ops = vec![0u8; cap as usize + 1];
                let mut clip = vec![0u32; 4 * n.max(1)];
                let mut res = b2a_results {
                    score: score.as_mut_ptr(),
                    xstart: xs.as_mut_ptr(),
                    xend: xe.as_mut_ptr(),
                    ystart: ys.as_mut_ptr(),
                    yend: ye.as_mut_ptr(),
                    ops_off: ops_off.as_mut_ptr(),
                    ops: ops.as_mut_ptr(),
                    ops_capacity: cap + 1,
                    clip_len: clip.as_mut_ptr(),
                    status: std::ptr::null_mut(),
                };
                let is_banded = banded.is_some();
                let rc = match banded {
                    None if !self.multi.is_null() => {
                        let rc = unsafe { b2a_multi_align_batch(self.multi, mode, &cs, &cp, &mut res, std::ptr::null_mut()) };
                        if rc != 0 {
                            let msg = unsafe { CStr::from_ptr(b2a_multi_last_error(self.multi)) }.to_string_lossy().into_owned();
                            panic!("{}", msg);
                        }
                        rc
                    }
                    None => unsafe { b2a_align_batch(self.engine, mode, &cs, &cp, &mut res, std::ptr::null_mut()) },
                    Some(BandedCall { k, w, matches: None, .. }) => unsafe {
                        b2a_align_batch_banded(self.engine, mode, &cs, k, w, &cp, &mut res, std::ptr::null_mut())
                    },
                    Some(BandedCall { k, w, matches: Some(ms), paths, allowed_mismatches, use_lcskpp_union }) => {
                        // CSR form of the per-pair matches (and paths), include/b200align.h b2a_band_hints
                        assert!(ms.len() == n, "one match list per pair");
                        let mut match_off = vec![0u64; n + 1];
                        let mut match_xy: Vec<u32> = Vec::new();
                        for (p, m) in ms.iter().enumerate() {
                            for &(a, b) in m.iter() {
                                match_xy.push(a);
                                match_xy.push(b);
                            }
                            match_off[p + 1] = (match_xy.len() / 2) as u64;
                        }
                        match_xy.push(0); // never a dangling pointer for an empty list
                        let mut path_off = vec![0u64; n + 1];
                        let mut path_idx: Vec<u32> = Vec::new();
                        if let Some(ps) = paths {
                            assert!(ps.len() == n, "one path per pair");
                            for (p, path) in ps.iter().enumerate() {
                                path_idx.extend(path.iter().map(|&i| i as u32));
                                path_off[p + 1] = path_idx.len() as u64;
                            }
                        }
                        path_idx.push(0);
                        let h = b2a_band_hints {
                            match_off: match_off.as_ptr(),
                            match_xy: match_xy.as_ptr(),
                            path_off: if paths.is_some() { path_off.as_ptr() } else { std::ptr::null() },
                            path_idx: if paths.is_some() { path_idx.as_ptr() } else { std::ptr::null() },
                            allowed_mismatches: allowed_mismatches.map(|v| v as i32).unwrap_or(-1),
                            use_lcskpp_union: use_lcskpp_union as i32,
                        };
                        unsafe {
                            b2a_align_batch_banded_hinted(self.engine, mode, &cs, k, w, &cp, &h, &mut res, std::ptr::null_mut())
                        }
                    }
                };
                if rc != 0 {
                    let msg = unsafe { CStr::from_ptr(b2a_last_error(self.engine)) }.to_string_lossy().into_owned();
                    panic!("{}", msg); // the reference panics on the same conditions (assert!, mod.rs:905)
                }
                let amode = match mode {
                    1 => AlignmentMode::Global,
                    2 => AlignmentMode::Semiglobal,
                    3 => AlignmentMode::Local,
                    _ => AlignmentMode::Custom,
                };
                (0..n)
                    .map(|p| {
                        let mut k = 0;
                        let operations = ops[ops_off[p] as usize..ops_off[p + 1] as usize]
                            .iter()
                            .map(|c| match c {
                                0 => AlignmentOperation::Match,
                                1 => AlignmentOperation::Subst,
                                2 => AlignmentOperation::Del,
                                3 => AlignmentOperation::Ins,
                                4 => {
                                    k += 1;
                                    AlignmentOperation::Xclip(clip[4 * p + k - 1] as usize)
                                }
                                _ => {
                                    k += 1;
                                    AlignmentOperation::Yclip(clip[4 * p + k - 1] as usize)
                                }
                            })
                            .collect();
                        // banded.rs:407-420: a band above MAX_CELLS returns the empty alignment (score MIN_SCORE,
                        // xlen = ylen = 0); global/semiglobal/local then overwrite only `.mode` (banded.rs:889-890)
                        let operations: Vec<AlignmentOperation> = operations;
                        let refused = is_banded && score[p] == MIN_SCORE && operations.is_empty();
                        Alignment {
                            score: score[p],
                            ystart: ys[p] as usize,
                            xstart: xs[p] as usize,
                            yend: ye[p] as usize,
                            xend: xe[p] as usize,
                            ylen: if refused { 0 } else { pairs[p].1.len() },
                            xlen: if refused { 0 } else { pairs[p].0.len() },
                            operations,
                            mode: amode,
                        }
                    })
                    .collect()
            }

            /// Score-only batch (b2a_score_batch): (score, xend, yend) of the Alignment `batch` returns, without the
            /// traceback.  Panics where the reference would on the part of the walk it replays (include/b200align.h).
            pub(crate) fn scores(&mut self, mode: i32, pairs: &[(&[u8], &[u8])]) -> Vec<(i32, usize, usize)> {
                let n = pairs.len();
                let (mut x_off, mut y_off, mut x_len, mut y_len) = (Vec::with_capacity(n), Vec::with_capacity(n), Vec::with_capacity(n), Vec::with_capacity(n));
                let mut blob: Vec<u8> = Vec::new();
                let mut present = [false; 256];
                for (x, y) in pairs {
                    for (s, off) in [(x, &mut x_off), (y, &mut y_off)] {
                        while blob.len() % 16 != 0 {
                            blob.push(0);
                        }
                        off.push(blob.len() as u64);
                        blob.extend_from_slice(s);
                        for &b in s.iter() {
                            present[b as usize] = true;
                        }
                    }
                    x_len.push(x.len() as u32);
                    y_len.push(y.len() as u32);
                }
                let alphabet: Vec<u8> = (0..=255u8).filter(|b| present[*b as usize]).collect();
                let mut table = vec![0i32; 256 * 256];
                for &a in &alphabet {
                    for &b in &alphabet {
                        table[a as usize * 256 + b as usize] = self.scoring.match_fn.score(a, b);
                    }
                }
                let (ms, mm) = self.scoring.match_scores.unwrap_or((0, 0));
                let cs = b2a_scoring {
                    gap_open: self.scoring.gap_open,
                    gap_extend: self.scoring.gap_extend,
                    xclip_prefix: self.scoring.xclip_prefix,
                    xclip_suffix: self.scoring.xclip_suffix,
                    yclip_prefix: self.scoring.yclip_prefix,
                    yclip_suffix: self.scoring.yclip_suffix,
                    match_score: ms,
                    mismatch_score: mm,
                    has_match_scores: self.scoring.match_scores.is_some() as i32,
                    table: table.as_ptr(),
                    alphabet: alphabet.as_ptr(),
                    alphabet_len: alphabet.len() as u32,
                };
                let cp = b2a_pairs {
                    seq_blob: blob.as_ptr(),
                    x_off: x_off.as_ptr(),
                    x_len: x_len.as_ptr(),
                    y_off: y_off.as_ptr(),
                    y_len: y_len.as_ptr(),
                    blob_bytes: blob.len() as u64,
                    n_pairs: n as u64,
                };
                let (mut score, mut xe, mut ye) = (vec![0i32; n], vec![0u32; n], vec![0u32; n]);
                let mut res = b2a_score_results {
                    score: score.as_mut_ptr(),
                    xend: xe.as_mut_ptr(),
                    yend: ye.as_mut_ptr(),
                    status: std::ptr::null_mut(),
                };
                let rc = unsafe { b2a_score_batch(self.engine, mode, &cs, &cp, &mut res, std::ptr::null_mut()) };
                if rc != 0 {
                    let msg = unsafe { CStr::from_ptr(b2a_last_error(self.engine)) }.to_string_lossy().into_owned();
                    panic!("{}", msg);
                }
                (0..n).map(|p| (score[p], xe[p] as usize, ye[p] as usize)).collect()
            }

            pub fn custom_scores_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<(i32, usize, usize)> { self.scores(0, pairs) }
            pub fn global_scores_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<(i32, usize, usize)> { self.scores(1, pairs) }
            pub fn semiglobal_scores_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<(i32, usize, usize)> { self.scores(2, pairs) }
            pub fn local_scores_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<(i32, usize, usize)> { self.scores(3, pairs) }

            pub fn custom_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { self.batch(0, None, pairs) }
            pub fn global_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { self.batch(1, None, pairs) }
            pub fn semiglobal_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { self.batch(2, None, pairs) }
            pub fn local_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { self.batch(3, None, pairs) }

            /// mod.rs:591
            pub fn custom(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.batch(0, None, &[(x, y)]).remove(0) }
            /// mod.rs:925
            pub fn global(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.batch(1, None, &[(x, y)]).remove(0) }
            /// mod.rs:954
            pub fn semiglobal(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.batch(2, None, &[(x, y)]).remove(0) }
            /// mod.rs:986
            pub fn local(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.batch(3, None, &[(x, y)]).remove(0) }
        }

        // ------------------------------------------------------------ TracebackCell, mod.rs:1026-1114
        /// The reference's public packed traceback cell: three 4-bit move codes, I in the low nibble, then D, then S.
        /// The engine keeps its own 4-bit traceback on the device; this host type exists for callers that named it.
        #[derive(Default, Copy, Clone, Eq, PartialEq, Ord, PartialOrd, Hash, Debug)]
        pub struct TracebackCell {
            v: u16,
        }
        #[derive(Copy, Clone)]
        enum Layer {
            I = 0,
            D = 4,
            S = 8,
        }
        const LARGEST_MOVE: u16 = 8; // TB_YCLIP_SUFFIX
        impl TracebackCell {
            pub fn new() -> TracebackCell {
                TracebackCell { v: 0 }
            }
            fn put(&mut self, layer: Layer, code: u16) {
                assert!(code <= LARGEST_MOVE, "Expected a value <= TB_MAX while setting traceback bits");
                let shift = layer as u16;
                self.v &= !(0xF << shift);
                self.v |= code << shift;
            }
            fn take(self, layer: Layer) -> u16 {
                (self.v >> (layer as u16)) & 0xF
            }
            pub fn set_i_bits(&mut self, value: u16) { self.put(Layer::I, value) }
            pub fn set_d_bits(&mut self, value: u16) { self.put(Layer::D, value) }
            pub fn set_s_bits(&mut self, value: u16) { self.put(Layer::S, value) }
            pub fn get_i_bits(self) -> u16 { self.take(Layer::I) }
            pub fn get_d_bits(self) -> u16 { self.take(Layer::D) }
            pub fn get_s_bits(self) -> u16 { self.take(Layer::S) }
            pub fn set_all(&mut self, value: u16) {
                for layer in [Layer::I, Layer::D, Layer::S] {
                    self.put(layer, value);
                }
            }
        }

        // ------------------------------------------------------------ banded::Aligner, banded.rs:122-1004
        pub mod banded {
            use super::{Alignment, BandedCall, MatchFunc, Scoring};

            /// Same constructors and methods as `bio::alignment::pairwise::banded::Aligner` (k = k-mer length,
            /// w = band half-width, banded.rs:150-267); every method is a batch of one, `*_batch` is the GPU form.
            pub struct Aligner<F: MatchFunc> {
                inner: super::Aligner<F>,
                k: usize,
                w: usize,
            }

            impl<F: MatchFunc> Aligner<F> {
                pub fn new(gap_open: i32, gap_extend: i32, match_fn: F, k: usize, w: usize) -> Self {
                    Aligner { inner: super::Aligner::new(gap_open, gap_extend, match_fn), k, w }
                }
                pub fn with_capacity(m: usize, n: usize, gap_open: i32, gap_extend: i32, match_fn: F, k: usize, w: usize) -> Self {
                    Aligner { inner: super::Aligner::with_capacity(m, n, gap_open, gap_extend, match_fn), k, w }
                }
                pub fn with_scoring(scoring: Scoring<F>, k: usize, w: usize) -> Self {
                    Aligner { inner: super::Aligner::with_scoring(scoring), k, w }
                }
                pub fn with_capacity_and_scoring(m: usize, n: usize, scoring: Scoring<F>, k: usize, w: usize) -> Self {
                    Aligner { inner: super::Aligner::with_capacity_and_scoring(m, n, scoring), k, w }
                }
                pub fn get_mut_scoring(&mut self) -> &mut Scoring<F> {
                    &mut self.inner.scoring
                }
                fn call<'a>(&self) -> BandedCall<'a> {
                    BandedCall { k: self.k as u32, w: self.w as u32, matches: None, paths: None, allowed_mismatches: None, use_lcskpp_union: false }
                }

                pub fn custom_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { let c = self.call(); self.inner.batch(0, Some(c), pairs) }
                pub fn global_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { let c = self.call(); self.inner.batch(1, Some(c), pairs) }
                pub fn semiglobal_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { let c = self.call(); self.inner.batch(2, Some(c), pairs) }
                pub fn local_batch(&mut self, pairs: &[(&[u8], &[u8])]) -> Vec<Alignment> { let c = self.call(); self.inner.batch(3, Some(c), pairs) }
                /// banded.rs:282
                pub fn custom(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.custom_batch(&[(x, y)]).remove(0) }
                /// banded.rs:872
                pub fn global(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.global_batch(&[(x, y)]).remove(0) }
                /// banded.rs:901
                pub fn semiglobal(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.semiglobal_batch(&[(x, y)]).remove(0) }
                /// banded.rs:975
                pub fn local(&mut self, x: &[u8], y: &[u8]) -> Alignment { self.local_batch(&[(x, y)]).remove(0) }

                /// banded.rs:294 / 938: the prehash of y only spares the reference its own hashing; the matches
                /// (find_kmer_matches_seq2_hashed) and therefore the results are those of custom / semiglobal.
                pub fn custom_with_prehash<H>(&mut self, x: &[u8], y: &[u8], _y_kmer_hash: &H) -> Alignment { self.custom(x, y) }
                pub fn semiglobal_with_prehash<H>(&mut self, x: &[u8], y: &[u8], _y_kmer_hash: &H) -> Alignment { self.semiglobal(x, y) }

                /// banded.rs:313
                pub fn custom_with_matches(&mut self, x: &[u8], y: &[u8], matches: &[(u32, u32)]) -> Alignment {
                    self.custom_with_matches_batch(&[(x, y)], &[matches]).remove(0)
                }
                pub fn custom_with_matches_batch(&mut self, pairs: &[(&[u8], &[u8])], matches: &[&[(u32, u32)]]) -> Vec<Alignment> {
                    let mut c = self.call();
                    c.matches = Some(matches);
                    self.inner.batch(0, Some(c), pairs)
                }
                /// banded.rs:338
                pub fn custom_with_expanded_matches(&mut self, x: &[u8], y: &[u8], matches: Vec<(u32, u32)>,
                                                    allowed_mismatches: Option<usize>, use_lcskpp_union: bool) -> Alignment {
                    self.custom_with_expanded_matches_batch(&[(x, y)], &[&matches[..]], allowed_mismatches, use_lcskpp_union).remove(0)
                }
                pub fn custom_with_expanded_matches_batch(&mut self, pairs: &[(&[u8], &[u8])], matches: &[&[(u32, u32)]],
                                                          allowed_mismatches: Option<usize>, use_lcskpp_union: bool) -> Vec<Alignment> {
                    let mut c = self.call();
                    c.matches = Some(matches);
                    c.allowed_mismatches = allowed_mismatches;
                    c.use_lcskpp_union = use_lcskpp_union;
                    self.inner.batch(0, Some(c), pairs)
                }
                /// banded.rs:391
                pub fn custom_with_match_path(&mut self, x: &[u8], y: &[u8], matches: &[(u32, u32)], path: &[usize]) -> Alignment {
                    self.custom_with_match_path_batch(&[(x, y)], &[matches], &[path]).remove(0)
                }
                pub fn custom_with_match_path_batch(&mut self, pairs: &[(&[u8], &[u8])], matches: &[&[(u32, u32)]],
                                                    paths: &[&[usize]]) -> Vec<Alignment> {
                    let mut c = self.call();
                    c.matches = Some(matches);
                    c.paths = Some(paths);
                    self.inner.batch(0, Some(c), pairs)
                }
            }
        }
    }
}
