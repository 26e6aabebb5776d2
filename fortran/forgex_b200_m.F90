! forgex_b200_m -- ISO_C_BINDING interface to libforgex_b200.so (include/forgex_b200.h) and the batch forms
! that Forgex's Fortran API gains on top of it.
!
! STATUS: UNVERIFIED.  This image has no Fortran front end (no gfortran / flang / nvfortran / ifx), here or on
! the GPU box, so this file has never been compiled.  It is kept deliberately thin: every procedure is one
! interface block or a few lines of marshalling around a C entry point that IS exercised by the Python and C
! tests.  INTEGRATION.md shows where it plugs into the reference (src/forgex.F90, src/api_internal_m.F90).
!
! What stays as it is in Forgex: operator(.in.), operator(.match.), regex, regex_f, is_valid_regex
! (src/forgex.F90:24-54).  What is new: a compiled-pattern handle and batch generics
!     fx_pattern_t            compile once (the reference recompiles per call: src/forgex.F90:98, :139-140)
!     match_batch / in_batch  one pattern against n fixed-length strings (character(len=*) :: strs(:)) or against
!                             a flat buffer + offsets (variable length; trailing blanks are text to Forgex)
!     regex_batch             (from, to) per string
!     regex_buffer            one pattern against one huge buffer, 64-bit positions
!     regex_count_batch / regex_all_batch / regex_buffer_all   every match, the way a caller loops regex on text(to+1:)
!     is_valid_regex_batch    is_valid_regex over an array of patterns, one call
!     *_dev / window forms    device pointers (type(c_ptr)) + a CUDA stream, for CUDA Fortran / OpenACC hosts and for
!                             a text that is split across GPUs
!
! `pure`: Forgex's operators are `pure elemental` and `regex` is a `pure subroutine` (src/forgex.F90:24-54).  A bind(C)
! interface body may be declared PURE -- the declaration is the programmer's promise, the compiler does not look into
! the C code -- but a pure FUNCTION may only have intent(in) / value dummies.  The C ABI therefore has value-returning
! forms of the two operators (fx_in_value, fx_match_value) and a subroutine-shaped regex (fx_regex_sub); they are
! declared pure below, so the operators keep every attribute they have today (INTEGRATION.md 2.1).  The promise holds
! in the sense Fortran cares about: no Fortran-visible state is touched; the calls allocate and free device memory
! internally and are re-entrant.
module forgex_b200_m
   use, intrinsic :: iso_c_binding
   use, intrinsic :: iso_fortran_env, only: int64
   implicit none
   private

   integer(c_int), parameter, public :: FX_OP_MATCH = 0, FX_OP_IN = 1, FX_OP_REGEX = 2
   integer(c_int), parameter, public :: FX_OK = 0
   integer(c_int), parameter, public :: FX_ERR_TREE_NODE_LIMIT = 101, FX_ERR_DFA_STATE_CAP = 102, &
                                        FX_ERR_PREFILTER_UNSUPPORTED = 103, FX_ERR_BAD_ARGUMENT = 104, &
                                        FX_ERR_NO_DEVICE = 105, FX_ERR_WORK_BUDGET = 106

   type, public :: fx_pattern_t
      type(c_ptr) :: handle = c_null_ptr
      integer(c_int) :: status = -1
   contains
      procedure :: compile => pattern__compile
      procedure :: free    => pattern__free
   end type fx_pattern_t

   public :: match_batch, in_batch, regex_batch, regex_buffer, regex_count_batch, regex_all_batch, regex_buffer_all, &
             is_valid_regex_batch

   interface match_batch
      module procedure :: match_batch__fixed, match_batch__ragged
   end interface
   interface in_batch
      module procedure :: in_batch__fixed, in_batch__ragged
   end interface

   ! ---- C entry points (include/forgex_b200.h) -------------------------------------------------------
   interface
      function fx_compile(pattern, plen, op, out) bind(c, name='fx_compile') result(status)
         import :: c_char, c_int64_t, c_int, c_ptr
         character(kind=c_char), intent(in) :: pattern(*)
         integer(c_int64_t), value :: plen
         integer(c_int), value :: op
         type(c_ptr), intent(out) :: out
         integer(c_int) :: status
      end function
      function fx_pattern_free(p) bind(c, name='fx_pattern_free') result(status)
         import :: c_ptr, c_int
         type(c_ptr), value :: p
         integer(c_int) :: status
      end function
      function fx_match_fixed(p, buf, n, stride, out) bind(c, name='fx_match_fixed') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int8_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), value :: n, stride
         integer(c_int8_t), intent(out) :: out(*)
         integer(c_int) :: status
      end function
      function fx_in_fixed(p, buf, n, stride, out) bind(c, name='fx_in_fixed') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int8_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), value :: n, stride
         integer(c_int8_t), intent(out) :: out(*)
         integer(c_int) :: status
      end function
      function fx_match_batch(p, buf, offsets, n, out) bind(c, name='fx_match_batch') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int8_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n
         integer(c_int8_t), intent(out) :: out(*)
         integer(c_int) :: status
      end function
      function fx_in_batch(p, buf, offsets, n, out) bind(c, name='fx_in_batch') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int8_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n
         integer(c_int8_t), intent(out) :: out(*)
         integer(c_int) :: status
      end function
      function fx_regex_batch(p, buf, offsets, n, from, to) bind(c, name='fx_regex_batch') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n
         integer(c_int64_t), intent(out) :: from(*), to(*)
         integer(c_int) :: status
      end function
      function fx_regex_buffer(p, buf, length, from, to) bind(c, name='fx_regex_buffer') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), value :: length
         integer(c_int64_t), intent(out) :: from, to
         integer(c_int) :: status
      end function
      ! one pattern, one text: drop-in bodies for operator__in / operator__match / subroutine__regex
      function fx_in(pattern, plen, text, tlen, res) bind(c, name='fx_in') result(status)
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int), intent(out) :: res
         integer(c_int) :: status
      end function
      function fx_match(pattern, plen, text, tlen, res) bind(c, name='fx_match') result(status)
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int), intent(out) :: res
         integer(c_int) :: status
      end function
      function fx_regex(pattern, plen, text, tlen, from, to, length, syntax_status) bind(c, name='fx_regex') result(status)
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int64_t), intent(out) :: from, to, length
         integer(c_int), intent(out) :: syntax_status
         integer(c_int) :: status
      end function
      ! ---- pure forms for the existing pure operators (see the header comment) ----
      pure function fx_in_value(pattern, plen, text, tlen) bind(c, name='fx_in_value') result(res)
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int) :: res                      ! 1 / 0, negative = -status
      end function
      pure function fx_match_value(pattern, plen, text, tlen) bind(c, name='fx_match_value') result(res)
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int) :: res
      end function
      pure subroutine fx_regex_sub(pattern, plen, text, tlen, from, to, length, syntax_status, rc) bind(c, name='fx_regex_sub')
         import :: c_char, c_int64_t, c_int
         character(kind=c_char), intent(in) :: pattern(*), text(*)
         integer(c_int64_t), value :: plen, tlen
         integer(c_int64_t), intent(out) :: from, to, length
         integer(c_int), intent(out) :: syntax_status, rc
      end subroutine
      pure function fx_is_valid_regex(pattern, plen, status) bind(c, name='fx_is_valid_regex') result(valid)
         import :: c_char, c_int64_t, c_int, c_ptr
         character(kind=c_char), intent(in) :: pattern(*)
         integer(c_int64_t), value :: plen
         type(c_ptr), value :: status                ! c_null_ptr: not wanted (keeps the function pure)
         integer(c_int) :: valid
      end function
      function fx_is_valid_regex_batch(patterns, offsets, n, valid, status) bind(c, name='fx_is_valid_regex_batch') result(rc)
         import :: c_char, c_int64_t, c_int8_t, c_int32_t, c_int
         character(kind=c_char), intent(in) :: patterns(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n
         integer(c_int8_t), intent(out) :: valid(*)
         integer(c_int32_t), intent(out) :: status(*)
         integer(c_int) :: rc
      end function
      ! ---- all matches / counts ----
      function fx_regex_count_batch(p, buf, offsets, n, counts) bind(c, name='fx_regex_count_batch') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n
         integer(c_int64_t), intent(out) :: counts(*)
         integer(c_int) :: status
      end function
      function fx_regex_buffer_all(p, buf, length, from, to, capacity, count) bind(c, name='fx_regex_buffer_all') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), value :: length, capacity
         integer(c_int64_t), intent(out) :: from(*), to(*), count
         integer(c_int) :: status
      end function
      function fx_regex_all_batch(p, buf, offsets, n, rows, from, to, capacity) bind(c, name='fx_regex_all_batch') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int
         type(c_ptr), value :: p
         character(kind=c_char), intent(in) :: buf(*)
         integer(c_int64_t), intent(in) :: offsets(*)
         integer(c_int64_t), value :: n, capacity
         integer(c_int64_t), intent(out) :: rows(*)
         integer(c_int64_t), intent(inout) :: from(*), to(*)      ! only the first min(rows(n+1), capacity) are written
         integer(c_int) :: status
      end function
      ! ---- device-pointer forms: buffers are type(c_ptr) device addresses (c_loc of a CUDA Fortran device array,
      !      acc_deviceptr, ...), stream = a cudaStream_t as c_ptr (c_null_ptr = default stream); asynchronous ----
      function fx_match_fixed_dev(p, d_buf, n, stride, d_out, stream) bind(c, name='fx_match_fixed_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_out, stream
         integer(c_int64_t), value :: n, stride
         integer(c_int) :: status
      end function
      function fx_in_fixed_dev(p, d_buf, n, stride, d_out, stream) bind(c, name='fx_in_fixed_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_out, stream
         integer(c_int64_t), value :: n, stride
         integer(c_int) :: status
      end function
      function fx_match_batch_dev(p, d_buf, d_offsets, n, total_bytes, d_out, stream) bind(c, name='fx_match_batch_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_offsets, d_out, stream
         integer(c_int64_t), value :: n, total_bytes
         integer(c_int) :: status
      end function
      function fx_in_batch_dev(p, d_buf, d_offsets, n, total_bytes, d_out, stream) bind(c, name='fx_in_batch_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_offsets, d_out, stream
         integer(c_int64_t), value :: n, total_bytes
         integer(c_int) :: status
      end function
      function fx_regex_batch_dev(p, d_buf, d_offsets, n, total_bytes, d_from, d_to, stream) bind(c, name='fx_regex_batch_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_offsets, d_from, d_to, stream
         integer(c_int64_t), value :: n, total_bytes
         integer(c_int) :: status
      end function
      function fx_regex_count_batch_dev(p, d_buf, d_offsets, n, total_bytes, d_counts, stream) bind(c, name='fx_regex_count_batch_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_offsets, d_counts, stream
         integer(c_int64_t), value :: n, total_bytes
         integer(c_int) :: status
      end function
      function fx_regex_buffer_work_bytes(length) bind(c, name='fx_regex_buffer_work_bytes') result(nbytes)
         import :: c_int64_t
         integer(c_int64_t), value :: length
         integer(c_int64_t) :: nbytes
      end function
      function fx_regex_buffer_dev(p, d_buf, length, d_from_to, d_work, stream) bind(c, name='fx_regex_buffer_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_from_to, d_work, stream
         integer(c_int64_t), value :: length
         integer(c_int) :: status
      end function
      function fx_regex_buffer_all_dev(p, d_buf, length, d_from, d_to, capacity, count, d_work, stream) &
            bind(c, name='fx_regex_buffer_all_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_from, d_to, d_work, stream
         integer(c_int64_t), value :: length, capacity
         integer(c_int64_t), intent(out) :: count          ! host memory
         integer(c_int) :: status
      end function
      function fx_regex_all_batch_work_bytes(n) bind(c, name='fx_regex_all_batch_work_bytes') result(nbytes)
         import :: c_int64_t
         integer(c_int64_t), value :: n
         integer(c_int64_t) :: nbytes
      end function
      function fx_regex_all_batch_dev(p, d_buf, d_offsets, n, total_bytes, d_rows, d_from, d_to, capacity, d_work, stream) &
            bind(c, name='fx_regex_all_batch_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_buf, d_offsets, d_rows, d_from, d_to, d_work, stream
         integer(c_int64_t), value :: n, total_bytes, capacity
         integer(c_int) :: status
      end function
      ! ---- window forms: one text split across GPUs (one MPI rank / coarray image per GPU; see INTEGRATION.md 3) ----
      function fx_buffer_scan_dev(p, d_window, window_len, start_lo, start_hi, origin, is_first, is_last, d_best, stream) &
            bind(c, name='fx_buffer_scan_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_window, d_best, stream
         integer(c_int64_t), value :: window_len, start_lo, start_hi, origin
         integer(c_int), value :: is_first, is_last
         integer(c_int) :: status
      end function
      function fx_buffer_scan_all_dev(p, d_window, window_len, start_lo, start_hi, origin, is_first, is_last, d_best, stream) &
            bind(c, name='fx_buffer_scan_all_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_window, d_best, stream
         integer(c_int64_t), value :: window_len, start_lo, start_hi, origin
         integer(c_int), value :: is_first, is_last
         integer(c_int) :: status
      end function
      function fx_buffer_finish_dev(p, d_window, window_len, origin, is_last, d_key, d_from_to, stream) &
            bind(c, name='fx_buffer_finish_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_window, d_key, d_from_to, stream
         integer(c_int64_t), value :: window_len, origin
         integer(c_int), value :: is_last
         integer(c_int) :: status
      end function
      ! linear-time window form (UNVERIFIED like the rest of this module): slab map per rank, the host combine of the
      ! gathered maps (FX_STATEMAP_MAP_WORDS = 98 int64 per rank), the backward walk (FX_STATEMAP_WALK_WORDS = 4 int64)
      function fx_statemap_window_dev(p, d_window, window_len, slab_lo, slab_hi, origin, d_map, d_work, stream) &
            bind(c, name='fx_statemap_window_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_window, d_map, d_work, stream
         integer(c_int64_t), value :: window_len, slab_lo, slab_hi, origin
         integer(c_int) :: status
      end function
      function fx_statemap_combine(p, maps, nmaps, text_len, out) bind(c, name='fx_statemap_combine') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p
         integer(c_int64_t), intent(in) :: maps(*)
         integer(c_int64_t), value :: nmaps, text_len
         integer(c_int64_t), intent(out) :: out(2)
         integer(c_int) :: status
      end function
      function fx_statemap_back_dev(p, d_window, window_len, origin, text_len, d_walk, stream) &
            bind(c, name='fx_statemap_back_dev') result(status)
         import :: c_ptr, c_int64_t, c_int
         type(c_ptr), value :: p, d_window, d_walk, stream
         integer(c_int64_t), value :: window_len, origin, text_len
         integer(c_int) :: status
      end function
      ! ---- the Fortran-side compile route (forgex_b200_tables_m) ----
      function fx_compile_from_dfa(op, cuts, ncls, delta, nstates, accept, q0, all, all_len, prefix, prefix_len, &
                                   suffix, suffix_len, out) bind(c, name='fx_compile_from_dfa') result(status)
         import :: c_ptr, c_char, c_int64_t, c_int32_t, c_int8_t, c_int
         integer(c_int), value :: op
         integer(c_int32_t), intent(in) :: cuts(*), delta(*)
         integer(c_int32_t), value :: ncls, nstates, q0
         integer(c_int8_t), intent(in) :: accept(*)
         character(kind=c_char), intent(in) :: all(*), prefix(*), suffix(*)
         integer(c_int64_t), value :: all_len, prefix_len, suffix_len
         type(c_ptr), intent(out) :: out
         integer(c_int) :: status
      end function
   end interface
   public :: fx_in, fx_match, fx_regex, fx_in_value, fx_match_value, fx_regex_sub, fx_is_valid_regex, fx_compile_from_dfa
   public :: fx_match_fixed_dev, fx_in_fixed_dev, fx_match_batch_dev, fx_in_batch_dev, fx_regex_batch_dev, fx_regex_count_batch_dev
   public :: fx_regex_buffer_work_bytes, fx_regex_buffer_dev, fx_regex_buffer_all_dev
   public :: fx_regex_all_batch_work_bytes, fx_regex_all_batch_dev
   public :: fx_buffer_scan_dev, fx_buffer_scan_all_dev, fx_buffer_finish_dev
   public :: fx_statemap_window_dev, fx_statemap_combine, fx_statemap_back_dev

contains

   subroutine pattern__compile(self, pattern, op)
      class(fx_pattern_t), intent(inout) :: self
      character(*), intent(in) :: pattern      ! NOT trimmed here: each entry point applies Forgex's own
      integer(c_int), intent(in) :: op          ! preprocessing (src/forgex.F90:95, :182-190, :260) inside fx_compile
      self%status = fx_compile(pattern, int(len(pattern), c_int64_t), op, self%handle)
   end subroutine pattern__compile

   subroutine pattern__free(self)
      class(fx_pattern_t), intent(inout) :: self
      integer(c_int) :: ignore
      if (c_associated(self%handle)) ignore = fx_pattern_free(self%handle)
      self%handle = c_null_ptr
   end subroutine pattern__free

   ! fixed-length strings: a Fortran character array is already one contiguous buffer of n*len bytes
   subroutine match_batch__fixed(pat, strs, res, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in), contiguous :: strs(:)
      logical, intent(out) :: res(:)
      integer, intent(out) :: status
      integer(c_int8_t), allocatable :: out(:)
      allocate(out(size(strs)))
      status = fx_match_fixed(pat%handle, strs, int(size(strs), c_int64_t), int(len(strs), c_int64_t), out)
      res = out /= 0
   end subroutine match_batch__fixed

   subroutine in_batch__fixed(pat, strs, res, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in), contiguous :: strs(:)
      logical, intent(out) :: res(:)
      integer, intent(out) :: status
      integer(c_int8_t), allocatable :: out(:)
      allocate(out(size(strs)))
      status = fx_in_fixed(pat%handle, strs, int(size(strs), c_int64_t), int(len(strs), c_int64_t), out)
      res = out /= 0
   end subroutine in_batch__fixed

   ! variable-length strings: flat buffer + offsets(0:n), 0-based byte offsets, offsets(0) = 0
   subroutine match_batch__ragged(pat, buf, offsets, res, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(in) :: offsets(0:)
      logical, intent(out) :: res(:)
      integer, intent(out) :: status
      integer(c_int8_t), allocatable :: out(:)
      allocate(out(size(res)))
      status = fx_match_batch(pat%handle, buf, offsets, int(size(res), c_int64_t), out)
      res = out /= 0
   end subroutine match_batch__ragged

   subroutine in_batch__ragged(pat, buf, offsets, res, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(in) :: offsets(0:)
      logical, intent(out) :: res(:)
      integer, intent(out) :: status
      integer(c_int8_t), allocatable :: out(:)
      allocate(out(size(res)))
      status = fx_in_batch(pat%handle, buf, offsets, int(size(res), c_int64_t), out)
      res = out /= 0
   end subroutine in_batch__ragged

   subroutine regex_batch(pat, buf, offsets, from, to, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(in) :: offsets(0:)
      integer(int64), intent(out) :: from(:), to(:)    ! 1-based inclusive, relative to each string; 0/0 = no match
      integer, intent(out) :: status
      status = fx_regex_batch(pat%handle, buf, offsets, int(size(from), c_int64_t), from, to)
   end subroutine regex_batch

   subroutine regex_buffer(pat, buf, from, to, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(out) :: from, to           ! 64-bit: the reference's default-integer indices stop at 2 GiB
      integer, intent(out) :: status
      status = fx_regex_buffer(pat%handle, buf, int(len(buf, kind=int64), c_int64_t), from, to)
   end subroutine regex_buffer

   ! matches per string, counted the way a caller loops `regex` on text(to+1:) (README.md:197-222)
   subroutine regex_count_batch(pat, buf, offsets, counts, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(in) :: offsets(0:)
      integer(int64), intent(out) :: counts(:)
      integer, intent(out) :: status
      status = fx_regex_count_batch(pat%handle, buf, offsets, int(size(counts), c_int64_t), counts)
   end subroutine regex_count_batch

   ! every match of every string: string i's spans are from(rows(i-1)+1 : rows(i)), to(...) (rows(0:n), rows(0) = 0),
   ! in the string's own coordinates; rows is always complete, at most min(size(from), size(to)) spans are stored
   subroutine regex_all_batch(pat, buf, offsets, rows, from, to, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(in) :: offsets(0:)
      integer(int64), intent(out) :: rows(0:)
      integer(int64), intent(inout) :: from(:), to(:)
      integer, intent(out) :: status
      status = fx_regex_all_batch(pat%handle, buf, offsets, int(size(rows) - 1, c_int64_t), rows, from, to, &
                                  int(min(size(from), size(to)), c_int64_t))
   end subroutine regex_all_batch

   ! every match of one buffer, in order; at most size(from) spans are stored, count may be larger
   subroutine regex_buffer_all(pat, buf, from, to, count, status)
      type(fx_pattern_t), intent(in) :: pat
      character(len=*), intent(in) :: buf
      integer(int64), intent(out) :: from(:), to(:), count
      integer, intent(out) :: status
      status = fx_regex_buffer_all(pat%handle, buf, int(len(buf, kind=int64), c_int64_t), from, to, &
                                   int(min(size(from), size(to)), c_int64_t), count)
   end subroutine regex_buffer_all

   ! is_valid_regex over an array of patterns in one call; trailing blanks of an element are part of the element
   ! exactly as they are for the elemental is_valid_regex (src/forgex.F90:58-71 trims inside)
   subroutine is_valid_regex_batch(patterns, valid, codes)
      character(len=*), intent(in), contiguous :: patterns(:)
      logical, intent(out) :: valid(:)
      integer, intent(out), optional :: codes(:)
      integer(c_int64_t), allocatable :: offsets(:)
      integer(c_int8_t), allocatable :: v(:)
      integer(c_int32_t), allocatable :: st(:)
      integer :: i, rc
      allocate(offsets(0:size(patterns)), v(size(patterns)), st(size(patterns)))
      do i = 0, size(patterns)
         offsets(i) = int(i, c_int64_t) * len(patterns)
      end do
      rc = fx_is_valid_regex_batch(patterns, offsets, int(size(patterns), c_int64_t), v, st)
      valid = v /= 0
      if (present(codes)) codes = st
   end subroutine is_valid_regex_batch

end module forgex_b200_m
