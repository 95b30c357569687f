{-|
Module      : Qubism.Backend.FFI
Description : foreign import ccall bindings of include/qubism_sv.h (libqubism_sv.so)

UNVERIFIED BY COMPILATION: there is no GHC in the build image (SURVEY.md 8c).  Kept small and
mechanical on purpose; every binding is one line of the C header.
-}
{-# LANGUAGE ForeignFunctionInterface #-}
module Qubism.Backend.FFI where

import Data.Complex        (Complex)
import Data.Int            (Int64)
import Data.Word           (Word64)
import Foreign.C.String    (CString)
import Foreign.C.Types
import Foreign.ForeignPtr  (FinalizerPtr)
import Foreign.Ptr         (Ptr)

data QbCtx
data QbState
type C = Complex Double   -- Storable (Complex Double) == qb_c64 (re, im)

-- context -------------------------------------------------------------------------------
foreign import ccall safe   "qb_init"            c_qb_init        :: CInt -> Ptr (Ptr QbCtx) -> IO CInt
foreign import ccall safe   "qb_shutdown"        c_qb_shutdown    :: Ptr QbCtx -> IO CInt
foreign import ccall unsafe "qb_last_error"      c_qb_last_error  :: IO CString
-- state lifetime ------------------------------------------------------------------------
foreign import ccall safe   "qb_state_create"    c_qb_state_create    :: Ptr QbCtx -> CInt -> CInt -> Ptr (Ptr QbState) -> IO CInt
foreign import ccall safe   "qb_state_from_host" c_qb_state_from_host :: Ptr QbCtx -> CInt -> Ptr C -> Ptr (Ptr QbState) -> IO CInt
foreign import ccall safe   "qb_state_clone"     c_qb_state_clone     :: Ptr QbState -> Ptr (Ptr QbState) -> IO CInt
foreign import ccall        "&qb_state_free"     p_qb_state_free      :: FinalizerPtr QbState
foreign import ccall unsafe "qb_state_nqubits"   c_qb_state_nqubits   :: Ptr QbState -> IO CInt
foreign import ccall safe   "qb_state_read"      c_qb_state_read      :: Ptr QbState -> Word64 -> Word64 -> Ptr C -> IO CInt
-- gates (enqueue only: cheap, but they take the context mutex, so `safe`) ----------------
foreign import ccall safe   "qb_apply_1q"        c_qb_apply_1q        :: Ptr QbState -> CInt -> Ptr C -> IO CInt
foreign import ccall safe   "qb_apply_1q_range"  c_qb_apply_1q_range  :: Ptr QbState -> CInt -> CInt -> Ptr C -> IO CInt
foreign import ccall safe   "qb_apply_ctrl_1q"   c_qb_apply_ctrl_1q   :: Ptr QbState -> Ptr CInt -> CInt -> CInt -> Ptr C -> IO CInt
foreign import ccall safe   "qb_apply_cnot"      c_qb_apply_cnot      :: Ptr QbState -> CInt -> CInt -> IO CInt
foreign import ccall safe   "qb_apply_kq"        c_qb_apply_kq        :: Ptr QbState -> Ptr CInt -> CInt -> Ptr C -> Ptr CInt -> CInt -> IO CInt
foreign import ccall safe   "qb_flush"           c_qb_flush           :: Ptr QbState -> IO CInt
-- measurement ---------------------------------------------------------------------------
foreign import ccall safe   "qb_sumsq"           c_qb_sumsq           :: Ptr QbState -> CInt -> Ptr CDouble -> Ptr CDouble -> IO CInt
foreign import ccall safe   "qb_collapse"        c_qb_collapse        :: Ptr QbState -> CInt -> CInt -> IO CInt
foreign import ccall safe   "qb_measure_qubit"   c_qb_measure_qubit   :: Ptr QbState -> CInt -> CDouble -> Ptr CInt -> Ptr CDouble -> IO CInt
-- vector space / Hilbert space ----------------------------------------------------------
-- (qb_c64 by value is passed as two doubles: a tiny C shim `qb_scale_ri(s, re, im)` is the
--  portable spelling when the platform ABI is in doubt)
foreign import ccall safe   "qb_axpy_ri"         c_qb_axpy_ri         :: Ptr QbState -> CDouble -> CDouble -> Ptr QbState -> IO CInt
foreign import ccall safe   "qb_scale_ri"        c_qb_scale_ri        :: Ptr QbState -> CDouble -> CDouble -> IO CInt
foreign import ccall safe   "qb_neg"             c_qb_neg             :: Ptr QbState -> IO CInt
foreign import ccall safe   "qb_dotc"            c_qb_dotc            :: Ptr QbState -> Ptr QbState -> Ptr C -> IO CInt
foreign import ccall safe   "qb_norm2"           c_qb_norm2           :: Ptr QbState -> Ptr CDouble -> IO CInt
foreign import ccall safe   "qb_normalize"       c_qb_normalize       :: Ptr QbState -> IO CInt
foreign import ccall safe   "qb_tensor"          c_qb_tensor          :: Ptr QbState -> Ptr QbState -> Ptr (Ptr QbState) -> IO CInt
-- observables -----------------------------------------------------------------------------
foreign import ccall safe   "qb_expect_pauli"    c_qb_expect_pauli    :: Ptr QbState -> Ptr Word64 -> Ptr Word64 -> Int64 -> Ptr CDouble -> IO CInt
-- Pauli rotations ------------------------------------------------------------------------
foreign import ccall safe   "qb_apply_pauli_rot" c_qb_apply_pauli_rot :: Ptr QbState -> Ptr Word64 -> Ptr Word64 -> Ptr CDouble -> Int64 -> IO CInt
