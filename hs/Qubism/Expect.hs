{-|
Module      : Qubism.Expect
Description : expectation values of Pauli strings, Pauli rotations, Pauli sums, adjoint gradients, exact
              time evolution and Lanczos ground states, computed on the device (qb_expect_pauli,
              qb_apply_pauli_rot, qb_pauli_sum, qb_pauli_rot_grad, qb_pauli_evolve, qb_pauli_ground)

@expectPauli terms sv@ is @[realPart (sv <.> (p #> sv)) | p <- terms]@ for the Pauli strings @p@ that
@terms@ name (QGate.hs:90-108 for pauliX / pauliY / pauliZ), without building any @p #> sv@: one
read-only sweep of the state per distinct X mask.  A pure observation: no clone, @sv@ keeps its value.
Not normalised, like the reference's @<.>@.

@pauliRotate rots sv@ applies @exp (-i theta/2 p)@ for each @(p, theta)@ of @rots@ in order, as a new value
(clone + in-place apply, like the other pure operations of the shim): one read + write sweep of the state per
run of rotations whose X qubits fit one tile together.

@pauliSum terms sv@ is @sum_t c_t (p_t #> sv)@ for the @(p_t, c_t)@ of @terms@, as a new value; @sv@ keeps its own.

@pauliRotGrad rots h sv@ is @(e, grad)@ with @e = sum_t h_t realPart (psi <.> (p_t #> psi))@ for
@psi = pauliRotate rots sv@ and @grad !! k = d e / d theta_k@ (the adjoint method: about one forward pass,
one @pauliSum@ and one backward pass, whatever the number of angles).

@pauliEvolve h t sv@ is @exp (-i t H) #> sv@ for @H = sum_t h_t p_t@ (real coefficients), as a new value: a
Chebyshev expansion exact to double precision (clone + in-place evolution).

@pauliGround h tol maxiter sv@ is @(e, x)@: the lowest Lanczos Ritz value @e@ of @H = sum_t h_t p_t@ on the
Krylov space of @sv@ (the lowest eigenvalue among the eigenvectors @sv@ overlaps), stopped once the Ritz
residual estimate is at most @tol@ or after @maxiter@ steps, and its normalised Ritz vector @x@ as a new value
(clone + in-place Lanczos).  UNVERIFIED BY COMPILATION (no GHC in the build image).
-}
{-# LANGUAGE DataKinds, KindSignatures, ScopedTypeVariables #-}
module Qubism.Expect
  ( Pauli (..)
  , expectPauli
  , pauliRotate
  , pauliSum
  , pauliRotGrad
  , pauliEvolve
  , pauliGround
  ) where

import GHC.TypeLits
import Data.Bits        (setBit, testBit, (.|.))
import Data.Complex     (Complex)
import Data.Finite      (Finite, getFinite)
import Data.Word        (Word64)
import Foreign
import System.IO.Unsafe (unsafePerformIO)

import Qubism.StateVec       (StateVec (UnsafeMkStateVec), withSV, cloneSV)
import Qubism.Backend.FFI

data Pauli = I | X | Y | Z deriving (Eq, Ord, Show, Read, Enum, Bounded)

-- | One term = the product of @onJust q p@ over its pairs; each qubit at most once (the rest are I).
expectPauli :: KnownNat n => [[(Finite n, Pauli)]] -> StateVec n -> [Double]
expectPauli terms sv = unsafePerformIO $
  withArrayLen xs $ \k px -> withArray zs $ \pz -> allocaArray k $ \po -> withSV sv $ \s -> do
    rc <- c_qb_expect_pauli s px pz (fromIntegral k) po
    if rc /= 0 then error ("qubism_sv: status " ++ show rc) else map realToFrac <$> peekArray k po
  where
    (xs, zs) = unzip (map masks terms)

-- | A string with X / Y on more than QB_PAULI_ROT_MAX_X (12) qubits is an error (QB_ERR_UNSUPPORTED).
pauliRotate :: KnownNat n => [([(Finite n, Pauli)], Double)] -> StateVec n -> StateVec n
pauliRotate rots sv = unsafePerformIO $ do
  r <- cloneSV sv
  withArrayLen xs $ \k px -> withArray zs $ \pz -> withArray (map realToFrac thetas) $ \pt -> withSV r $ \p -> do
    rc <- c_qb_apply_pauli_rot p px pz pt (fromIntegral k)
    if rc /= 0 then error ("qubism_sv: status " ++ show rc) else pure r
  where
    (terms, thetas) = unzip rots
    (xs, zs) = unzip (map masks terms)

pauliSum :: KnownNat n => [([(Finite n, Pauli)], Complex Double)] -> StateVec n -> StateVec n
pauliSum terms sv = unsafePerformIO $
  withArrayLen xs $ \k px -> withArray zs $ \pz -> withArray cs $ \pc -> withSV sv $ \p -> alloca $ \pp -> do
    rc <- c_qb_pauli_sum p px pz pc (fromIntegral k) pp
    if rc /= 0 then error ("qubism_sv: status " ++ show rc)
               else peek pp >>= fmap UnsafeMkStateVec . newForeignPtr p_qb_state_free
  where
    (ps, cs) = unzip terms
    (xs, zs) = unzip (map masks ps)

-- | Real coefficients: H is Hermitian.  The same strings are errors as for pauliRotate.
pauliRotGrad :: KnownNat n => [([(Finite n, Pauli)], Double)] -> [([(Finite n, Pauli)], Double)] -> StateVec n
             -> (Double, [Double])
pauliRotGrad rots h sv = unsafePerformIO $
  withArrayLen rxs $ \k prx -> withArray rzs $ \prz -> withArray (map realToFrac thetas) $ \pt ->
  withArrayLen hxs $ \m phx -> withArray hzs $ \phz -> withArray (map realToFrac hcs) $ \phc ->
  alloca $ \pe -> allocaArray k $ \pg -> withSV sv $ \p -> do
    rc <- c_qb_pauli_rot_grad p prx prz pt (fromIntegral k) phx phz phc (fromIntegral m) pe pg
    if rc /= 0 then error ("qubism_sv: status " ++ show rc)
               else (,) <$> (realToFrac <$> peek pe) <*> (map realToFrac <$> peekArray k pg)
  where
    (rterms, thetas) = unzip rots
    (rxs, rzs) = unzip (map masks rterms)
    (hterms, hcs) = unzip h
    (hxs, hzs) = unzip (map masks hterms)

-- | Real coefficients: H is Hermitian.  The same strings are errors as for pauliRotate.
pauliEvolve :: KnownNat n => [([(Finite n, Pauli)], Double)] -> Double -> StateVec n -> StateVec n
pauliEvolve h t sv = unsafePerformIO $ do
  r <- cloneSV sv
  withArrayLen xs $ \k px -> withArray zs $ \pz -> withArray (map realToFrac hcs) $ \pc -> withSV r $ \p -> do
    rc <- c_qb_pauli_evolve p px pz pc (fromIntegral k) (realToFrac t) nullPtr
    if rc /= 0 then error ("qubism_sv: status " ++ show rc) else pure r
  where
    (terms, hcs) = unzip h
    (xs, zs) = unzip (map masks terms)

-- | Real coefficients: H is Hermitian.  The same strings are errors as for pauliRotate.
pauliGround :: KnownNat n => [([(Finite n, Pauli)], Double)] -> Double -> Int -> StateVec n -> (Double, StateVec n)
pauliGround h tol maxiter sv = unsafePerformIO $ do
  r <- cloneSV sv
  withArrayLen xs $ \k px -> withArray zs $ \pz -> withArray (map realToFrac hcs) $ \pc -> withSV r $ \p ->
    alloca $ \pe -> alloca $ \pr -> alloca $ \pm -> do
      rc <- c_qb_pauli_ground p px pz pc (fromIntegral k) (realToFrac tol) (fromIntegral maxiter) 1 pe pr pm
                              nullPtr nullPtr
      if rc /= 0 then error ("qubism_sv: status " ++ show rc) else (\e -> (realToFrac e, r)) <$> peek pe
  where
    (terms, hcs) = unzip h
    (xs, zs) = unzip (map masks terms)

-- bit q of the X / Z mask = qubit q: X = x only, Z = z only, Y = both
masks :: [(Finite n, Pauli)] -> (Word64, Word64)
masks = foldr add (0, 0)
  where
    add (q, p) (x, z)
      | testBit (x .|. z) i = error "expectPauli: a qubit appears twice in one term"
      | otherwise = case p of
          I -> (x, z)
          X -> (setBit x i, z)
          Y -> (setBit x i, setBit z i)
          Z -> (x, setBit z i)
      where i = fromIntegral (getFinite q)
