{-|
Module      : Qubism.Expect
Description : expectation values of Pauli strings and Pauli rotations, computed on the device
              (qb_expect_pauli, qb_apply_pauli_rot)

@expectPauli terms sv@ is @[realPart (sv <.> (p #> sv)) | p <- terms]@ for the Pauli strings @p@ that
@terms@ name (QGate.hs:90-108 for pauliX / pauliY / pauliZ), without building any @p #> sv@: one
read-only sweep of the state per distinct X mask.  A pure observation: no clone, @sv@ keeps its value.
Not normalised, like the reference's @<.>@.

@pauliRotate rots sv@ applies @exp (-i theta/2 p)@ for each @(p, theta)@ of @rots@ in order, as a new value
(clone + in-place apply, like the other pure operations of the shim): one read + write sweep of the state per
run of rotations whose X qubits fit one tile together.  UNVERIFIED BY COMPILATION (no GHC in the build image).
-}
{-# LANGUAGE DataKinds, KindSignatures, ScopedTypeVariables #-}
module Qubism.Expect
  ( Pauli (..)
  , expectPauli
  , pauliRotate
  ) where

import GHC.TypeLits
import Data.Bits        (setBit, testBit, (.|.))
import Data.Finite      (Finite, getFinite)
import Data.Word        (Word64)
import Foreign
import System.IO.Unsafe (unsafePerformIO)

import Qubism.StateVec       (StateVec, withSV, cloneSV)
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
