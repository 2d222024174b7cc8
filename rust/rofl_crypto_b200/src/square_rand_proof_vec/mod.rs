//! Replaces rofl_crypto/src/square_rand_proof_vec/mod.rs (keep errors.rs): create_l2rangeproof_vec_existing :18-70, create_l2rangeproof_vec :72-127,
//! verify_l2rangeproof_vec :129-160 (SquareRandProof 192 B over SquareRandProofCommitments 96 B).
use curve25519_dalek_ng::ristretto::RistrettoPoint;
use curve25519_dalek_ng::scalar::Scalar;

pub mod errors;
pub use self::errors::L2RangeProofError;
use crate::b200::{self, ffi};
use crate::square_rand_proof::pedersen::SquareRandProofCommitments;
use crate::square_rand_proof::{ProofError, SquareRandProof};

fn prove(value_vec: &Vec<f32>, existing: Option<&[u8]>, r1: &Vec<Scalar>, r2: &Vec<Scalar>) -> Result<(Vec<SquareRandProof>, Vec<SquareRandProofCommitments>), L2RangeProofError> {
    if value_vec.len() != r1.len() { return Err(L2RangeProofError::WrongNumBlindingFactors); }
    let d = value_vec.len();
    let (mut proofs, mut commits) = (vec![0u8; 192 * d], vec![0u8; 96 * d]);
    let (b1, b2) = (b200::scs(r1), b200::scs(r2));
    let seed = b200::seed();
    let rc = unsafe {
        ffi::rofl_square_rand_prove(b200::ctx(), value_vec.as_ptr(), existing.map_or(std::ptr::null(), |e| e.as_ptr()), b1.as_ptr(), b2.as_ptr(), d, b200::n_bits(), b200::frac(),
                                    seed.as_ptr(), proofs.as_mut_ptr(), commits.as_mut_ptr())
    };
    if rc != 0 { panic!("square rand proofs: rofl_b200 error {}: {}", rc, b200::last_error()); }
    Ok((proofs.chunks_exact(192).map(|p| SquareRandProof::from_bytes(p).expect("malformed proof")).collect(),
        commits.chunks_exact(96).map(|c| SquareRandProofCommitments::from_bytes(c).expect("malformed commitments")).collect()))
}
pub fn create_l2rangeproof_vec_existing(value_vec: &Vec<f32>, value_com_vec: Vec<RistrettoPoint>, random_vec: &Vec<Scalar>, random_vec_2: &Vec<Scalar>)
    -> Result<(Vec<SquareRandProof>, Vec<SquareRandProofCommitments>), L2RangeProofError> { prove(value_vec, Some(&b200::pts(&value_com_vec)), random_vec, random_vec_2) }
pub fn create_l2rangeproof_vec(value_vec: &Vec<f32>, random_vec: &Vec<Scalar>, random_vec_2: &Vec<Scalar>)
    -> Result<(Vec<SquareRandProof>, Vec<SquareRandProofCommitments>), L2RangeProofError> { prove(value_vec, None, random_vec, random_vec_2) }

pub fn verify_l2rangeproof_vec(randproof_vec: &Vec<SquareRandProof>, commit_vec: &Vec<SquareRandProofCommitments>) -> Result<bool, L2RangeProofError> {
    if randproof_vec.len() != commit_vec.len() { return Err(L2RangeProofError::WrongNumberOfElGamalPairs); }
    let (mut p, mut c) = (Vec::with_capacity(192 * randproof_vec.len()), Vec::with_capacity(96 * commit_vec.len()));
    for x in randproof_vec { p.extend_from_slice(&x.to_bytes()); }
    for x in commit_vec { c.extend_from_slice(&x.to_bytes()); }
    match unsafe { ffi::rofl_square_rand_verify(b200::ctx(), p.as_ptr(), c.as_ptr(), randproof_vec.len()) } {
        1 => Ok(true),
        0 => Ok(false),
        _ => Err(ProofError::FormatError.into()),
    }
}

/// Server side, the square-rand proofs of all clients of a round in one batched check (random linear combinations over every element; the
/// reference calls verify_l2rangeproof_vec once per client).  Every client must have the same number of elements.  One verdict per client,
/// identical to verify_l2rangeproof_vec's.
pub fn verify_l2rangeproof_vec_batch(randproofs: &[&Vec<SquareRandProof>], commits: &[&Vec<SquareRandProofCommitments>]) -> Vec<Result<bool, L2RangeProofError>> {
    let k = randproofs.len();
    assert!(k > 0 && commits.len() == k);
    let d = commits[0].len();
    let (mut p, mut c) = (Vec::with_capacity(192 * d * k), Vec::with_capacity(96 * d * k));
    for (ps, cs) in randproofs.iter().zip(commits) {
        if ps.len() != cs.len() || cs.len() != d { panic!("verify_l2rangeproof_vec_batch: every client needs {} proofs and commitments", d); }
        for x in ps.iter() { p.extend_from_slice(&x.to_bytes()); }
        for x in cs.iter() { c.extend_from_slice(&x.to_bytes()); }
    }
    let mut ok = vec![0i32; k];
    let seed = b200::seed();
    let rc = unsafe { ffi::rofl_square_rand_verify_batch(b200::ctx(), k, p.as_ptr(), c.as_ptr(), d, seed.as_ptr(), ok.as_mut_ptr()) };
    assert!(rc == 0, "verify_l2rangeproof_vec_batch: rofl_b200 error {}: {}", rc, b200::last_error());
    ok.into_iter().map(|r| match r { 1 => Ok(true), 0 => Ok(false), _ => Err(ProofError::FormatError.into()) }).collect()
}
