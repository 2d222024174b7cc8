//! Replaces rofl_crypto/src/rand_proof_vec/mod.rs (keep errors.rs): create_randproof_vec :14-47, create_randproof_vec_existing :49-89, verify_randproof_vec :91-118.
use curve25519_dalek_ng::ristretto::RistrettoPoint;
use curve25519_dalek_ng::scalar::Scalar;

mod errors;
pub use self::errors::RandProofError;
use crate::b200::{self, ffi};
use crate::rand_proof::{ElGamalPair, ProofError, RandProof};

fn prove(value_vec: &Vec<f32>, existing: Option<&[u8]>, random_vec: &Vec<Scalar>) -> Result<(Vec<RandProof>, Vec<ElGamalPair>), RandProofError> {
    if value_vec.len() != random_vec.len() { return Err(RandProofError::WrongNumBlindingFactors); }
    let d = value_vec.len();
    let (mut proofs, mut pairs) = (vec![0u8; 128 * d], vec![0u8; 64 * d]);
    let bl = b200::scs(random_vec);
    let seed = b200::seed();
    let rc = unsafe {
        ffi::rofl_rand_prove(b200::ctx(), value_vec.as_ptr(), existing.map_or(std::ptr::null(), |e| e.as_ptr()), bl.as_ptr(), d, b200::n_bits(), b200::frac(), seed.as_ptr(),
                             proofs.as_mut_ptr(), pairs.as_mut_ptr())
    };
    if rc != 0 { panic!("rand proofs: rofl_b200 error {}: {}", rc, b200::last_error()); }
    Ok((proofs.chunks_exact(128).map(|p| RandProof::from_bytes(p).expect("malformed proof")).collect(),
        pairs.chunks_exact(64).map(|c| ElGamalPair::from_bytes(c).expect("malformed pair")).collect()))
}
pub fn create_randproof_vec(value_vec: &Vec<f32>, random_vec: &Vec<Scalar>) -> Result<(Vec<RandProof>, Vec<ElGamalPair>), RandProofError> { prove(value_vec, None, random_vec) }
pub fn create_randproof_vec_existing(value_vec: &Vec<f32>, existing_value_com_vec: Vec<RistrettoPoint>, random_vec: &Vec<Scalar>)
    -> Result<(Vec<RandProof>, Vec<ElGamalPair>), RandProofError> { prove(value_vec, Some(&b200::pts(&existing_value_com_vec)), random_vec) }

pub fn verify_randproof_vec(randproof_vec: &Vec<RandProof>, commit_vec: &Vec<ElGamalPair>) -> Result<bool, RandProofError> {
    if randproof_vec.len() != commit_vec.len() { return Err(RandProofError::WrongNumberOfElGamalPairs); }
    let (mut p, mut c) = (Vec::with_capacity(128 * randproof_vec.len()), Vec::with_capacity(64 * commit_vec.len()));
    for x in randproof_vec { p.extend_from_slice(&x.to_bytes()); }
    for x in commit_vec { c.extend_from_slice(&x.to_bytes()); }
    match unsafe { ffi::rofl_rand_verify(b200::ctx(), p.as_ptr(), c.as_ptr(), randproof_vec.len()) } {
        1 => Ok(true),
        0 => Ok(false),
        _ => Err(ProofError::FormatError.into()),
    }
}

/// Server side, the rand proofs of all clients of a round in one batched check (random linear combinations over every element; the reference
/// calls verify_randproof_vec once per client).  Every client must have the same number of elements.  One verdict per client, identical to
/// verify_randproof_vec's.
pub fn verify_randproof_vec_batch(randproofs: &[&Vec<RandProof>], commits: &[&Vec<ElGamalPair>]) -> Vec<Result<bool, RandProofError>> {
    let k = randproofs.len();
    assert!(k > 0 && commits.len() == k);
    let d = commits[0].len();
    let (mut p, mut c) = (Vec::with_capacity(128 * d * k), Vec::with_capacity(64 * d * k));
    for (ps, cs) in randproofs.iter().zip(commits) {
        if ps.len() != cs.len() || cs.len() != d { panic!("verify_randproof_vec_batch: every client needs {} proofs and pairs", d); }
        for x in ps.iter() { p.extend_from_slice(&x.to_bytes()); }
        for x in cs.iter() { c.extend_from_slice(&x.to_bytes()); }
    }
    let mut ok = vec![0i32; k];
    let seed = b200::seed();
    let rc = unsafe { ffi::rofl_rand_verify_batch(b200::ctx(), k, p.as_ptr(), c.as_ptr(), d, seed.as_ptr(), ok.as_mut_ptr()) };
    assert!(rc == 0, "verify_randproof_vec_batch: rofl_b200 error {}: {}", rc, b200::last_error());
    ok.into_iter().map(|r| match r { 1 => Ok(true), 0 => Ok(false), _ => Err(ProofError::FormatError.into()) }).collect()
}
