//! `crypto/bls/src/impls/b200.rs` — Lighthouse BLS backend on liblhb200.so (B200, sm_100a).
//!
//! Drop this file next to `impls/blst.rs`, add `pub mod b200;` to `impls/mod.rs` (behind `#[cfg(feature = "b200")]`), a
//! cargo feature `b200 = []` in `crypto/bls/Cargo.toml`, and in `crypto/bls/src/lib.rs`:
//!
//! ```ignore
//! #[cfg(feature = "b200")]
//! define_mod!(b200_implementations, crate::impls::b200::types);
//! #[cfg(all(feature = "b200", not(feature = "fake_crypto")))]
//! pub use b200_implementations::*;
//! // and in `enum Error`:   #[cfg(feature = "b200")] B200Error(i32),
//! ```
//!
//! Every trait of a backend is implemented: `TPublicKey`, `TAggregatePublicKey`, `TSignature`,
//! `TAggregateSignature`, `TSecretKey` and the free function `verify_signature_sets` (compare `impls/blst.rs`, whose line
//! numbers are cited at each method).  Point types hold canonical bytes, like `impls/fake_crypto.rs`; every group
//! operation is a call through the C ABI of `include/lhb200.h` (there is no CPU arithmetic here, and no fallback: a
//! non-zero status maps to `false` for verifications — fail closed — and to `Error::B200Error` for decoding).
//!
//! NOT COMPILED IN THIS REPOSITORY: the build image has no Rust toolchain.  The C ABI underneath is exercised, entry
//! point by entry point and against the oracle, from `tests/` (ctypes) and `tests/cpp` (C++).
#![cfg(feature = "b200")]

use crate::{
    generic_aggregate_public_key::TAggregatePublicKey,
    generic_aggregate_signature::TAggregateSignature,
    generic_public_key::{
        GenericPublicKey, TPublicKey, PUBLIC_KEY_BYTES_LEN, PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN,
    },
    generic_secret_key::{TSecretKey, SECRET_KEY_BYTES_LEN},
    generic_signature::{TSignature, SIGNATURE_BYTES_LEN},
    Error, Hash256, ZeroizeHash, INFINITY_SIGNATURE,
};
use rand::Rng;
use std::os::raw::c_char;
use std::sync::Once;

// ------------------------------------------------------------------------------------------------- C ABI (lhb200.h)
#[link(name = "lhb200")]
extern "C" {
    fn lhb200_init(device: i32) -> i32;
    #[allow(dead_code)]
    fn lhb200_last_error() -> *const c_char;
    fn lhb200_verify_signature_sets(
        sigs: *const u8,
        msgs: *const u8,
        pks: *const u8,
        pk_offsets: *const u32,
        rands: *const u64,
        n_sets: u32,
        ok: *mut u8,
        set_status: *mut u8,
    ) -> i32;
    fn lhb200_verify_signature_set_groups(
        sigs: *const u8,
        msgs: *const u8,
        pks: *const u8,
        pk_offsets: *const u32,
        rands: *const u64,
        n_sets: u32,
        group_offsets: *const u32,
        n_groups: u32,
        ok: *mut u8,
        set_status: *mut u8,
    ) -> i32;
    fn lhb200_aggregate_verify(sig96: *const u8, msgs: *const u8, pks96: *const u8, n: u32, ok: *mut u8) -> i32;
    fn lhb200_g2_aggregate(sigs96: *const u8, n: u32, out96: *mut u8) -> i32;
    fn lhb200_g1_aggregate(pks96: *const u8, n: u32, out48: *mut u8, out96: *mut u8) -> i32;
    fn lhb200_g1_decompress_validate(pk48: *const u8, n: u32, pk96: *mut u8, status: *mut u8) -> i32;
    fn lhb200_g1_deserialize_uncompressed(pks96: *const u8, n: u32, pk48: *mut u8, status: *mut u8) -> i32;
    fn lhb200_g2_decompress(sig96: *const u8, n: u32, out192: *mut u8, status: *mut u8) -> i32;
    fn lhb200_sk_to_pk(sk32: *const u8, n: u32, pk48: *mut u8, pk96: *mut u8) -> i32;
    fn lhb200_sign(sk32: *const u8, msg32: *const u8, n: u32, sig96: *mut u8) -> i32;
}

/// One process drives one GPU (`LHB200_DEVICE`, default 0).  Called lazily by every entry point.
fn ensure_init() -> bool {
    static INIT: Once = Once::new();
    static mut READY: bool = false;
    INIT.call_once(|| {
        let device = std::env::var("LHB200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        unsafe { READY = lhb200_init(device) == 0 };
    });
    unsafe { READY }
}

/// The group order r (big-endian), for `SecretKey::deserialize` (blst rejects scalars >= r).
const CURVE_ORDER_BE: [u8; 32] = [
    0x73, 0xed, 0xa7, 0x53, 0x29, 0x9d, 0x7d, 0x48, 0x33, 0x39, 0xd8, 0x08, 0x09, 0xa1, 0xd8, 0x05, 0x53, 0xbd, 0xa4, 0x02,
    0xff, 0xfe, 0x5b, 0xfe, 0xff, 0xff, 0xff, 0xff, 0x00, 0x00, 0x00, 0x01,
];

/// Provides the externally-facing, core BLS types.
pub mod types {
    pub use super::verify_signature_set_groups;
    pub use super::verify_signature_sets;
    pub use super::AggregatePublicKey;
    pub use super::AggregateSignature;
    pub use super::PublicKey;
    pub use super::SecretKey;
    pub use super::Signature;
    pub use super::SignatureSet;
}

pub type SignatureSet<'a> = crate::generic_signature_set::GenericSignatureSet<
    'a,
    PublicKey,
    AggregatePublicKey,
    Signature,
    AggregateSignature,
>;

// ------------------------------------------------------------------------------------------ verify_signature_sets
/// `impls/blst.rs:37-119`.  Sets are flattened into the SoA buffers of `lhb200_verify_signature_sets`; the library
/// draws the 64-bit blinding scalars itself (`rands = NULL`: ChaCha20 keyed from getrandom(2), zeros skipped).
pub fn verify_signature_sets<'a>(signature_sets: impl ExactSizeIterator<Item = &'a SignatureSet<'a>>) -> bool {
    let sets = signature_sets.collect::<Vec<_>>();
    if sets.is_empty() {
        return false; // blst.rs:42-44
    }
    let n = sets.len();
    let mut sigs = Vec::with_capacity(n * SIGNATURE_BYTES_LEN);
    let mut msgs = Vec::with_capacity(n * 32);
    let mut offsets: Vec<u32> = Vec::with_capacity(n + 1);
    let n_keys: usize = sets.iter().map(|s| s.signing_keys.len()).sum();
    let mut pks = Vec::with_capacity(n_keys * PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN);
    offsets.push(0);
    for set in &sets {
        match set.signature.point() {
            Some(point) => sigs.extend_from_slice(&point.0), // subgroup check happens on the device (blst.rs:73-77)
            None => return false,                            // "empty" signature (blst.rs:79-82)
        }
        if set.signing_keys.is_empty() {
            return false; // blst.rs:86-89
        }
        msgs.extend_from_slice(set.message.as_bytes());
        for pk in set.signing_keys.iter() {
            pks.extend_from_slice(&pk.point().uncompressed);
        }
        offsets.push((pks.len() / PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN) as u32);
    }
    if !ensure_init() {
        return false;
    }
    let mut ok = 0u8;
    let rc = unsafe {
        lhb200_verify_signature_sets(
            sigs.as_ptr(),
            msgs.as_ptr(),
            pks.as_ptr(),
            offsets.as_ptr(),
            std::ptr::null(),
            n as u32,
            &mut ok,
            std::ptr::null_mut(),
        )
    };
    rc == 0 && ok == 1
}

/// Many independent `verify_signature_sets` calls in one device pass (`lhb200_verify_signature_set_groups`): element g
/// is `verify_signature_sets(groups[g].iter())`, an empty group is false.  What the batch fallbacks of
/// `attestation_verification/batch.rs` need: one call that names the bad items.  Fails closed: any library error makes
/// every element false.  An "empty" signature or a set without keys fails its own group only (the device reports them).
pub fn verify_signature_set_groups(groups: &[&[SignatureSet]]) -> Vec<bool> {
    let n_groups = groups.len();
    let n: usize = groups.iter().map(|g| g.len()).sum();
    let mut sigs = Vec::with_capacity(n * SIGNATURE_BYTES_LEN);
    let mut msgs = Vec::with_capacity(n * 32);
    let mut offsets: Vec<u32> = Vec::with_capacity(n + 1);
    let mut group_offsets: Vec<u32> = Vec::with_capacity(n_groups + 1);
    let n_keys: usize = groups.iter().flat_map(|g| g.iter()).map(|s| s.signing_keys.len()).sum();
    let mut pks = Vec::with_capacity(n_keys * PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN);
    offsets.push(0);
    group_offsets.push(0);
    for group in groups {
        for set in group.iter() {
            match set.signature.point() {
                Some(point) => sigs.extend_from_slice(&point.0),
                None => sigs.extend_from_slice(&[0u8; SIGNATURE_BYTES_LEN]), // "empty": status 1 on the device
            }
            msgs.extend_from_slice(set.message.as_bytes());
            for pk in set.signing_keys.iter() {
                pks.extend_from_slice(&pk.point().uncompressed);
            }
            offsets.push((pks.len() / PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN) as u32);
        }
        group_offsets.push((offsets.len() - 1) as u32);
    }
    let mut ok = vec![0u8; n_groups];
    if n == 0 || !ensure_init() {
        return vec![false; n_groups];
    }
    let rc = unsafe {
        lhb200_verify_signature_set_groups(
            sigs.as_ptr(),
            msgs.as_ptr(),
            pks.as_ptr(),
            offsets.as_ptr(),
            std::ptr::null(),
            n as u32,
            group_offsets.as_ptr(),
            n_groups as u32,
            ok.as_mut_ptr(),
            std::ptr::null_mut(),
        )
    };
    ok.iter().map(|&v| rc == 0 && v == 1).collect()
}

/// One set, explicit keys: `Signature::verify` / `fast_aggregate_verify` (blst.rs:196-200, :250-261).
fn verify_one(sig: &[u8; SIGNATURE_BYTES_LEN], msg: Hash256, pks: &[&PublicKey]) -> bool {
    if pks.is_empty() || !ensure_init() {
        return false;
    }
    let mut flat = Vec::with_capacity(pks.len() * PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN);
    for pk in pks {
        flat.extend_from_slice(&pk.uncompressed);
    }
    let offsets = [0u32, pks.len() as u32];
    let mut ok = 0u8;
    let rc = unsafe {
        lhb200_verify_signature_sets(
            sig.as_ptr(),
            msg.as_bytes().as_ptr(),
            flat.as_ptr(),
            offsets.as_ptr(),
            std::ptr::null(),
            1,
            &mut ok,
            std::ptr::null_mut(),
        )
    };
    rc == 0 && ok == 1
}

// ------------------------------------------------------------------------------------------------------ PublicKey
/// A validated G1 key: both serialisations, like the affine point blst caches
/// (`validator_pubkey_cache.rs:116-118` decompresses once at import; `:195-199` persists the 96-byte form).
#[derive(Clone)]
pub struct PublicKey {
    compressed: [u8; PUBLIC_KEY_BYTES_LEN],
    uncompressed: [u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN],
}

impl TPublicKey for PublicKey {
    fn serialize(&self) -> [u8; PUBLIC_KEY_BYTES_LEN] {
        self.compressed
    }

    fn serialize_uncompressed(&self) -> [u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN] {
        self.uncompressed
    }

    /// blst.rs:130-140 (`key_validate`: decompress, on-curve, subgroup; the infinity check is done by
    /// `generic_public_key.rs:86-94` on the bytes and again here through status 1).
    fn deserialize(bytes: &[u8]) -> Result<Self, Error> {
        if bytes.len() != PUBLIC_KEY_BYTES_LEN {
            return Err(Error::InvalidByteLength { got: bytes.len(), expected: PUBLIC_KEY_BYTES_LEN });
        }
        if !ensure_init() {
            return Err(Error::B200Error(-1));
        }
        let mut uncompressed = [0u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN];
        let mut status = 0u8;
        let rc = unsafe { lhb200_g1_decompress_validate(bytes.as_ptr(), 1, uncompressed.as_mut_ptr(), &mut status) };
        if rc != 0 {
            return Err(Error::B200Error(rc));
        }
        match status {
            0 => {
                let mut compressed = [0u8; PUBLIC_KEY_BYTES_LEN];
                compressed.copy_from_slice(bytes);
                Ok(Self { compressed, uncompressed })
            }
            1 => Err(Error::InvalidInfinityPublicKey),
            s => Err(Error::B200Error(s as i32)), // 2 bad encoding / not on curve, 3 not in the subgroup
        }
    }

    /// blst.rs:142-150: encoding and curve check only.
    fn deserialize_uncompressed(bytes: &[u8]) -> Result<Self, Error> {
        if bytes.len() != PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN {
            return Err(Error::InvalidByteLength { got: bytes.len(), expected: PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN });
        }
        if !ensure_init() {
            return Err(Error::B200Error(-1));
        }
        let mut compressed = [0u8; PUBLIC_KEY_BYTES_LEN];
        let mut status = 0u8;
        let rc = unsafe { lhb200_g1_deserialize_uncompressed(bytes.as_ptr(), 1, compressed.as_mut_ptr(), &mut status) };
        if rc != 0 {
            return Err(Error::B200Error(rc));
        }
        match status {
            0 => {
                let mut uncompressed = [0u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN];
                uncompressed.copy_from_slice(bytes);
                Ok(Self { compressed, uncompressed })
            }
            1 => Err(Error::InvalidInfinityPublicKey),
            s => Err(Error::B200Error(s as i32)),
        }
    }
}

impl Eq for PublicKey {}

impl PartialEq for PublicKey {
    fn eq(&self, other: &Self) -> bool {
        self.compressed[..] == other.compressed[..]
    }
}

// --------------------------------------------------------------------------------------------- AggregatePublicKey
#[derive(Clone)]
pub struct AggregatePublicKey(PublicKey);

impl TAggregatePublicKey<PublicKey> for AggregatePublicKey {
    fn to_public_key(&self) -> GenericPublicKey<PublicKey> {
        GenericPublicKey::from_point(self.0.clone())
    }

    /// blst.rs:178-184: keys are "already checked for subgroup and infinity".
    fn aggregate(pubkeys: &[GenericPublicKey<PublicKey>]) -> Result<Self, Error> {
        if pubkeys.is_empty() || !ensure_init() {
            return Err(Error::B200Error(-2));
        }
        let mut flat = Vec::with_capacity(pubkeys.len() * PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN);
        for pk in pubkeys {
            flat.extend_from_slice(&pk.point().uncompressed);
        }
        let mut compressed = [0u8; PUBLIC_KEY_BYTES_LEN];
        let mut uncompressed = [0u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN];
        let rc = unsafe {
            lhb200_g1_aggregate(flat.as_ptr(), pubkeys.len() as u32, compressed.as_mut_ptr(), uncompressed.as_mut_ptr())
        };
        if rc != 0 {
            return Err(Error::B200Error(rc));
        }
        Ok(Self(PublicKey { compressed, uncompressed }))
    }
}

impl Eq for AggregatePublicKey {}

impl PartialEq for AggregatePublicKey {
    fn eq(&self, other: &Self) -> bool {
        self.0 == other.0
    }
}

// ------------------------------------------------------------------------------------------------------ Signature
/// The 96 canonical (compressed) bytes; decode errors surface at `deserialize` (blst.rs:192-194).
#[derive(Clone)]
pub struct Signature([u8; SIGNATURE_BYTES_LEN]);

fn decode_signature(bytes: &[u8]) -> Result<[u8; SIGNATURE_BYTES_LEN], Error> {
    if bytes.len() != SIGNATURE_BYTES_LEN {
        return Err(Error::InvalidByteLength { got: bytes.len(), expected: SIGNATURE_BYTES_LEN });
    }
    if !ensure_init() {
        return Err(Error::B200Error(-1));
    }
    let mut affine = [0u8; 192];
    let mut status = 0u8;
    let rc = unsafe { lhb200_g2_decompress(bytes.as_ptr(), 1, affine.as_mut_ptr(), &mut status) };
    if rc != 0 {
        return Err(Error::B200Error(rc));
    }
    if status == 2 {
        return Err(Error::B200Error(2)); // bad encoding / not on the curve (no subgroup check here, like blst)
    }
    let mut out = [0u8; SIGNATURE_BYTES_LEN];
    out.copy_from_slice(bytes);
    Ok(out)
}

impl TSignature<PublicKey> for Signature {
    fn serialize(&self) -> [u8; SIGNATURE_BYTES_LEN] {
        self.0
    }

    fn deserialize(bytes: &[u8]) -> Result<Self, Error> {
        decode_signature(bytes).map(Self)
    }

    /// blst.rs:196-200: subgroup-checks the signature, keys are pre-validated.
    fn verify(&self, pubkey: &PublicKey, msg: Hash256) -> bool {
        verify_one(&self.0, msg, &[pubkey])
    }
}

impl PartialEq for Signature {
    fn eq(&self, other: &Self) -> bool {
        self.0[..] == other.0[..]
    }
}

impl Eq for Signature {}

impl std::hash::Hash for Signature {
    fn hash<H: std::hash::Hasher>(&self, state: &mut H) {
        self.0.hash(state);
    }
}

// --------------------------------------------------------------------------------------------- AggregateSignature
#[derive(Clone)]
pub struct AggregateSignature([u8; SIGNATURE_BYTES_LEN]);

impl AggregateSignature {
    /// self <- self + other on the device (`lhb200_g2_aggregate` over the two encodings).
    fn add_bytes(&mut self, other: &[u8; SIGNATURE_BYTES_LEN]) {
        if !ensure_init() {
            return;
        }
        let mut pair = [0u8; 2 * SIGNATURE_BYTES_LEN];
        pair[..SIGNATURE_BYTES_LEN].copy_from_slice(&self.0);
        pair[SIGNATURE_BYTES_LEN..].copy_from_slice(other);
        let mut out = [0u8; SIGNATURE_BYTES_LEN];
        // blst.rs:232 ignores the error of add_signature the same way
        if unsafe { lhb200_g2_aggregate(pair.as_ptr(), 2, out.as_mut_ptr()) } == 0 {
            self.0 = out;
        }
    }
}

impl TAggregateSignature<PublicKey, AggregatePublicKey, Signature> for AggregateSignature {
    fn infinity() -> Self {
        Self(INFINITY_SIGNATURE)
    }

    /// blst.rs:230-233: "signature has already been subgroup checked".
    fn add_assign(&mut self, other: &Signature) {
        self.add_bytes(&other.0)
    }

    /// blst.rs:235-237
    fn add_assign_aggregate(&mut self, other: &Self) {
        self.add_bytes(&other.0)
    }

    fn serialize(&self) -> [u8; SIGNATURE_BYTES_LEN] {
        self.0
    }

    /// blst.rs:243-248
    fn deserialize(bytes: &[u8]) -> Result<Self, Error> {
        decode_signature(bytes).map(Self)
    }

    /// blst.rs:250-261
    fn fast_aggregate_verify(&self, msg: Hash256, pubkeys: &[&GenericPublicKey<PublicKey>]) -> bool {
        let pks = pubkeys.iter().map(|pk| pk.point()).collect::<Vec<_>>();
        verify_one(&self.0, msg, &pks)
    }

    /// blst.rs:263-273
    fn aggregate_verify(&self, msgs: &[Hash256], pubkeys: &[&GenericPublicKey<PublicKey>]) -> bool {
        if msgs.is_empty() || msgs.len() != pubkeys.len() || !ensure_init() {
            return false;
        }
        let mut flat_msgs = Vec::with_capacity(msgs.len() * 32);
        let mut flat_pks = Vec::with_capacity(pubkeys.len() * PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN);
        for (m, pk) in msgs.iter().zip(pubkeys.iter()) {
            flat_msgs.extend_from_slice(m.as_bytes());
            flat_pks.extend_from_slice(&pk.point().uncompressed);
        }
        let mut ok = 0u8;
        let rc = unsafe {
            lhb200_aggregate_verify(self.0.as_ptr(), flat_msgs.as_ptr(), flat_pks.as_ptr(), msgs.len() as u32, &mut ok)
        };
        rc == 0 && ok == 1
    }
}

impl Eq for AggregateSignature {}

impl PartialEq for AggregateSignature {
    fn eq(&self, other: &Self) -> bool {
        self.0[..] == other.0[..]
    }
}

// ------------------------------------------------------------------------------------------------------ SecretKey
#[derive(Clone)]
pub struct SecretKey([u8; SECRET_KEY_BYTES_LEN]);

impl TSecretKey<Signature, PublicKey> for SecretKey {
    /// blst.rs:276-281 (`key_gen` from 32 random bytes); here the scalar is drawn directly and reduced by rejection.
    fn random() -> Self {
        let rng = &mut rand::thread_rng();
        loop {
            let mut bytes: [u8; SECRET_KEY_BYTES_LEN] = rng.gen();
            bytes[0] &= 0x7f;
            if bytes.iter().any(|b| *b != 0) && bytes[..] < CURVE_ORDER_BE[..] {
                return Self(bytes);
            }
        }
    }

    /// blst.rs:287-289
    fn sign(&self, msg: Hash256) -> Signature {
        let mut out = [0u8; SIGNATURE_BYTES_LEN];
        if ensure_init() {
            unsafe { lhb200_sign(self.0.as_ptr(), msg.as_bytes().as_ptr(), 1, out.as_mut_ptr()) };
        }
        Signature(out)
    }

    /// blst.rs:283-285
    fn public_key(&self) -> PublicKey {
        let mut compressed = [0u8; PUBLIC_KEY_BYTES_LEN];
        let mut uncompressed = [0u8; PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN];
        if ensure_init() {
            unsafe { lhb200_sk_to_pk(self.0.as_ptr(), 1, compressed.as_mut_ptr(), uncompressed.as_mut_ptr()) };
        }
        PublicKey { compressed, uncompressed }
    }

    fn serialize(&self) -> ZeroizeHash {
        self.0.into()
    }

    /// blst.rs:295-297 (`from_bytes`: 32 bytes, non-zero — checked by generic_secret_key.rs — and below r).
    fn deserialize(bytes: &[u8]) -> Result<Self, Error> {
        if bytes.len() != SECRET_KEY_BYTES_LEN {
            return Err(Error::InvalidSecretKeyLength { got: bytes.len(), expected: SECRET_KEY_BYTES_LEN });
        }
        if bytes[..] >= CURVE_ORDER_BE[..] {
            return Err(Error::B200Error(2));
        }
        let mut sk = [0u8; SECRET_KEY_BYTES_LEN];
        sk.copy_from_slice(bytes);
        Ok(Self(sk))
    }
}
