"""rofl_service::flserver::params -- the two optimised encodings end to end (params.rs:699-743 EncParamsRangeCompressed,
:787-885 EncParamsL2Compressed, :181-291 EncModelParams::verify).  A message is a dict of the wire fields of flservice.proto
(`enc_values`, `rand_proof`, `range_proof`, `square_proof`, `square_range_proof`, `range_bits`, `l2_range_bits`) as uint8 arrays in the
fixed-width layouts of SURVEY Appendix C; the protobuf framing itself is the service's business."""
from . import fp


def _c():
    from . import context
    return context()


class EncParamsRangeCompressed:
    @staticmethod
    def encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, seed=None):
        rc, msg = _c().enc_range_compressed_encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, fp.N_BITS, fp.FRAC, seed)
        if rc:
            raise RuntimeError(f"encrypt failed ({rc}); the reference unwrap()s here")
        return msg

    @staticmethod
    def verify(msg, check_percentage=1.0, seed=None):
        return bool(_c().enc_range_compressed_verify(msg, check_percentage, seed))


class EncParamsL2Compressed:
    @staticmethod
    def encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, l2_range, seed=None):
        rc, msg = _c().enc_l2_compressed_encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, l2_range, fp.N_BITS, fp.FRAC, seed)
        if rc:
            raise RuntimeError(f"encrypt failed ({rc}); the reference unwrap()s here")
        return msg

    @staticmethod
    def verify(msg, seed=None):
        return bool(_c().enc_l2_compressed_verify(msg, seed))


class EncParamsRange:
    """params.rs:467-510 / :186-203 -- un-optimised L-inf encoding: one RandProof per element"""
    @staticmethod
    def encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, check_percentage=1.0, seed=None):
        rc, msg = _c().enc_range_encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, check_percentage, fp.N_BITS, fp.FRAC, seed)
        if rc:
            raise RuntimeError(f"encrypt failed ({rc}); the reference unwrap()s here")
        return msg

    @staticmethod
    def verify(msg, check_percentage=1.0, seed=None):
        return bool(_c().enc_range_verify(msg, check_percentage, seed))


class EncParamsL2:
    """params.rs:607-646 / :205-233 -- un-optimised L2 encoding: one SquareRandProof per element"""
    @staticmethod
    def encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, l2_range, seed=None):
        rc, msg = _c().enc_l2_encrypt(plaintext_vec, blinding_vec, prove_range, n_partition, l2_range, fp.N_BITS, fp.FRAC, seed)
        if rc:
            raise RuntimeError(f"encrypt failed ({rc}); the reference unwrap()s here")
        return msg

    @staticmethod
    def verify(msg, seed=None):
        return bool(_c().enc_l2_verify(msg, seed))


class EncModelParamsAccumulator:
    """params.rs:74-148 -- the server's per-round sum of the clients' encrypted updates, kept on the device: accumulate_other adds one
    verified message as it arrives (O(D) state however many clients), extract checks that every accumulated R is B and decrypts L.
    The accumulation starts at the unity (B, B) as in the reference, so every decrypted value is one raw LSB (2^-frac) high (SURVEY App. B.1)."""
    _REC_BYTES = {"range": 64, "rangecompressed": 64, "l2": 96, "l2compressed": 96}

    def __init__(self, acc):
        self._acc = acc

    @classmethod
    def unity(cls, D, enc_type):
        """EncModelParams::unity (params.rs:165-179); enc_type: Range, L2, RangeCompressed or L2Compressed (an `Enc` prefix, case and '_' ignored)"""
        key = enc_type.replace("_", "").lower()
        key = key[3:] if key.startswith("enc") else key
        if key not in cls._REC_BYTES:
            raise ValueError(f"no device accumulator for enc_type {enc_type!r}")
        return cls(_c().accumulator(D, cls._REC_BYTES[key], 1))

    def accumulate_other(self, msg):
        """adds one message (a dict as the encoders return it) through its enc_values; raises if a point of it does not decode"""
        added = self._acc.add(msg["enc_values"].reshape(1, self._acc.D, self._acc.rec_bytes))
        if added[0] != 1:
            raise RuntimeError(f"accumulate failed ({int(added[0])}): a point of the message does not decode")

    @property
    def count(self):
        return self._acc.count

    def extract(self, table_size=1 << 16, bsgs_bits=16):
        """EncModelParamsAccumulator::extract (params.rs:126-147) -> float32[D]; raises when an R is not B (-8) or a value has no log in range (-5)"""
        rc, _, f = self._acc.extract(table_size, bsgs_bits, fp.N_BITS, fp.FRAC)
        if rc:
            raise RuntimeError(f"extract failed ({rc})")
        return f

    def close(self):
        self._acc.close()
