"""Synthetic DKIM-signed emails for benchmarks and tests (BASELINE.md section 2, SURVEY 8(d) "Synthetic input
generator", appendix A.10).  Headers follow the 7-field template of
/root/reference/packages/circuits/tests/test-emails/test.eml; the body is printable ASCII with CRLF every 76 chars."""
from __future__ import annotations
import base64
import hashlib
import random

import numpy as np
from cryptography.hazmat.primitives import hashes, serialization
from cryptography.hazmat.primitives.asymmetric import padding, rsa

from .dkim import format_relaxed_line, relaxed_body

SEED_BASE = 0x5EED0000
_SMALL_PRIMES = [p for p in range(3, 2000, 2) if all(p % q for q in range(3, int(p ** 0.5) + 1, 2))]


def _probable_prime(n: int, rng: random.Random) -> bool:
    if any(n % p == 0 for p in _SMALL_PRIMES):
        return n in _SMALL_PRIMES
    d, s = n - 1, 0
    while d % 2 == 0:
        d, s = d // 2, s + 1
    for _ in range(40):                                  # Miller-Rabin
        x = pow(rng.randrange(2, n - 1), d, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = pow(x, 2, n)
            if x == n - 1:
                break
        else:
            return False
    return True


def generate_key(bits: int = 2048, seed: int | None = None):
    """A fresh RSA key, or with `seed` the same key on every call, so that benchmark inputs repeat from run to run."""
    e = 65537
    if seed is None:
        return rsa.generate_private_key(public_exponent=e, key_size=bits)
    rng = random.Random(seed)

    def prime():
        while True:
            c = rng.getrandbits(bits // 2) | (3 << (bits // 2 - 2)) | 1     # top two bits set: n has exactly `bits` bits
            if c % e != 1 and _probable_prime(c, rng):
                return c

    p = prime()
    q = prime()
    while q == p:
        q = prime()
    d = pow(e, -1, (p - 1) * (q - 1))
    return rsa.RSAPrivateNumbers(p, q, d, rsa.rsa_crt_dmp1(d, p), rsa.rsa_crt_dmq1(d, q), rsa.rsa_crt_iqmp(p, q),
                                 rsa.RSAPublicNumbers(e, p * q)).private_key()


def key_record(key) -> str:
    der = key.public_key().public_bytes(serialization.Encoding.DER, serialization.PublicFormat.SubjectPublicKeyInfo)
    return "v=DKIM1; k=rsa; p=" + base64.b64encode(der).decode()


def synthetic_body(index: int, length: int = 1024, marker: str | None = None) -> bytes:
    """Exactly `length` canonical bytes: 76 printable characters (0x21-0x7E, no leading/trailing blanks) + CRLF per line."""
    rng = np.random.default_rng(SEED_BASE + index)
    out = bytearray()
    if marker:
        out += marker.encode() + b"\r\n"
    while len(out) < length:
        room = length - len(out)
        if room <= 2:
            # cannot place a text line and CRLF: extend the previous line instead
            out = out[:-2] + bytes(rng.integers(0x21, 0x7F, size=room, dtype=np.uint8)) + b"\r\n"
            break
        n = min(76, room - 2)
        out += bytes(rng.integers(0x21, 0x7F, size=n, dtype=np.uint8)) + b"\r\n"
    assert len(out) == length and relaxed_body(bytes(out)) == bytes(out)
    return bytes(out)


def make_signed_email(index: int, key, body_len: int = 1024, domain: str = "example.com", selector: str = "sel",
                      marker: str | None = None, body_override: bytes | None = None) -> bytes:
    body = body_override if body_override is not None else synthetic_body(index, body_len, marker)
    headers = [
        b"from: sender%04d@%s" % (index, domain.encode()),
        b"Content-Type: text/plain; charset=us-ascii",
        b"Mime-Version: 1.0 (Synthetic %d)" % index,
        b"Subject: synthetic email %d" % index,
        b"Message-Id: <%08x@%s>" % (SEED_BASE + index, domain.encode()),
        b"Date: Sat, 14 Oct 2023 22:09:12 +0300",
        b"to: rcpt%04d@%s" % (index, domain.encode()),
    ]
    bh = base64.b64encode(hashlib.sha256(relaxed_body(body)).digest()).decode()
    h_list = "from:Content-Type:Mime-Version:Subject:Message-Id:Date:to"
    sig_value = (f"v=1; a=rsa-sha256; c=relaxed/relaxed; d={domain}; s={selector}; t=1697310552; bh={bh}; "
                 f"h={h_list}; b=")
    dkim_line = b"DKIM-Signature: " + sig_value.encode()
    # signing input: relaxed(each header named in h=, picked bottom-up) + CRLF, then relaxed(DKIM-Signature, b= empty)
    by_name = {h.split(b":", 1)[0].strip().lower(): h for h in headers}
    signing = b"".join(format_relaxed_line(by_name[n.lower().encode()], b"\r\n") for n in h_list.split(":"))
    signing += format_relaxed_line(dkim_line)
    sig = key.sign(signing, padding.PKCS1v15(), hashes.SHA256())
    dkim_full = dkim_line + base64.b64encode(sig)
    return dkim_full + b"\r\n" + b"\r\n".join(headers) + b"\r\n\r\n" + body
