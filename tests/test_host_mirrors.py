"""Host-side mirrors of @zk-email/helpers (input side of the boundary), pinned on what the reference's tests and
fixtures pin offline: the canonicalisation / hashing of packages/circuits/tests/test-emails/test.eml (SURVEY 8(c)), the
selector scenarios of packages/helpers/tests/input-generators.test.ts:39-63 (fed from a locally built DKIM result because
the reference fetches the key from DNS), sha256Pad / generatePartialSHA semantics and their error strings."""
import base64
import hashlib
import os
import re
import pytest

import zkemail_b200 as z
from zkemail_b200 import dkim
from zkemail_b200.dkim import DKIMVerificationResult

EMAILS = os.path.join(os.path.dirname(__file__), "golden", "emails")


def _fake_dkim_result(raw: bytes) -> DKIMVerificationResult:
    parsed, body = dkim.split_message(raw)
    line = [l for k, l in parsed if k == "dkim-signature"][0]
    tags = dkim.parse_tag_list(re.sub(r"\r?\n[ \t]*", " ", line.decode("latin-1").split(":", 1)[1]))
    hc, bc = (tags.get("c", "simple/simple").split("/") + ["simple"])[:2]
    canon_body = dkim.relaxed_body(body) if bc == "relaxed" else dkim.simple_body(body)
    headers = dkim.signed_header_bytes(parsed, line, tags["h"], hc)
    return DKIMVerificationResult(publicKey=(1 << 2047) | 12345, signature=(1 << 2040) | 999, headers=headers, body=canon_body,
                                  bodyHash=re.sub(r"\s+", "", tags["bh"]), signingDomain=tags["d"], selector=tags["s"],
                                  algo="rsa-sha256", format=tags.get("c", ""), modulusLength=2048)


def test_test_eml_canonicalisation_kats():
    """rsa.test.ts:40-43 message limbs and the bh= tag, reproduced from test.eml (no key needed)."""
    dk = _fake_dkim_result(open(os.path.join(EMAILS, "test.eml"), "rb").read())
    assert len(dk.headers) == 472
    d = int.from_bytes(hashlib.sha256(dk.headers).digest(), "big")
    assert [(d >> (121 * i)) & ((1 << 121) - 1) for i in range(3)] == [
        1156466847851242602709362303526378170, 191372789510123109308037416804949834, 7204]
    assert base64.b64encode(hashlib.sha256(dk.body).digest()).decode() == dk.bodyHash == "7xQMDuoVVU4m0W0WRVSrVXMeGSIASsnucK9dJsrc+vU="


def test_body_hashes_of_helper_fixtures():
    for name in ("email-good.eml", "email-good-large.eml"):
        dk = _fake_dkim_result(open(os.path.join(EMAILS, name), "rb").read())
        assert base64.b64encode(hashlib.sha256(dk.body).digest()).decode() == dk.bodyHash, name


def test_inputs_shape_and_ignore_body_hash():       # input-generators.test.ts:9-37
    dk = _fake_dkim_result(open(os.path.join(EMAILS, "email-good.eml"), "rb").read())
    inputs = z.generate_email_verifier_inputs_from_dkim_result(dk)
    for k in ("emailHeader", "pubkey", "signature", "precomputedSHA", "emailBody", "emailBodyLength", "bodyHashIndex"):
        assert k in inputs
    assert len(inputs["emailHeader"]) == 1024 and len(inputs["emailBody"]) == 1536 and len(inputs["pubkey"]) == 17
    assert all(isinstance(v, str) for v in inputs["emailHeader"])
    inputs = z.generate_email_verifier_inputs_from_dkim_result(dk, {"ignoreBodyHashCheck": True})
    for k in ("precomputedSHA", "emailBody", "emailBodyLength", "bodyHashIndex"):
        assert k not in inputs


def test_sha_precompute_selector():                  # input-generators.test.ts:39-53
    dk = _fake_dkim_result(open(os.path.join(EMAILS, "email-good-large.eml"), "rb").read())
    inputs = z.generate_email_verifier_inputs_from_dkim_result(dk, {"shaPrecomputeSelector": "thousands"})
    body = bytes(int(b) for b in inputs["emailBody"]).decode("latin-1")
    assert body.startswith("h hundreds of thousands of blocks.")
    # the midstate really is the SHA-256 state after the cut-off prefix
    pre = bytes(int(b) for b in inputs["precomputedSHA"])
    cut = len(dk.body) - (int(inputs["emailBodyLength"]) - (int(inputs["emailBodyLength"]) - 0)) if False else None
    padded, plen = z.sha256_pad(dk.body, max(1536, ((len(dk.body) + 63 + 65) // 64) * 64))
    cutoff = plen - int(inputs["emailBodyLength"])
    assert cutoff % 64 == 0 and pre == z.partial_sha(padded, cutoff)


def test_invalid_selector_message():                 # input-generators.test.ts:55-63
    dk = _fake_dkim_result(open(os.path.join(EMAILS, "email-good.eml"), "rb").read())
    with pytest.raises(ValueError, match='SHA precompute selector "Bla Bla" not found in cleaned body'):
        z.generate_email_verifier_inputs_from_dkim_result(dk, {"shaPrecomputeSelector": "Bla Bla"})


def test_sha256_pad_and_partial_sha():
    for n in (0, 1, 55, 56, 63, 64, 119, 120, 1000):
        msg = bytes((i * 7 + 1) & 0xFF for i in range(n))
        padded, plen = z.sha256_pad(msg, 1536)
        assert len(padded) == 1536 and plen % 64 == 0 and plen >= n + 9
        assert padded[:n] == msg and padded[n] == 0x80 and set(padded[plen:]) <= {0}
        assert int.from_bytes(padded[plen - 8:plen], "big") == 8 * n
        # hashing the padded blocks from the IV gives the digest: partial_sha over everything == final state
        st = z.partial_sha(padded, plen)
        assert st == hashlib.sha256(msg).digest()
    with pytest.raises(AssertionError, match="Padding to max length did not complete properly"):
        z.sha256_pad(b"x" * 100, 64)


def test_remaining_body_too_long_message():
    body = b"a" * 3000
    padded, plen = z.sha256_pad(body, 3072)
    with pytest.raises(ValueError, match=r"Remaining body 3072 after the selector is longer than max \(1536\)"):
        z.generate_partial_sha(padded, plen, None, 1536)


def test_to_circom_bigint_bytes():
    x = (1 << 2047) + 0xDEADBEEF
    limbs = z.to_circom_bigint_bytes(x)
    assert len(limbs) == 17 and sum(int(l) << (121 * i) for i, l in enumerate(limbs)) == x
    assert all(int(l) < (1 << 121) for l in limbs)


def test_dkim_verify_roundtrip_and_failures():
    key = z.synthetic.generate_key()
    email = z.synthetic.make_signed_email(3, key)
    rec = z.synthetic.key_record(key)
    dk = z.verify_dkim_signature(email, resolver=lambda n, t: [rec])
    assert dk.signingDomain == "example.com" and dk.modulusLength == 2048 and len(dk.body) == 1024
    assert pow(dk.signature, 65537, dk.publicKey) & ((1 << 256) - 1) == int.from_bytes(hashlib.sha256(dk.headers).digest(), "big")
    with pytest.raises(ValueError, match="DKIM signature not found for domain other.org"):
        z.verify_dkim_signature(email, domain="other.org", resolver=lambda n, t: [rec])
    tampered = email.replace(b"Subject: synthetic", b"Subject: Synthetic")
    with pytest.raises(ValueError, match="bad signature"):
        z.verify_dkim_signature(tampered, resolver=lambda n, t: [rec])
    with pytest.raises(ValueError, match="body hash did not verify"):
        z.verify_dkim_signature(email + b"extra line\r\n", resolver=lambda n, t: [rec])
    # dkim.test.ts:19-29 (invalid selector): "DKIM signature verification failed for domain icloud.com. Reason: no key"
    with pytest.raises(ValueError, match="DKIM signature verification failed for domain example.com. Reason: no key"):
        z.verify_dkim_signature(email)      # offline default resolver: no record from any source


def test_seeded_key_repeats_and_signs():
    """generate_key(seed=...) gives the same 2048-bit key on every call (benchmark inputs repeat from run to run)."""
    key, again, other = (z.synthetic.generate_key(seed=s) for s in (7, 7, 8))
    rec = z.synthetic.key_record(key)
    assert rec == z.synthetic.key_record(again) and rec != z.synthetic.key_record(other)
    assert key.key_size == 2048 and key.private_numbers().public_numbers.e == 65537
    email = z.synthetic.make_signed_email(3, key)
    assert email == z.synthetic.make_signed_email(3, again)
    assert z.verify_dkim_signature(email, resolver=lambda n, t: [rec]).modulusLength == 2048


def test_dkim_key_retry_and_sanitizers():
    """dkim/index.ts:49-66, :105-131 and dkim/sanitizers.ts: every key record of the selector is tried; when the first
    attempt ends in "bad signature" the sanitizers are tried in order and the passing one is reported."""
    from zkemail_b200 import dkim
    key, other = z.synthetic.generate_key(), z.synthetic.generate_key()
    rec, wrong = z.synthetic.key_record(key), z.synthetic.key_record(other)
    email = z.synthetic.make_signed_email(4, key)
    # DNS + archive style key lists: a stale key first, garbage in between, the right key last
    dk = z.verify_dkim_signature(email, resolver=lambda n, t: [wrong, "v=DKIM1; k=rsa; p=", "not a record", rec])
    assert dk.publicKey == key.public_key().public_numbers().n and dk.appliedSanitization is None
    with pytest.raises(ValueError, match="Reason: bad signature"):
        z.verify_dkim_signature(email, resolver=lambda n, t: [wrong])
    resolver = lambda n, t: [rec]
    # removeLabels: a mailing list prefixed the subject after signing
    labelled = email.replace(b"Subject: synthetic", b"Subject: [zk-list] synthetic")
    dk = z.verify_dkim_signature(labelled, resolver=resolver)
    assert dk.appliedSanitization == "removeLabels" and dk.headers == z.verify_dkim_signature(email, resolver=resolver).headers
    with pytest.raises(ValueError, match="Reason: bad signature"):
        z.verify_dkim_signature(labelled, resolver=resolver, enable_sanitization=False)
    # sanitizeTabs: a quoted-printable re-encoding turned a tab of a signed header into =09
    tabbed = z.synthetic.make_signed_email(5, key).replace(b"Subject: synthetic", b"Subject: \tsynthetic")
    # (relaxed canonicalisation folds the tab into one space, so this variant verifies as it is)
    assert z.verify_dkim_signature(tabbed, resolver=resolver).appliedSanitization is None
    garbled = email.replace(b"Subject: synthetic", b"Subject: =09synthetic")
    dk = z.verify_dkim_signature(garbled, resolver=resolver)
    assert dk.appliedSanitization == "sanitizeTabs"
    # revertGoogleMessageId: ARC forwarding replaced the Message-ID header and kept the original one
    mid = b"<%08x@example.com>" % (z.synthetic.SEED_BASE + 4)
    # (the original id sits below Message-ID, as in Gmail's forwards: the reference's string search relies on that order)
    forwarded = (b"ARC-Authentication-Results: i=1; mx.google.com\r\n" +
                 email.replace(b"Message-Id: " + mid, b"Message-ID: <replaced-by-google@mail.gmail.com>")
                      .replace(b"\r\n\r\n", b"\r\nX-Google-Original-Message-ID: " + mid + b"\r\n\r\n", 1))
    dk = z.verify_dkim_signature(forwarded, resolver=resolver)
    assert dk.appliedSanitization == "revertGoogleMessageId"
    # the sanitizer list and their order are the reference's (sanitizers.ts:65)
    assert [f.__name__ for f in dkim.sanitizers] == ["revertGoogleMessageId", "removeLabels", "insert13Before10", "sanitizeTabs"]
    assert dkim.insert13Before10("a\nb\r\nc\n") == "a\r\nb\r\nc\r\n"
    assert dkim.removeLabels("Subject: [x] [y] z") == "Subject: z"          # greedy, as the JS regex
    # a tampered body is not a "bad signature": no sanitizer runs, the body-hash reason is reported (dkim.test.ts:31-44)
    with pytest.raises(ValueError, match="Reason: body hash did not verify"):
        z.verify_dkim_signature(labelled + b"x\r\n", resolver=resolver)


def test_reference_emails_reach_the_key_lookup():
    """email-good.eml / email-good-large.eml of the reference's helper tests (tests/golden/emails, verbatim copies):
    parsing, canonicalisation and the body hash succeed offline; only the icloud.com key is missing (DNS), which the
    reference reports as "no key" (dkim.test.ts:19-29)."""
    import os
    base = os.path.join(os.path.dirname(__file__), "golden", "emails")
    for name in ("email-good.eml", "email-good-large.eml"):
        raw = open(os.path.join(base, name), "rb").read()
        seen = []
        def resolver(n, t):
            seen.append(n)
            raise LookupError("offline")
        with pytest.raises(ValueError, match="DKIM signature verification failed for domain icloud.com. Reason: no key"):
            z.verify_dkim_signature(raw, resolver=resolver)
        assert seen and seen[0].endswith("._domainkey.icloud.com")      # body hash verified, then the key was asked for
        tampered = raw + b"one more line\r\n"
        with pytest.raises(ValueError, match="Reason: body hash did not verify"):
            z.verify_dkim_signature(tampered, resolver=resolver)
