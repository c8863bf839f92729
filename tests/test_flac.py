"""CPU tests of the FLAC output format (kkx_infer_batch_flac, kkx.h): a numpy reference encoder that follows the
bitstream rules of kkx.h literally (the GPU encoder must match it byte for byte, tests/test_flac_gpu.py), and a
decoder written from the format description (RFC 9639) that shares nothing with the encoder but the two CRCs.  Every
encoded signal must decode to exactly its samples."""
import shutil
import subprocess

import numpy as np
import pytest

BLOCK = 4096
RATES = (8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000)
RATE_CODES = {8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10, 12000: 12, 11025: 13}
BS_CODES = {4096: 12, 192: 1, 576: 2, 1152: 3, 2304: 4, 256: 8, 512: 9, 1024: 10, 2048: 11}
CONSTANT, FIXED, VERBATIM = "CONSTANT", "FIXED", "VERBATIM"


# ---------------------------------------------------------------------------------------------------- CRCs
def flac_crc8(data: bytes) -> int:
    """CRC-8 of a frame header: polynomial x^8 + x^2 + x + 1 (0x07), initial value 0."""
    crc = 0
    for byte in data:
        crc ^= byte
        for _ in range(8):
            crc = ((crc << 1) ^ 0x07) & 0xFF if crc & 0x80 else (crc << 1) & 0xFF
    return crc


def _crc16_table():
    tab = []
    for i in range(256):
        c = i << 8
        for _ in range(8):
            c = ((c << 1) ^ 0x8005) & 0xFFFF if c & 0x8000 else (c << 1) & 0xFFFF
        tab.append(c)
    return tab


_CRC16 = _crc16_table()


def flac_crc16(data: bytes) -> int:
    """CRC-16 of a frame: polynomial x^16 + x^15 + x^2 + 1 (0x8005), initial value 0, unreflected."""
    crc = 0
    tab = _CRC16
    for byte in data:
        crc = ((crc << 8) & 0xFFFF) ^ tab[(crc >> 8) ^ byte]
    return crc


# ---------------------------------------------------------------------------------------------------- encoder
def _pack_bits(vals, nbits) -> bytes:
    """MSB-first concatenation of fields (value, width), zero-padded to a byte boundary."""
    vals = np.asarray(vals, dtype=np.uint64)
    nbits = np.asarray(nbits, dtype=np.int64)
    keep = nbits > 0
    vals, nbits = vals[keep], nbits[keep]
    total = int(nbits.sum())
    starts = np.cumsum(nbits) - nbits
    field = np.repeat(np.arange(len(nbits)), nbits)
    within = np.arange(total, dtype=np.int64) - starts[field]
    shift = (nbits[field] - 1 - within).astype(np.uint64)
    bits = ((vals[field] >> shift) & np.uint64(1)).astype(np.uint8)
    return np.packbits(bits).tobytes()   # packbits pads the last byte with zeros


def _utf8(v: int) -> bytes:
    if v < 0x80:
        return bytes([v])
    n = 2
    while v >= 1 << (5 * n + 1):
        n += 1
    out = [0x80 | ((v >> (6 * i)) & 0x3F) for i in range(n - 1)][::-1]
    return bytes([((0xFF00 >> n) & 0xFF) | (v >> (6 * (n - 1)))] + out)


def _fold(e):
    return np.where(e >= 0, 2 * e, -2 * e - 1)


def _best_fixed(x):
    """Cheapest FIXED encoding of block x (int64): (bits, order, porder, [k per partition])."""
    bs = len(x)
    ks = np.arange(15)
    best = None
    for o in range(5):
        if o >= bs:
            break
        u = _fold(np.diff(x, n=o))                     # residuals of the fixed order-o predictor, samples o..bs-1
        cs = np.zeros((len(u) + 1, 15), dtype=np.int64)
        cs[1:] = np.cumsum(u[:, None] >> ks[None, :], axis=0)
        for q in range(9):
            if bs % (1 << q) or (bs >> q) <= o:
                continue
            ps = bs >> q
            lo = np.maximum(np.arange(1 << q) * ps - o, 0)
            hi = (np.arange(1 << q) + 1) * ps - o
            cnt = (hi - lo)[:, None]
            cost = cs[hi] - cs[lo] + cnt * (ks[None, :] + 1)   # [partition, k]
            kbest = np.argmin(cost, axis=1)                      # first minimum: the smaller k
            bits = 8 + 16 * o + 6 + int((4 + cost[np.arange(1 << q), kbest]).sum())
            if best is None or bits < best[0]:
                best = (bits, o, q, kbest.tolist())
    return best


def _subframe(x):
    """(kind, field values, field widths, order) of one block's subframe."""
    bs = len(x)
    if np.all(x == x[0]):
        return CONSTANT, [0x00, int(x[0]) & 0xFFFF], [8, 16], 0
    bits, o, q, kbest = _best_fixed(x)
    if 8 + 16 * bs < bits:
        return VERBATIM, [0x02] + [int(v) & 0xFFFF for v in x], [8] + [16] * bs, 0
    vals = [0x10 | (o << 1)] + [int(v) & 0xFFFF for v in x[:o]] + [q]
    nb = [8] + [16] * o + [6]
    u = _fold(np.diff(x, n=o))
    ps = bs >> q
    for j, k in enumerate(kbest):
        part = u[max(j * ps - o, 0):(j + 1) * ps - o]
        vals.append(k)
        nb.append(4)
        # code: (u >> k) zeros, then the (k + 1)-bit value 1 followed by the low k bits
        pv = np.empty(2 * len(part), dtype=np.int64)
        pn = np.empty(2 * len(part), dtype=np.int64)
        pv[0::2] = 0
        pn[0::2] = part >> k
        pv[1::2] = (1 << k) | (part & ((1 << k) - 1))
        pn[1::2] = k + 1
        vals.extend(pv.tolist())
        nb.extend(pn.tolist())
    return FIXED, vals, nb, o


def flac_encode_ref(pcm, rate: int) -> bytes:
    """The FLAC file kkx_infer_batch_flac returns for the 16-bit samples pcm at sample rate `rate` (kkx.h rules)."""
    x = np.asarray(pcm, dtype=np.int64)
    n = len(x)
    assert n >= 1 and rate in RATE_CODES
    frames = []
    for i in range((n + BLOCK - 1) // BLOCK):
        blk = x[i * BLOCK:(i + 1) * BLOCK]
        bs = len(blk)
        if bs in BS_CODES:
            bc, extra = BS_CODES[bs], b""
        elif bs <= 256:
            bc, extra = 6, bytes([bs - 1])
        else:
            bc, extra = 7, (bs - 1).to_bytes(2, "big")
        rc = RATE_CODES[rate]
        rextra = bytes([rate // 1000]) if rc == 12 else rate.to_bytes(2, "big") if rc == 13 else b""
        head = bytes([0xFF, 0xF8, (bc << 4) | rc, 0x08]) + _utf8(i) + extra + rextra
        head += bytes([flac_crc8(head)])
        _, vals, nb, _ = _subframe(blk)
        body = head + _pack_bits(vals, nb)
        frames.append(body + flac_crc16(body).to_bytes(2, "big"))
    sizes = [len(f) for f in frames]
    info = (BLOCK.to_bytes(2, "big") * 2 + min(sizes).to_bytes(3, "big") + max(sizes).to_bytes(3, "big") +
            ((rate << 44) | (0 << 41) | (15 << 36) | n).to_bytes(8, "big") + bytes(16))
    return b"fLaC" + bytes([0x80, 0, 0, 34]) + info + b"".join(frames)


# ---------------------------------------------------------------------------------------------------- decoder
class _Bits:
    def __init__(self, data: bytes):
        self.data = data
        self.pos = 0
        self.ones = np.flatnonzero(np.unpackbits(np.frombuffer(data, dtype=np.uint8)))

    def read(self, n: int) -> int:
        if n == 0:
            return 0
        r = self.pos & 7
        nbytes = (r + n + 7) // 8
        b0 = self.pos >> 3
        if b0 + nbytes > len(self.data):
            raise ValueError("read past the end of the stream")
        chunk = int.from_bytes(self.data[b0:b0 + nbytes], "big")
        self.pos += n
        return (chunk >> (8 * nbytes - r - n)) & ((1 << n) - 1)

    def signed(self, n: int) -> int:
        v = self.read(n)
        return v - (1 << n) if v >> (n - 1) else v

    def unary(self) -> int:
        i = int(np.searchsorted(self.ones, self.pos))
        if i == len(self.ones):
            raise ValueError("unterminated unary code")
        q = int(self.ones[i]) - self.pos
        self.pos += q + 1
        return q


_FIXED_COEF = {0: (), 1: (1,), 2: (2, -1), 3: (3, -3, 1), 4: (4, -6, 4, -1)}
_BS_TABLE = {1: 192, 2: 576, 3: 1152, 4: 2304, 5: 4608, 8: 256, 9: 512, 10: 1024, 11: 2048, 12: 4096, 13: 8192,
             14: 16384, 15: 32768}
_RATE_TABLE = {1: 88200, 2: 176400, 3: 192000, 4: 8000, 5: 16000, 6: 22050, 7: 24000, 8: 32000, 9: 44100, 10: 48000,
               11: 96000}


def flac_decode_ref(data: bytes):
    """Decodes a mono 16-bit FLAC stream with CONSTANT / VERBATIM / FIXED subframes; raises on anything else and on
    any CRC, sync, frame-number or length mismatch.  Returns (int16 samples, info dict)."""
    if data[:4] != b"fLaC":
        raise ValueError("missing fLaC marker")
    p = 4
    info = None
    while True:
        last, btype, blen = data[p] >> 7, data[p] & 0x7F, int.from_bytes(data[p + 1:p + 4], "big")
        body = data[p + 4:p + 4 + blen]
        if len(body) != blen:
            raise ValueError("truncated metadata block")
        if info is None:
            if btype != 0 or blen != 34:
                raise ValueError("the first metadata block must be STREAMINFO")
            v = int.from_bytes(body[10:18], "big")
            info = dict(min_block=int.from_bytes(body[0:2], "big"), max_block=int.from_bytes(body[2:4], "big"),
                        min_frame=int.from_bytes(body[4:7], "big"), max_frame=int.from_bytes(body[7:10], "big"),
                        rate=v >> 44, channels=((v >> 41) & 7) + 1, bits=((v >> 36) & 31) + 1,
                        total=v & ((1 << 36) - 1), md5=bytes(body[18:34]))
        p += 4 + blen
        if last:
            break
    if info["channels"] != 1 or info["bits"] != 16:
        raise ValueError("only mono 16-bit streams are decoded")
    info.update(frame_sizes=[], kinds=[], block_sizes=[], header_codes=[])
    br = _Bits(data)
    br.pos = 8 * p
    out = []
    frame_no = 0
    while br.pos < 8 * len(data):
        start = br.pos >> 3
        if br.read(15) != 0x7FFC:
            raise ValueError(f"frame {frame_no}: bad sync code")
        if br.read(1):
            raise ValueError("variable-blocksize streams are not decoded")
        bcode, rcode = br.read(4), br.read(4)
        if br.read(4) != 0 or br.read(3) != 4 or br.read(1) != 0:
            raise ValueError("not a mono 16-bit frame (or reserved bit set)")
        lead = br.read(8)
        nb = 0
        while nb < 8 and lead & (0x80 >> nb):
            nb += 1
        if nb == 1 or nb > 7:
            raise ValueError("bad frame number coding")
        num = lead & (0x7F >> nb) if nb else lead
        for _ in range(max(nb - 1, 0)):
            c = br.read(8)
            if c >> 6 != 2:
                raise ValueError("bad frame number continuation byte")
            num = (num << 6) | (c & 0x3F)
        if num != frame_no:
            raise ValueError(f"frame number {num}, expected {frame_no}")
        if bcode == 6:
            bs = br.read(8) + 1
        elif bcode == 7:
            bs = br.read(16) + 1
        elif bcode in _BS_TABLE:
            bs = _BS_TABLE[bcode]
        else:
            raise ValueError(f"reserved block-size code {bcode}")
        if rcode == 12:
            rate = br.read(8) * 1000
        elif rcode == 13:
            rate = br.read(16)
        elif rcode == 14:
            rate = br.read(16) * 10
        elif rcode == 0:
            rate = info["rate"]
        elif rcode in _RATE_TABLE:
            rate = _RATE_TABLE[rcode]
        else:
            raise ValueError(f"invalid sample-rate code {rcode}")
        if rate != info["rate"]:
            raise ValueError(f"frame rate {rate} differs from STREAMINFO {info['rate']}")
        hend = br.pos >> 3
        if br.read(8) != flac_crc8(data[start:hend]):
            raise ValueError(f"frame {frame_no}: header CRC-8 mismatch")
        if br.read(1):
            raise ValueError("subframe padding bit set")
        stype = br.read(6)
        if br.read(1):
            raise ValueError("wasted bits are not decoded")
        if stype == 0:
            kind = CONSTANT
            x = [br.signed(16)] * bs
        elif stype == 1:
            kind = VERBATIM
            x = [br.signed(16) for _ in range(bs)]
        elif 8 <= stype <= 12:
            kind = FIXED
            order = stype - 8
            if order > bs:
                raise ValueError("predictor order exceeds the block size")
            x = [br.signed(16) for _ in range(order)]
            if br.read(2) != 0:
                raise ValueError("only Rice coding method 0 is decoded")
            porder = br.read(4)
            if bs % (1 << porder) or (bs >> porder) < order:
                raise ValueError("invalid partition order")
            res = []
            for j in range(1 << porder):
                k = br.read(4)
                if k == 15:
                    raise ValueError("Rice escape codes are not decoded")
                for _ in range((bs >> porder) - (order if j == 0 else 0)):
                    u = (br.unary() << k) | br.read(k)
                    res.append(u >> 1 if u & 1 == 0 else -(u >> 1) - 1)
            coef = _FIXED_COEF[order]
            for e in res:
                x.append(e + sum(c * x[-1 - i] for i, c in enumerate(coef)))
        else:
            raise ValueError(f"subframe type {stype} is not decoded")
        if br.pos & 7:
            if br.read(8 - (br.pos & 7)):
                raise ValueError("nonzero frame padding")
        fend = br.pos >> 3
        if br.read(16) != flac_crc16(data[start:fend]):
            raise ValueError(f"frame {frame_no}: CRC-16 mismatch")
        if max(x) > 32767 or min(x) < -32768:
            raise ValueError("sample outside 16 bits")
        out.append(np.asarray(x, dtype=np.int16))
        info["frame_sizes"].append(fend + 2 - start)
        info["kinds"].append(kind)
        info["block_sizes"].append(bs)
        info["header_codes"].append((bcode, rcode))
        frame_no += 1
    bss = info["block_sizes"]
    if sum(bss) != info["total"]:
        raise ValueError(f"frames hold {sum(bss)} samples, STREAMINFO says {info['total']}")
    if any(b != info["min_block"] for b in bss[:-1]) or (bss and bss[-1] > info["max_block"]):
        raise ValueError("block sizes disagree with STREAMINFO")
    return (np.concatenate(out) if out else np.zeros(0, np.int16)), info


# ---------------------------------------------------------------------------------------------------- signals
LENGTHS = (1, 2, 5, 16, 4095, 4096, 4097, 4096 * 3 + 192, 600 * 37)
LONG = 4096 * 2100 + 1   # frame numbers past 2047: 3-byte UTF-8 coding


def harmonic_tone(n=12 * BLOCK, rate=24000):
    """150 Hz with harmonics h = 1..8 of amplitude 1/h, a raised-cosine envelope over the whole signal, peak 0.3."""
    t = np.arange(n) / rate
    s = sum(np.sin(2 * np.pi * 150 * h * t) / h for h in range(1, 9))
    s = s * (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(n) / (n - 1)))
    return np.round(s * (0.3 * 32767 / np.abs(s).max())).astype(np.int16)


def signal(kind, n, seed=0):
    i = np.arange(n)
    if kind == "zero":
        return np.zeros(n, np.int16)
    if kind == "const":
        return np.full(n, -1234, np.int16)
    if kind == "alternating":
        return np.where(i % 2 == 0, 32767, -32768).astype(np.int16)
    if kind == "noise":
        return np.random.default_rng(seed + n).integers(-32768, 32768, n).astype(np.int16)
    if kind == "sine":   # slow, full scale
        return np.round(32767 * np.sin(2 * np.pi * i / 9000.0)).astype(np.int16)
    raise ValueError(kind)


SIGNALS = ("zero", "const", "alternating", "noise", "sine")


def long_signal():
    """LONG samples: silence, then a tone in the last frames (FIXED frames with 3-byte frame numbers)."""
    x = np.zeros(LONG, np.int16)
    x[-3 * BLOCK:] = harmonic_tone(3 * BLOCK + 1)[:3 * BLOCK]
    x[-1] = 7
    return x


def all_cases():
    """(name, pcm) of every round-trip case; the GPU test packs them into one ragged batch."""
    cases = [(f"{k}-{n}", signal(k, n)) for n in LENGTHS for k in SIGNALS]
    cases.append(("harmonic", harmonic_tone()))
    cases.append(("long", long_signal()))
    return cases


def rate_case(rate):
    return np.concatenate([harmonic_tone(5000), signal("noise", 300)])


# ---------------------------------------------------------------------------------------------------- tests
def test_crc_check_values():
    assert flac_crc8(b"123456789") == 0xF4
    assert flac_crc16(b"123456789") == 0xFEE8


def test_utf8_frame_numbers():
    assert _utf8(0) == b"\x00" and _utf8(0x7F) == b"\x7f"
    assert _utf8(0x80) == b"\xc2\x80" and _utf8(0x7FF) == b"\xdf\xbf"
    assert _utf8(0x800) == b"\xe0\xa0\x80" and _utf8(2100) == bytes([0xE0, 0xA0 | (2100 >> 6 & 0x1F), 0x80 | (2100 & 0x3F)])


_CASES = all_cases()


@pytest.mark.parametrize("name,pcm", _CASES, ids=[c[0] for c in _CASES])
def test_round_trip(name, pcm):
    data = flac_encode_ref(pcm, 24000)
    dec, info = flac_decode_ref(data)
    assert np.array_equal(dec, pcm)
    n = len(pcm)
    # STREAMINFO equals the stream; no frame exceeds its verbatim size
    assert info["total"] == n and info["rate"] == 24000 and info["min_block"] == info["max_block"] == BLOCK
    assert info["md5"] == bytes(16)
    assert info["min_frame"] == min(info["frame_sizes"]) and info["max_frame"] == max(info["frame_sizes"])
    assert len(data) == 42 + sum(info["frame_sizes"])
    for i, (size, bs) in enumerate(zip(info["frame_sizes"], info["block_sizes"])):
        assert bs == min(BLOCK, n - i * BLOCK)
        hdr = 4 + len(_utf8(i)) + (0 if bs in BS_CODES else 1 if bs <= 256 else 2) + 1
        assert size <= hdr + 1 + 2 * bs + 2
    kinds = info["kinds"]
    if name.startswith(("zero", "const")):
        assert set(kinds) == {CONSTANT}
    if name.startswith("alternating"):
        assert all(k == (CONSTANT if bs == 1 else VERBATIM) for k, bs in zip(kinds, info["block_sizes"]))
    if name.startswith("sine") and n >= BLOCK:
        assert kinds[0] == FIXED
    if name == "long":
        assert kinds[0] == CONSTANT and kinds[-2] == FIXED and info["header_codes"][-1][0] == 6
    if name.startswith("noise") and n >= BLOCK:
        assert FIXED in kinds or VERBATIM in kinds


def test_short_last_block_codes():
    for bs, code in ((192, 1), (1, 6), (256, 8), (257, 7), (4095, 7), (2048, 11)):
        _, info = flac_decode_ref(flac_encode_ref(signal("noise", BLOCK + bs), 24000))
        assert info["header_codes"][-1][0] == code and info["block_sizes"][-1] == bs


def test_harmonic_tone_compresses_below_half():
    pcm = harmonic_tone()
    data = flac_encode_ref(pcm, 24000)
    assert len(data) < 0.5 * 2 * len(pcm), len(data) / (2 * len(pcm))


def test_high_orders_win_on_a_slow_sine():
    data = flac_encode_ref(signal("sine", 3 * BLOCK), 24000)
    _, info = flac_decode_ref(data)
    assert data[42 + 4 + 1 + 1] >> 1 & 7 >= 2   # first frame's FIXED order (header: 4 bytes + 1 number + CRC-8)
    assert set(info["kinds"]) == {FIXED}


@pytest.mark.parametrize("rate", RATES)
def test_every_rate(rate):
    pcm = rate_case(rate)
    data = flac_encode_ref(pcm, rate)
    dec, info = flac_decode_ref(data)
    assert np.array_equal(dec, pcm) and info["rate"] == rate
    assert all(rc == RATE_CODES[rate] for _, rc in info["header_codes"])
    first = data[42:]
    extra = {12000: bytes([12]), 11025: (11025).to_bytes(2, "big")}.get(rate, b"")
    assert first[4 + 1:4 + 1 + len(extra)] == extra   # the rate field follows the 1-byte frame number 0


def test_decoder_rejects_corruption():
    data = bytearray(flac_encode_ref(signal("sine", 5000), 16000))
    for pos in (44, 50, len(data) - 1):
        bad = bytearray(data)
        bad[pos] ^= 0x10
        with pytest.raises(ValueError):
            flac_decode_ref(bytes(bad))


def _third_party_decoders():
    out = []
    try:
        import soundfile  # noqa: F401
        out.append("soundfile")
    except Exception:
        pass
    for tool in ("flac", "ffmpeg"):
        if shutil.which(tool):
            out.append(tool)
    return out


@pytest.mark.parametrize("name", ["harmonic", "noise-4097", "alternating-12480", "const-5"])
def test_third_party_decoder(name, tmp_path):
    decs = _third_party_decoders()
    if not decs:
        pytest.skip("no third-party FLAC decoder (soundfile, flac or ffmpeg) is available")
    pcm = dict(_CASES)[name]
    path = tmp_path / "x.flac"
    path.write_bytes(flac_encode_ref(pcm, 24000))
    for dec in decs:
        if dec == "soundfile":
            import soundfile
            got, sr = soundfile.read(str(path), dtype="int16")
            assert sr == 24000
        elif dec == "flac":
            raw = tmp_path / "x.raw"
            subprocess.run(["flac", "-d", "-f", "--force-raw-format", "--endian=little", "--sign=signed", "-o",
                            str(raw), str(path)], check=True, capture_output=True)
            got = np.fromfile(raw, dtype="<i2")
        else:
            r = subprocess.run(["ffmpeg", "-v", "error", "-i", str(path), "-f", "s16le", "-"], check=True,
                               capture_output=True)
            got = np.frombuffer(r.stdout, dtype="<i2")
        assert np.array_equal(np.asarray(got).reshape(-1), pcm), dec
