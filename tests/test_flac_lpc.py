"""CPU tests of FLAC linear prediction ("flac_lpc_order", kkx.h): a numpy / binary64 reference encoder that follows the
LPC rules of kkx.h literally (the GPU encoder must match it byte for byte, tests/test_flac_lpc_gpu.py), built on the
FIXED encoder of tests/test_flac.py, and an LPC-capable decoder written from the format description (RFC 9639) that
shares nothing with the encoder but the bit reader and the two CRCs.  Every encoded signal must decode to exactly its
samples, and LPC must never make a file larger than the encoder without it."""
import ctypes as C
import functools
import math

import numpy as np
import pytest

from tests.test_flac import (BLOCK, BS_CODES, CONSTANT, FIXED, RATE_CODES, RATES, VERBATIM, _BS_TABLE, _CASES,
                             _FIXED_COEF, _RATE_TABLE, _Bits, _best_fixed, _fold, _pack_bits, _subframe, _utf8,
                             _third_party_decoders, flac_crc8, flac_crc16, flac_encode_ref, harmonic_tone, rate_case,
                             signal)

LPC = "LPC"
MAX_ORDER = 12
PREC = 12          # quantised coefficient precision (bits)
ORDERS = (1, 4, 8, 12)


# ---------------------------------------------------------------------------------------------------- the window
def lpc_window_numpy():
    """M[k] = nint(2^15 * 0.5 * (1 - cos(pi (k + 0.5) / 1024))), nint(v) = floor(v + 0.5) (rule 2)."""
    k = np.arange(1024)
    return np.floor(2.0 ** 15 * 0.5 * (1.0 - np.cos(np.pi * (k + 0.5) / 1024)) + 0.5).astype(np.int64)


@functools.lru_cache(maxsize=1)
def lpc_window():
    """The library's table (kkx_test_flac_lpc_window): the only cosine values the encoder uses."""
    from kokorox_b200.onn import load_library
    m = np.zeros(1024, np.int32)
    assert load_library().kkx_test_flac_lpc_window(m.ctypes.data_as(C.POINTER(C.c_int32))) == 0
    return m.astype(np.int64)


# ---------------------------------------------------------------------------------------------------- encoder
def lpc_design(x, p):
    """Rules 2-5 for the block x (int64): (shift, [q_1..q_p]) or None when the frame has no LPC candidate.  Python
    floats are IEEE binary64 with one rounding per operation, evaluated in the order written."""
    bs = len(x)
    M = lpc_window()
    L = bs >> 2
    W = np.full(bs, 1 << 15, np.int64)
    if L:
        i = np.arange(L)
        W[i] = M[(i * 1024) // L]
        W[bs - 1 - i] = M[(i * 1024) // L]
    xw = (x * W + (1 << 14)) >> 15
    R = [float(int(np.dot(xw[l:], xw[:bs - l]))) for l in range(p + 1)]   # exact in int64, exact as a double
    if R[0] == 0.0:
        return None
    a = [0.0] * (p + 1)
    err = R[0]
    for i in range(1, p + 1):
        acc = R[i]
        for j in range(1, i):
            acc = acc - a[j] * R[i - j]
        k = acc / err
        a = [0.0] + [a[j] - k * a[i - j] for j in range(1, i)] + [k] + [0.0] * (p - i)
        err = err * (1.0 - k * k)
        if not err > 0.0:
            return None
    cmax = max(abs(v) for v in a[1:])
    if cmax == 0.0:
        return None
    shift = min(15, PREC - 1 - math.frexp(cmax)[1])
    if shift < 0:
        return None
    scale = 2.0 ** shift
    ef, q = 0.0, []
    for j in range(1, p + 1):
        ef = ef + a[j] * scale
        qj = min(max(math.floor(ef + 0.5), -2048), 2047)
        q.append(qj)
        ef = ef - qj
    return shift, q


def lpc_residual(x, p, shift, q):
    """Rule 6: e[s] = x[s] - ((sum_j q_j x[s - j]) >> shift) for s = p..bs-1."""
    bs = len(x)
    acc = np.zeros(bs - p, np.int64)
    for j in range(1, p + 1):
        acc += q[j - 1] * x[p - j:bs - j]
    return x[p:] - (acc >> shift)


def _rice(u, bs, w):
    """Cheapest partitioned Rice coding of the residuals u (samples w..bs-1): (bits incl. the 6-bit method + order
    field, porder, [k per partition]); partition orders ascending, ties to the smaller order and the smaller k."""
    ks = np.arange(15)
    cs = np.zeros((len(u) + 1, 15), dtype=np.int64)
    cs[1:] = np.cumsum(u[:, None] >> ks[None, :], axis=0)
    best = None
    for q in range(9):
        if bs % (1 << q) or (bs >> q) <= w:
            continue
        ps = bs >> q
        lo = np.maximum(np.arange(1 << q) * ps - w, 0)
        hi = (np.arange(1 << q) + 1) * ps - w
        cost = cs[hi] - cs[lo] + (hi - lo)[:, None] * (ks[None, :] + 1)
        kbest = np.argmin(cost, axis=1)
        bits = 6 + int((4 + cost[np.arange(1 << q), kbest]).sum())
        if best is None or bits < best[0]:
            best = (bits, q, kbest.tolist())
    return best


def _residual_fields(u, bs, w, q, kbest, vals, nb):
    ps = bs >> q
    for j, k in enumerate(kbest):
        part = u[max(j * ps - w, 0):(j + 1) * ps - w]
        vals.append(k)
        nb.append(4)
        pv = np.empty(2 * len(part), dtype=np.int64)
        pn = np.empty(2 * len(part), dtype=np.int64)
        pv[0::2] = 0
        pn[0::2] = part >> k
        pv[1::2] = (1 << k) | (part & ((1 << k) - 1))
        pn[1::2] = k + 1
        vals.extend(pv.tolist())
        nb.extend(pn.tolist())


def lpc_subframe(x, p):
    """(kind, field values, field widths) of one block's subframe under rules 1-8."""
    bs = len(x)
    if p == 0 or p >= bs or np.all(x == x[0]):
        kind, vals, nb, _ = _subframe(x)
        return kind, vals, nb
    design = lpc_design(x, p)
    if design is not None:
        shift, q = design
        u = _fold(lpc_residual(x, p, shift, q))
        if u.max() < (1 << 20):
            rbits, porder, kbest = _rice(u, bs, p)
            bits = 8 + 16 * p + 4 + 5 + 12 * p + rbits
            fixed = _best_fixed(x)[0]
            if bits < fixed and bits <= 8 + 16 * bs:   # ties go to FIXED; VERBATIM only if strictly cheaper
                vals = [0x40 | ((p - 1) << 1)] + [int(v) & 0xFFFF for v in x[:p]] + [PREC - 1, shift]
                vals += [v & 0xFFF for v in q] + [porder]
                nb = [8] + [16] * p + [4, 5] + [PREC] * p + [6]
                _residual_fields(u, bs, p, porder, kbest, vals, nb)
                return LPC, vals, nb
    kind, vals, nb, _ = _subframe(x)
    return kind, vals, nb


@functools.lru_cache(maxsize=4096)
def _subframe_bytes(blk: bytes, p: int) -> bytes:
    """A subframe starts on a byte boundary (the frame header is whole bytes), so it packs on its own."""
    _, vals, nb = lpc_subframe(np.frombuffer(blk, np.int16).astype(np.int64), p)
    return _pack_bits(vals, nb)


def flac_lpc_encode_ref(pcm, rate: int, p: int) -> bytes:
    """The FLAC file kkx_infer_batch_flac returns with "flac_lpc_order" = p for the 16-bit samples pcm at `rate`."""
    x = np.asarray(pcm, dtype=np.int16)
    n = len(x)
    assert n >= 1 and rate in RATE_CODES and 0 <= p <= MAX_ORDER
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
        body = head + _subframe_bytes(blk.tobytes(), p)
        frames.append(body + flac_crc16(body).to_bytes(2, "big"))
    sizes = [len(f) for f in frames]
    info = (BLOCK.to_bytes(2, "big") * 2 + min(sizes).to_bytes(3, "big") + max(sizes).to_bytes(3, "big") +
            ((rate << 44) | (15 << 36) | n).to_bytes(8, "big") + bytes(16))
    return b"fLaC" + bytes([0x80, 0, 0, 34]) + info + b"".join(frames)


# ---------------------------------------------------------------------------------------------------- decoder
def _rice_residuals(br, bs, order):
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
    return res


def flac_lpc_decode_ref(data: bytes):
    """Decodes a mono 16-bit FLAC stream with CONSTANT / VERBATIM / FIXED / LPC subframes; raises on anything else and
    on any CRC, sync, frame-number or length mismatch.  Returns (int16 samples, info); info["subframes"] lists per
    frame (kind, order, precision, shift)."""
    if data[:4] != b"fLaC" or data[4] != 0x80 or data[5:8] != b"\x00\x00\x22":
        raise ValueError("expected fLaC and one STREAMINFO block")
    body = data[8:42]
    v = int.from_bytes(body[10:18], "big")
    info = dict(min_block=int.from_bytes(body[0:2], "big"), min_frame=int.from_bytes(body[4:7], "big"),
                max_frame=int.from_bytes(body[7:10], "big"), rate=v >> 44, channels=((v >> 41) & 7) + 1,
                bits=((v >> 36) & 31) + 1, total=v & ((1 << 36) - 1), frame_sizes=[], subframes=[])
    if info["channels"] != 1 or info["bits"] != 16:
        raise ValueError("only mono 16-bit streams are decoded")
    br = _Bits(data)
    br.pos = 8 * 42
    out = []
    frame_no = 0
    while br.pos < 8 * len(data):
        start = br.pos >> 3
        if br.read(16) != 0xFFF8:
            raise ValueError(f"frame {frame_no}: bad sync code or variable block size")
        bcode, rcode = br.read(4), br.read(4)
        if br.read(8) != 0x08:
            raise ValueError("not a mono 16-bit frame")
        lead = br.read(8)
        nb = 0
        while nb < 8 and lead & (0x80 >> nb):
            nb += 1
        num = lead & (0x7F >> nb) if nb else lead
        for _ in range(max(nb - 1, 0)):
            num = (num << 6) | (br.read(8) & 0x3F)
        if num != frame_no:
            raise ValueError(f"frame number {num}, expected {frame_no}")
        bs = br.read(8) + 1 if bcode == 6 else br.read(16) + 1 if bcode == 7 else _BS_TABLE[bcode]
        rate = (br.read(8) * 1000 if rcode == 12 else br.read(16) if rcode == 13 else _RATE_TABLE[rcode])
        if rate != info["rate"]:
            raise ValueError("frame rate differs from STREAMINFO")
        hend = br.pos >> 3
        if br.read(8) != flac_crc8(data[start:hend]):
            raise ValueError(f"frame {frame_no}: header CRC-8 mismatch")
        if br.read(1):
            raise ValueError("subframe padding bit set")
        stype = br.read(6)
        if br.read(1):
            raise ValueError("wasted bits are not decoded")
        sub = None
        if stype == 0:
            x = [br.signed(16)] * bs
            sub = (CONSTANT, 0, 0, 0)
        elif stype == 1:
            x = [br.signed(16) for _ in range(bs)]
            sub = (VERBATIM, 0, 0, 0)
        elif 8 <= stype <= 12:
            order = stype - 8
            x = [br.signed(16) for _ in range(order)]
            coef = _FIXED_COEF[order]
            for e in _rice_residuals(br, bs, order):
                x.append(e + sum(c * x[-1 - i] for i, c in enumerate(coef)))
            sub = (FIXED, order, 0, 0)
        elif stype >= 32:
            order = stype - 31
            if order > bs:
                raise ValueError("predictor order exceeds the block size")
            x = [br.signed(16) for _ in range(order)]
            prec = br.read(4) + 1
            if prec == 16:
                raise ValueError("invalid coefficient precision")
            shift = br.signed(5)
            if shift < 0:
                raise ValueError("negative shifts are not decoded")
            coef = [br.signed(prec) for _ in range(order)]   # coef[0] multiplies x[s - 1]
            for e in _rice_residuals(br, bs, order):
                x.append(e + (sum(c * x[-1 - i] for i, c in enumerate(coef)) >> shift))
            sub = (LPC, order, prec, shift)
        else:
            raise ValueError(f"subframe type {stype} is not decoded")
        if br.pos & 7 and br.read(8 - (br.pos & 7)):
            raise ValueError("nonzero frame padding")
        fend = br.pos >> 3
        if br.read(16) != flac_crc16(data[start:fend]):
            raise ValueError(f"frame {frame_no}: CRC-16 mismatch")
        if max(x) > 32767 or min(x) < -32768:
            raise ValueError("sample outside 16 bits")
        out.append(np.asarray(x, dtype=np.int16))
        info["frame_sizes"].append(fend + 2 - start)
        info["subframes"].append(sub)
        frame_no += 1
    dec = np.concatenate(out)
    if len(dec) != info["total"]:
        raise ValueError("frames and STREAMINFO disagree on the sample count")
    if info["min_frame"] != min(info["frame_sizes"]) or info["max_frame"] != max(info["frame_sizes"]):
        raise ValueError("STREAMINFO frame sizes disagree with the frames")
    return dec, info


# ---------------------------------------------------------------------------------------------------- signals
def formant_pulse_train(n=10 * BLOCK, rate=24000, seed=3):
    """A vowel stand-in: a pulse train gliding from 90 to 150 Hz through three formant resonators (700, 1200,
    2600 Hz), light noise, peak 0.3."""
    from scipy.signal import lfilter
    f0 = np.linspace(90.0, 150.0, n)
    phase = np.cumsum(f0 / rate)
    src = (np.diff(np.floor(phase), prepend=0.0) > 0).astype(np.float64)
    y = src
    for fc, bw in ((700.0, 110.0), (1200.0, 120.0), (2600.0, 160.0)):
        r = np.exp(-np.pi * bw / rate)
        y = lfilter([1.0 - r], [1.0, -2.0 * r * np.cos(2 * np.pi * fc / rate), r * r], y)
    y = y + 1e-3 * np.abs(y).max() * np.random.default_rng(seed).standard_normal(n)
    return np.round(y * (0.3 * 32767 / np.abs(y).max())).astype(np.int16)


# ---------------------------------------------------------------------------------------------------- tests
def test_window_table_is_the_numpy_design():
    assert np.array_equal(lpc_window(), lpc_window_numpy())
    m = lpc_window()
    assert m[0] == 0 and m[-1] == 32768 and np.all(np.diff(m) >= 0)


def _check_stream(data, pcm, rate, p):
    dec, info = flac_lpc_decode_ref(data)
    assert np.array_equal(dec, pcm) and info["rate"] == rate
    for kind, order, prec, shift in info["subframes"]:
        if kind == LPC:
            assert order == p <= MAX_ORDER and prec == PREC and 0 <= shift <= 15
    return info


@pytest.mark.parametrize("p", ORDERS)
def test_round_trip(p):
    lpc_frames = 0
    for name, pcm in _CASES:
        data = flac_lpc_encode_ref(pcm, 24000, p)
        info = _check_stream(data, pcm, 24000, p)
        lpc_frames += sum(s[0] == LPC for s in info["subframes"])
        ref = flac_encode_ref(pcm, 24000)
        assert len(data) <= len(ref), name   # a frame is never larger than without LPC
        if name.startswith(("noise", "zero", "const")) or not any(s[0] == LPC for s in info["subframes"]):
            assert data == ref, name         # LPC never chosen: the bytes of the encoder without it
    assert lpc_frames > 0


@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("p", ORDERS)
def test_every_rate(rate, p):
    pcm = rate_case(rate)
    data = flac_lpc_encode_ref(pcm, rate, p)
    _check_stream(data, pcm, rate, p)
    assert len(data) <= len(flac_encode_ref(pcm, rate))


def test_order_zero_is_the_encoder_without_lpc():
    for name, pcm in _CASES:
        assert flac_lpc_encode_ref(pcm, 16000, 0) == flac_encode_ref(pcm, 16000), name


def test_harmonic_tone_compresses():
    pcm = harmonic_tone()
    ratio = len(flac_lpc_encode_ref(pcm, 24000, 8)) / len(flac_encode_ref(pcm, 24000))
    assert ratio <= 0.80, ratio


def test_formant_pulse_train_compresses():
    pcm = formant_pulse_train()
    for p in (8, 12):
        data = flac_lpc_encode_ref(pcm, 24000, p)
        _check_stream(data, pcm, 24000, p)
        assert len(data) < len(flac_encode_ref(pcm, 24000)), p


def test_design_edge_cases():
    # a two-sample block: no taper (L = 0); orders >= bs have no candidate
    x = np.asarray([5, -3], np.int64)
    assert lpc_subframe(x, 2)[0] != LPC and lpc_subframe(x, 12)[0] != LPC
    # an exactly predictable ramp: order 1 is designed and decodes exactly
    pcm = (np.arange(3 * BLOCK) % 2000 * 7 - 7000).astype(np.int16)
    _check_stream(flac_lpc_encode_ref(pcm, 24000, 1), pcm, 24000, 1)
    # the only nonzero sample sits where the taper is 0: R0 = 0, no candidate
    assert lpc_design(np.asarray([1, 0, 0, 0, 0, 0, 0, 0], np.int64), 2) is None


def test_decoder_rejects_corruption():
    pcm = harmonic_tone(2 * BLOCK)
    data = flac_lpc_encode_ref(pcm, 24000, 8)
    assert any(s[0] == LPC for s in flac_lpc_decode_ref(data)[1]["subframes"])
    for pos in (50, 60, len(data) - 1):
        bad = bytearray(data)
        bad[pos] ^= 0x10
        with pytest.raises(ValueError):
            flac_lpc_decode_ref(bytes(bad))


@pytest.mark.parametrize("name", ["harmonic", "sine-22200", "long"])
def test_third_party_decoder(name, tmp_path):
    import subprocess
    decs = _third_party_decoders()
    if not decs:
        pytest.skip("no third-party FLAC decoder (soundfile, flac or ffmpeg) is available")
    pcm = dict(_CASES)[name]
    path = tmp_path / "x.flac"
    path.write_bytes(flac_lpc_encode_ref(pcm, 24000, 8))
    for dec in decs:
        if dec == "soundfile":
            import soundfile
            got, _ = soundfile.read(str(path), dtype="int16")
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
