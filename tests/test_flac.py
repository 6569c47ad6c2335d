"""FLAC decoding (audio_calm_b200.flac, csrc/acb_flac.cu) against the plain-Python RFC 9639 decoder in oracle/flac_oracle.py.

CPU: header parsing (metadata skipping, ID3v2 prefix, total = 0 recovery), rejections, CRC-8 / CRC-16 known values, the oracle on
every fixture against its recorded PCM hash, oracle-encoder round trips of every construct, the new ABI symbols.
GPU: every fixture and construct bit-exact in int16 and float32; uniform, ragged and per-clip launches agree; a planted false sync;
corrupt and truncated clips fail alone; guard bytes around each region are never read; the dataset driver on mixed .flac / .wav trees."""
import json
import os
import types

import numpy as np
import pytest
import torch

import audio_calm_b200 as acb
from audio_calm_b200 import _lib, flac
from audio_calm_b200.preprocess import process_dataset as pd
from oracle import flac_oracle as fo
from oracle.logmel_oracle import synth_clip

FIXTURES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "flac")


def _manifest():
    with open(os.path.join(FIXTURES, "MANIFEST.json")) as f:
        return json.load(f)["files"]


def _fixture(name):
    with open(os.path.join(FIXTURES, name), "rb") as f:
        return f.read()


def _sig(n, bps, channels=1, seed=1):
    x = np.cumsum(np.stack([synth_clip(n, seed + c) for c in range(channels)]).astype(np.float64), axis=1)
    x -= x.mean(axis=1, keepdims=True)
    x /= np.abs(x).max() + 1e-12
    return np.round(x * 0.9 * ((1 << (bps - 1)) - 1)).astype(np.int64)


# every construct of RFC 9639 the oracle encoder can be asked for: (name, pcm, sample rate, bps, encoder settings)
def _constructs():
    out = []
    for bps in (8, 12, 16, 20, 24):
        out.append((f"fixed4_{bps}", _sig(5000, bps, 1, 1), 16000, bps, dict(kind="fixed", order=4, partition_order=3)))
        out.append((f"verbatim_{bps}", _sig(3000, bps, 1, 2), 16000, bps, dict(kind="verbatim")))
    w = _sig(5000, 16, 1, 3) & ~15
    out += [
        ("constant", np.full((1, 4000), -1234, np.int64), 16000, 16, dict(kind="auto")),
        ("fixed0", _sig(3000, 16, 1, 4), 16000, 16, dict(kind="fixed", order=0)),
        ("lpc1", _sig(4000, 16, 1, 5), 16000, 16, dict(kind="lpc", order=1, precision=5)),
        ("lpc32_p15", _sig(9000, 16, 1, 6), 16000, 16, dict(kind="lpc", order=32, precision=15, block_size=4096)),
        ("lpc32_p15_24bit", _sig(9000, 24, 1, 7), 48000, 24, dict(kind="lpc", order=32, precision=15, block_size=4096, rice_method=1)),
        ("partition_order_15", _sig(2 ** 15 + 100, 16, 1, 8), 16000, 16, dict(kind="fixed", order=0, block_size=2 ** 15,
                                                                              partition_order=15)),
        ("escaped", _sig(6000, 16, 1, 9), 16000, 16, dict(kind="fixed", order=2, partition_order=3, escape=(0, 3, 5))),
        ("escaped_zero_bits", np.zeros((1, 4096), np.int64) + np.r_[np.zeros(2048), np.ones(2048)].astype(np.int64), 16000, 16,
         dict(kind="fixed", order=0, partition_order=1, escape=(0,))),
        ("rice5", _sig(5000, 16, 1, 10), 16000, 16, dict(kind="fixed", order=2, rice_method=1, partition_order=2)),
        ("wasted_bits", w, 16000, 16, dict(kind="lpc", order=8, wasted=True)),
        ("variable_blocks", _sig(7000, 16, 1, 11), 16000, 16, dict(block_sizes=[16, 4000, 1, 192, 2791], kind="lpc", order=1)),
        ("bs_uncommon_8", _sig(3000, 16, 1, 12), 16000, 16, dict(block_size=200, bs_code=6)),
        ("bs_uncommon_16", _sig(5000, 16, 1, 13), 16000, 16, dict(block_size=1000, bs_code=7)),
        ("sr_khz", _sig(3000, 16, 1, 14), 32000, 16, dict(sr_code=12)),
        ("sr_hz", _sig(3000, 16, 1, 15), 11025, 16, dict(sr_code=13)),
        ("sr_tens", _sig(3000, 16, 1, 16), 44100, 16, dict(sr_code=14)),
        ("sr_streaminfo", _sig(3000, 16, 1, 17), 16000, 16, dict(sr_code=0)),
        ("channels_6", _sig(3000, 16, 6, 18), 48000, 16, dict(kind="fixed", order=2)),
        ("false_sync", _sig(3000, 16, 1, 19), 16000, 16, dict(false_sync=True)),
    ]
    for st in ("independent", "left_side", "side_right", "mid_side"):
        for bps in (16, 24):
            out.append((f"{st}_{bps}", _sig(6000, bps, 2, 20), 44100, bps, dict(stereo=st, kind="lpc", order=12)))
    return out


CONSTRUCTS = _constructs()


def _expected(name, pcm, sr, kw):
    return fo.planted_samples(pcm, sr, kw.get("block_size", 1152)) if kw.get("false_sync") else pcm


# ------------------------------------------------------------------------------------------------ CPU
def test_crcs_match_known_values():
    assert flac.crc8(b"123456789") == 0xF4 and fo.crc8(b"123456789") == 0xF4                # CRC-8/SMBUS check value
    assert flac.crc16(b"123456789") == 0xFEE8 and fo.crc16(b"123456789") == 0xFEE8          # CRC-16/UMTS (BUYPASS) check value
    h = fo.frame_header(False, 4096, 16000, 0, 16, 0)
    assert flac.crc8(h[:-1]) == h[-1]


def test_parse_header_metadata_id3_and_total():
    x = _sig(5000, 16)
    base = flac.parse_flac(fo.encode(x, 16000, 16))
    assert (base.sample_rate, base.channels, base.bps, base.total_samples, base.max_block, base.variable) == (16000, 1, 16, 5000, 1152, False)
    both = fo.encode(x, 16000, 16, metadata=[(4, b"vorbis comment"), (1, b"\0" * 100), (6, b"picture")], id3=True)
    info = flac.parse_flac(both)
    assert info.total_samples == 5000 and both[info.audio_offset:info.audio_offset + 2] == b"\xff\xf8"
    assert info.audio_offset == base.audio_offset + 22 + 3 * 4 + 14 + 100 + 7
    for kw in (dict(), dict(block_sizes=[1000, 3000, 1000]), dict(block_size=1000, bs_code=7)):
        assert flac.parse_flac(fo.encode(x, 16000, 16, total_zero=True, **kw)).total_samples == 5000
    assert flac.parse_flac(fo.encode(x, 16000, 16, block_sizes=[1000, 3000, 1000])).variable


def test_rejections():
    good = fo.encode(_sig(3000, 16), 16000, 16)
    with pytest.raises(flac.FlacError, match="fLaC"):
        flac.parse_flac(b"RIFF" + good[4:])
    with pytest.raises(flac.FlacError, match="truncated"):
        flac.parse_flac(good[:20])
    with pytest.raises(flac.FlacError, match="STREAMINFO"):
        flac.parse_flac(b"fLaC" + bytes([0x84, 0, 0, 2, 0, 0]) + good[4:])
    s32 = bytearray(good)
    s32[4 + 4 + 12] = (s32[4 + 4 + 12] & 0xFE) | 1          # bits-per-sample - 1 = 31
    s32[4 + 4 + 13] |= 0xF0
    with pytest.raises(flac.FlacError) as e:
        flac.parse_flac(bytes(s32))
    assert e.value.code == _lib.ACB_ERR_UNSUPPORTED


@pytest.mark.parametrize("name", sorted(_manifest()))
def test_oracle_decodes_every_fixture(name):
    m = _manifest()[name]
    info, pcm = fo.decode(_fixture(name))
    assert pcm.shape == (m["channels"], m["samples"]) and info.sample_rate == m["sample_rate"] and info.bps == m["bps"]
    assert fo.pcm_sha256(pcm) == m["pcm_sha256"]
    h = flac.parse_flac(_fixture(name))
    assert (h.total_samples, h.channels, h.bps, h.sample_rate) == (m["samples"], m["channels"], m["bps"], m["sample_rate"])


@pytest.mark.parametrize("case", CONSTRUCTS, ids=[c[0] for c in CONSTRUCTS])
def test_oracle_round_trip_of_every_construct(case):
    name, pcm, sr, bps, kw = case
    info, out = fo.decode(fo.encode(pcm, sr, bps, **kw))
    assert np.array_equal(out, _expected(name, pcm, sr, kw))


def test_false_sync_is_planted():
    name, pcm, sr, bps, kw = next(c for c in CONSTRUCTS if c[0] == "false_sync")
    d = fo.encode(pcm, sr, bps, **kw)
    info = flac.parse_flac(d)
    syncs = [p for p in range(info.audio_offset, len(d) - 1) if fo.parse_frame_header(d, p) is not None]
    assert len(syncs) == len(range(0, pcm.shape[1], 1152)) + 1                    # every frame plus the planted one


def test_flac_symbols_exported(built_lib):
    assert _lib.exported_symbols_missing() == []
    lib = _lib.load()
    assert lib.acb_flac_candidate_capacity(800) == 116 and lib.acb_flac_candidate_capacity(-1) == -1
    assert lib.acb_flac_workspace_bytes(10, 3) == 10 * 24 + 16


# ------------------------------------------------------------------------------------------------ GPU
def _all_streams():
    out = [(n, _fixture(n), fo.decode(_fixture(n))[1]) for n in sorted(_manifest())]
    for name, pcm, sr, bps, kw in CONSTRUCTS:
        d = fo.encode(pcm, sr, bps, **kw)
        out.append((name, d, fo.decode(d)[1]))
    return out


def _check(res, streams, dtype):
    assert res.status.tolist() == [0] * len(streams)
    for i, (name, _, pcm) in enumerate(streams):
        got = res.clip(i).cpu().numpy()
        bps = res.infos[i].bps
        want = pcm.astype(np.int16) if dtype == torch.int16 else (pcm.astype(np.float64) / 2.0 ** (bps - 1)).astype(np.float32)
        assert got.dtype == want.dtype and np.array_equal(got, want), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.int16])
def test_every_stream_bit_exact(dtype):
    streams = _all_streams()
    if dtype == torch.int16:
        streams = [s for s in streams if flac.parse_flac(s[1]).bps == 16]
    res = acb.FlacDecoder("cuda:0").decode([s[1] for s in streams], dtype)
    _check(res, streams, dtype)


@pytest.mark.gpu
def test_launch_forms_are_bit_identical():
    dec = acb.FlacDecoder("cuda:0")
    streams = [s for s in _all_streams() if flac.parse_flac(s[1]).bps == 16]
    ragged = dec.decode([s[1] for s in streams], torch.int16)
    for i, s in enumerate(streams):                                               # per clip
        one = dec.decode([s[1]], torch.int16)
        assert one.status[0] == 0 and torch.equal(one.clip(0), ragged.clip(i)), s[0]
    d = fo.encode(_sig(16000, 16), 16000, 16, kind="lpc", order=8)                # uniform: the same stream many times
    uni = dec.decode([d] * 37, torch.float32)
    assert uni.status.tolist() == [0] * 37 and all(torch.equal(uni.clip(0), uni.clip(i)) for i in range(37))
    infos = [flac.parse_flac(s[1]) for s in streams]                              # caller-given offsets into a larger buffer
    offs = np.cumsum([0] + [i.channels * i.total_samples + 5 for i in infos[:-1]]).tolist()
    out = torch.full((offs[-1] + infos[-1].channels * infos[-1].total_samples + 5,), 7, dtype=torch.int16, device="cuda:0")
    st = dec.decode([s[1] for s in streams], torch.int16, out=out, out_offsets=offs)
    assert st.tolist() == [0] * len(streams)
    for i, (o, inf) in enumerate(zip(offs, infos)):
        n = inf.channels * inf.total_samples
        assert torch.equal(out[o:o + n].view(inf.channels, -1), ragged.clip(i)) and int(out[o + n]) == 7


@pytest.mark.gpu
def test_false_sync_rejected_and_clip_decodes():
    name, pcm, sr, bps, kw = next(c for c in CONSTRUCTS if c[0] == "false_sync")
    d = fo.encode(pcm, sr, bps, **kw)
    res = acb.FlacDecoder("cuda:0").decode([d], torch.int16)
    assert res.status[0] == 0
    assert np.array_equal(res.clip(0).cpu().numpy(), fo.planted_samples(pcm, sr, 1152).astype(np.int16))


@pytest.mark.gpu
def test_corrupt_and_truncated_clips_fail_alone():
    dec = acb.FlacDecoder("cuda:0")
    streams = [fo.encode(_sig(20000, 16, 1, s), 16000, 16, kind="lpc", order=8) for s in range(5)]
    good = dec.decode(streams, torch.int16)
    assert good.status.tolist() == [0] * 5
    flipped = bytearray(streams[1])
    info = flac.parse_flac(streams[1])
    flipped[info.audio_offset + 3000] ^= 0x10                                     # a residual bit of some frame
    truncated = streams[3][:-7]                                                   # the last frame loses its tail
    bad = dec.decode([streams[0], bytes(flipped), streams[2], truncated, streams[4]], torch.int16)
    assert bad.status.tolist() == [0, _lib.ACB_FLAC_NOT_TILED, 0, _lib.ACB_FLAC_NOT_TILED, 0]
    for i in (0, 2, 4):
        assert torch.equal(bad.clip(i), good.clip(i))


@pytest.mark.gpu
def test_guard_bytes_are_never_read():
    """Each region sits between guard bytes that would change the result if read: before it, a copy of another stream's frames;
    after it, the missing tail of its own last frame (a clip cut short must fail, not read on) or sync-like garbage."""
    dec = acb.FlacDecoder("cuda:0")
    streams = [fo.encode(_sig(9000 + 1000 * s, 16, 1, s), 16000, 16, kind="fixed", order=2) for s in range(4)]
    infos = [flac.parse_flac(s) for s in streams]
    regions = [s[i.audio_offset:] for s, i in zip(streams, infos)]
    buf, offs, cut_infos, expect = bytearray(), [], [], []
    for k, (r, inf) in enumerate(zip(regions, infos)):
        buf += regions[(k + 1) % 4][:200]                                        # guard before: frames of another stream
        offs.append(len(buf))
        cut = 5 if k % 2 else 0
        buf += r
        if not cut:
            buf += b"\xff\xf8" * 40                                              # guard after: sync bytes
        cut_infos.append(inf._replace(audio_length=len(r) - cut))
        expect.append(_lib.ACB_FLAC_NOT_TILED if cut else 0)
    data = torch.frombuffer(buf, dtype=torch.uint8).to("cuda:0")
    res = dec.decode_regions(None, cut_infos, torch.int16, data=data, byte_offsets=offs)
    assert res.status.tolist() == expect
    for k in (0, 2):
        assert np.array_equal(res.clip(k).cpu().numpy(), fo.decode(streams[k])[1].astype(np.int16))


def _wav_and_flac(root, rel, sr, pcm):
    from scipy.io import wavfile
    os.makedirs(os.path.dirname(str(root / rel)), exist_ok=True)
    wavfile.write(str(root / (rel + ".wav")), sr, np.ascontiguousarray(pcm.T.astype(np.int16)))
    with open(str(root / (rel + "_f.flac")), "wb") as f:
        f.write(fo.encode(pcm, sr, 16, kind="lpc", order=8, block_size=4096))


@pytest.mark.gpu
def test_driver_flac_and_wav_payloads_are_identical(tmp_path):
    root, out = tmp_path / "in", tmp_path / "out"
    cases = {"19/198/19-198-0001": (16000, _sig(40000, 16, 1, 1)), "19/198/19-198-0002": (16000, _sig(30000, 16, 2, 2)),
             "19/227/19-227-0001": (24000, _sig(36001, 16, 1, 3)), "26/495/26-495-0001": (48000, _sig(50000, 16, 2, 4))}
    for rel, (sr, pcm) in cases.items():
        _wav_and_flac(root, rel, sr, pcm)
    for d in ("19/198", "19/227", "26/495"):
        ids = sorted(os.path.splitext(f)[0] for f in os.listdir(str(root / d)))
        with open(str(root / d / (d.replace("/", "-") + ".trans.txt")), "w") as f:
            f.writelines(f"{i} TEXT OF {i.upper()}\n" for i in ids)
    bad = bytearray(fo.encode(_sig(20000, 16, 1, 9), 16000, 16, kind="lpc", order=8))
    bad[len(bad) // 2] ^= 0x01
    with open(str(root / "26/495/26-495-0009_f.flac"), "wb") as f:
        f.write(bytes(bad))
    args = types.SimpleNamespace(dataset_name="librispeech", in_dir=str(root), out_dir=str(out), vae_ckpt=None, mel_only=True,
                                 cv_tsv=None, num_gpus=1, workers_per_gpu=2, force=False)
    runner = pd.ShardRunner(args, 0, batch_samples=200000, decode_threads=2)
    runner.run(pd.scan_files(str(root)))
    assert [os.path.basename(e[0]) for e in runner.errors] == ["26-495-0009_f.flac"] and "FLAC" in runner.errors[0][1]
    for rel in cases:
        a = torch.load(str(out / (rel + ".pt")))["mel"]
        b = torch.load(str(out / (rel + "_f.pt")))["mel"]
        assert a.shape == b.shape and torch.equal(a, b), rel
    with open(str(out / "19/198/198.trans.txt")) as f:
        lines = sorted(f.read().splitlines())
    assert lines == sorted(f"{i} TEXT OF {i.upper()}" for i in ("19-198-0001", "19-198-0001_f", "19-198-0002", "19-198-0002_f"))
    assert not os.path.exists(str(out / "26/495/26-495-0009_f.pt"))
