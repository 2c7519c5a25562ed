"""The drop-in decoder's hash check, without the reference decoder: every committed capture of a decoded picture goes through
the library the way the drop-in DecoderApp calls it (upload, then ilf_deblock -> ilf_sao -> ilf_alf on the device, download;
vvcsoftware_vtm_b200/shim/ilf_shim.cpp), and the MD5 of each plane of the result must be the one the reference encoder wrote
for that picture into the committed bitstream's decoded-picture-hash SEI (PicYuvMD5.cpp, SEIDecodedPictureHash=1)."""
import hashlib
import os
import re

import numpy as np
import pytest

import golden_io as G
from test_gpu_parity import _ctx, _set_all

K = G.K
# pictures per committed 416x240 stream (tests/test_gpu_decoder_dropin.py STREAMS)
PICTURES = {"intra_416x240": 8, "ra_416x240": 17, "ldp_416x240": 6, "ldb_416x240": 6}
DECODED = [p for p in G.golden_files() if "_enc_" not in os.path.basename(p)]


def sei_picture_md5(stream):
    """[Y, Cb, Cr] MD5 digests of every picture of a committed stream, in decoding order: the payloads of its suffix SEI NAL
    units (type 40) that carry a decoded-picture hash (payloadType 132, payloadSize 49, hash_type 0 = MD5)."""
    with open(os.path.join(G.ROOT, "tests", "golden", "streams", stream + ".bin"), "rb") as fh:
        data = fh.read()
    out = []
    for nal in re.split(b"\x00\x00\x01", data)[1:]:
        nal = nal.rstrip(b"\x00").replace(b"\x00\x00\x03", b"\x00\x00")     # trailing zero bytes, emulation prevention
        if nal[0] >> 1 == 40 and nal[2:5] == b"\x84\x31\x00":
            out.append([nal[5 + 16 * i:21 + 16 * i] for i in range(3)])
    return out


def picture_md5(pic):
    """PicYuvMD5.cpp's digest of each plane: samples of more than 8 bits as two bytes, little endian."""
    return [hashlib.md5(np.ascontiguousarray(pic[k]).astype("<u2").tobytes()).digest() for k in K]


def _stream_and_index(path):
    stream, index = os.path.basename(path)[:-len(".npz")].rsplit("_", 1)
    return stream, int(index)


def test_captures_carry_their_streams_hash_sei():
    """The committed captures are the pictures the bitstreams' SEI describes (so the GPU test below checks against the encoder)."""
    for stream, n in PICTURES.items():
        assert len(sei_picture_md5(stream)) == n, stream
    for path in DECODED:
        c = G.load_golden(path)
        stream, index = _stream_and_index(path)
        last = [s for s in ("dbk", "sao", "alf") if f"{s}_y" in c][-1]
        assert picture_md5({k: c[f"{last}_{k}"] for k in K}) == sei_picture_md5(stream)[index], os.path.basename(path)


@pytest.mark.gpu
@pytest.mark.parametrize("path", DECODED, ids=os.path.basename)
def test_drop_in_call_sequence_passes_the_streams_hash_sei(path, ilf_lib):
    c = G.load_golden(path)
    stream, index = _stream_and_index(path)
    with _ctx(ilf_lib, c) as f:
        f.upload(0, *(c[f"pre_{k}"] for k in K))
        _set_all(f, 0, c)
        f.loop_filter_pic(0)
        if "sao_y" in c:
            f.sao_process(0)
        if "alf_y" in c:
            f.alf_process(0)
        got = picture_md5(f.download(0))
    want = sei_picture_md5(stream)[index]
    bad = [k for k, a, b in zip(K, got, want) if a != b]
    assert not bad, f"{stream} picture {index}: planes {bad} do not match the bitstream's decoded-picture hash"
