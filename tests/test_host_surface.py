"""The C++ host's drop-in surface: flattening identical to the reference object graph,
parser grammar / warnings / error strings, CLI messages and exit codes, PNG writer."""
import hashlib
import os
import subprocess
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, PKG_DIR, decode_png, quantize, scene_path

ALL_SCENES = sorted(p for p in list((GOLDEN / "inputs").glob("*.rti")) + list((GOLDEN / "excess_inputs").glob("*.rti"))
                    if p.name not in ("teapot.rti",))   # excess teapot.rti has no teapot.obj beside it


@pytest.mark.parametrize("path", ALL_SCENES, ids=lambda p: p.parent.name + "/" + p.name)
def test_flatten_is_byte_identical_to_reference_object_graph(pkg, reference, path):
    """Transforms (Eigen translate/scale/rotate/inverse/determinant restated in vecmath.h),
    the +-eps `tri` pair, .obj fan triangulation, normals, bounding boxes, materials, lights
    and camera: every byte of the flat descriptor equals what the reference builds."""
    ours = pkg.flat_arrays(pkg.HostScene.load(path).flat)
    theirs = pkg.flat_arrays(reference.flatten(reference.load(path)))
    for key, val in theirs.items():
        if isinstance(val, np.ndarray):
            assert np.array_equal(ours[key], val), key
        else:
            assert ours[key] == val, key


def _write(tmp_path, name, text):
    p = tmp_path / name
    p.write_text(text)
    return p


BAD_RTI = [
    ("cam 0 0 1\n", "line 1: cam requires 15 parameters"),
    ("sph 1 2 3\n", "line 1: sph requires 4 parameters"),
    ("\n\nltp 1 2 3 4 5\n", "line 3: ltp requires at least 6 parameters"),
    ("mat 1 2 3\n", "line 1: mat requires at least 13 parameters"),
    ("sph 1 2 x 4\n", "line 1: invalid number x"),
    ("ltd 0 0 0 1 1 1\n", "line 1: zero direction specified"),
    ("obj\n", "line 1: obj requires a filename"),
    ("obj \"nope.obj\"\n", "file not found: "),
    ("sph 1 2 3 \"4\n", "line 1: unclosed quotes"),
    ("sph 1 2 3 4\n", "At least one camera must be specified."),
]


@pytest.mark.parametrize("text,msg", BAD_RTI)
def test_rti_errors_match_reference(pkg, live_reference, tmp_path, text, msg):
    """The message the reference gives for this input; the whole string equals the live reference's where it is built."""
    p = _write(tmp_path, "bad.rti", text)
    with pytest.raises(pkg.RtError) as ours:
        pkg.HostScene.load(p)
    assert msg in str(ours.value)
    if live_reference is not None:
        with pytest.raises(RuntimeError) as theirs:
            live_reference.load(p)
        assert str(ours.value) == str(theirs.value)


BAD_OBJ = [
    ("v 1 2\n", "line 1: v requires 3 or 4 parameters"),
    ("v 1 2 3 0\n", "line 1: v must be a point vector"),
    ("vn 1 2\n", "line 1: vn requires 3 parameters"),
    ("v 0 0 0\nv 1 0 0\nf 1 2\n", "line 3: f requires at least 3 vertices"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 9\n", "line 4: vertex index out of range"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 -1\n", "line 4: index must be positive"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 x\n", "line 4: invalid integer x"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 /3\n", "line 4: vertex index is required"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1//5 2 3\n", "line 4: normal index out of range"),
]


@pytest.mark.parametrize("text,msg", BAD_OBJ)
def test_obj_errors_match_reference(pkg, live_reference, tmp_path, text, msg):
    """The message the reference gives for this input; the whole string equals the live reference's where it is built."""
    _write(tmp_path, "m.obj", text)
    p = _write(tmp_path, "s.rti", "cam 0 0 5 -1 -1 1 1 -1 1 -1 1 1 1 1 1\nobj m.obj\n")
    with pytest.raises(pkg.RtError) as ours:
        pkg.HostScene.load(p)
    assert msg in str(ours.value)
    if live_reference is not None:
        with pytest.raises(RuntimeError) as theirs:
            live_reference.load(p)
        assert str(ours.value) == str(theirs.value)


def test_grammar_corner_cases_flatten_like_reference(pkg, reference, tmp_path):
    """comments, quoted tokens, tabs/CR, partial numbers (stod prefix rule), extra parameters,
    unknown statements, optional parameters, polygon fans, v/vt/vn corners, degenerate faces,
    zero rotation, several input files populating one scene."""
    _write(tmp_path, "m.obj", "# c\nv 0 0 0\nv 1 0 0 1\nv 1 1 0\nv 0 1 0\nv 2 2 2\nvt 0 0\nvn 0 0 1\nvn 0 1 1\n"
                              "f 1/1/1 2/1/2 3//1 4\nf 1 1 2\nf 1 2 5\ng grp\n")
    a = _write(tmp_path, "a.rti",
               "# comment line\n\ncam 0 0 5 -1 -1 1 1 -1 1 -1 1 1 1 1 1   # trailing comment\n"
               "mat 0.1 0.2 0.3 \"0.4\" 0.5 0.6 0.7 0.8 0.9 3.5e0 0.1 0.2 0.3\r\n"
               "xft 1 2 3\n\txfr 0 0 0\nxfr 10 20 30\nxfs 1 2 0.5\nsph 0 0 0 1.25abc 7 8\nwhatever 1 2\n"
               "ltp 1 2 3 0.5 0.5 0.5\nltp 1 2 3 0.5 0.5 0.5 2\nltd 0 -2 0 1 1 1\nlta .1 .2 .3\n"
               "obj \"m.obj\" ignored\nxfz\ntri 0 0 0 1 0 0 0 1 0\n")
    b = _write(tmp_path, "b.rti", "mat 1 1 1 1 1 1 1 1 1 1 1 1 1 1 1 1 1.5\nxfs -1 1 1\nsph 1 1 1 2\n")
    ours = pkg.flat_arrays(pkg.HostScene.load(a, b).flat)
    theirs = pkg.flat_arrays(reference.flatten(reference.load(a, b)))
    assert theirs["num_geometries"] == 4 and theirs["num_lights"] == 4
    for key, val in theirs.items():
        if isinstance(val, np.ndarray):
            assert np.array_equal(ours[key], val), key
        else:
            assert ours[key] == val, key


def test_warnings_on_stderr(pkg, tmp_path, capfd):
    _write(tmp_path, "m.obj", "v 0 0 0\nv 1 0 0\nv 0 1 0\nusemtl x\nf 1 1 2\nf 1 2 3\n")
    p = _write(tmp_path, "s.rti", "cam 0 0 5 -1 -1 1 1 -1 1 -1 1 1 1 1 1\nfoo 1\nsph 0 0 0 1 9\nobj m.obj\n")
    pkg.HostScene.load(p)
    err = capfd.readouterr().err
    assert "Warning: line 2: unknown line type foo" in err
    assert "Warning: line 3: extra parameters found" in err
    assert "Warning: line 4: unknown obj line type usemtl" in err
    assert "Warning: line 5: degenerate face" in err


AS2 = PKG_DIR / "bin" / "as2"
CLI_ERRORS = [
    ([], "Error: At least one input file must be specified."),
    (["x.rti"], "Error: An output file must be specified."),
    (["-t", "0", "-o", "o.png", "x.rti"], "Error: Thread count must be positive."),
    (["-t", "zz", "-o", "o.png", "x.rti"], "Error: Thread count is invalid."),
    (["-w", "-3", "-o", "o.png", "x.rti"], "Error: Width and/or height must be positive."),
    (["-h", "abc", "-o", "o.png", "x.rti"], "Error: Width and/or height is invalid."),
    (["--bdepth", "-1", "-o", "o.png", "x.rti"], "Error: Bounce depth must be non-negative."),
    (["--aa", "0", "-o", "o.png", "x.rti"], "Error: Sample count must be between 1 and 16."),
    (["--aa", "q", "-o", "o.png", "x.rti"], "Error: Sample count is invalid."),
    (["--aa", "2", "--intersection-only", "-o", "o.png", "x.rti"], "Error: --aa cannot be combined with --intersection-only."),
    (["--help"], "Usage: "),
    (["-o", "/nonexistent-dir/o.png", "x.rti"], "Error: Output file is not writable."),
]


@pytest.mark.parametrize("argv,msg", CLI_ERRORS)
def test_cli_messages_and_exit_code(pkg, tmp_path, argv, msg):
    """src/options.cpp:20-90 and src/main.cpp:40-66: messages on stderr, exit code 1."""
    proc = subprocess.run([str(AS2)] + argv, cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode == 1
    assert msg in proc.stderr


def test_cli_parse_error_and_missing_camera(pkg, tmp_path):
    bad = _write(tmp_path, "bad.rti", "sph 1 2\n")
    proc = subprocess.run([str(AS2), "-o", "o.png", str(bad)], cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode == 1 and "Error: line 1: sph requires 4 parameters" in proc.stderr
    nocam = _write(tmp_path, "nocam.rti", "sph 1 2 3 4\n")
    proc = subprocess.run([str(AS2), "-o", "o.png", str(nocam)], cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode == 1 and "Error: At least one camera must be specified." in proc.stderr
    assert not (tmp_path / "o.png").exists()      # the probe file is removed (src/main.cpp:50)


def test_cli_without_gpu_fails_loudly(pkg, tmp_path):
    """No CPU fallback: on a box without a B200 the render step reports an error, exit 1."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    proc = subprocess.run([str(AS2), "-o", "o.png", "-w", "8", "-h", "8", str(scene_path("inputs/input-01.rti"))],
                          cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode == 1
    assert "Error: no usable CUDA device" in proc.stderr and "no CPU fallback" in proc.stderr


def test_png_writer_roundtrip_and_quantisation(pkg, tmp_path):
    rng = np.random.default_rng(3)
    rgb = rng.uniform(-0.2, 1.3, size=(37, 53, 3))
    rgb[0, 0] = [1.0, 0.999, 0.0]
    rgb[0, 1] = [np.nan, 254.5 / 255.0, 0.5]
    q = pkg.quantize_rgb8(rgb)
    assert np.array_equal(q, quantize(rgb))
    assert list(q[0, 0]) == [255, 254, 0]          # truncation, not rounding (src/writers.cpp:7)
    path = tmp_path / "o.png"
    pkg.write_png(path, q)
    assert np.array_equal(decode_png(path), q)
    raw = path.read_bytes()
    assert raw[:8] == b"\x89PNG\r\n\x1a\n" and raw[12:16] == b"IHDR"
    assert int.from_bytes(raw[16:20], "big") == 53 and int.from_bytes(raw[20:24], "big") == 37


def test_synthetic_scene_text_equals_in_memory(pkg, tmp_path):
    """The synthetic benchmark scene written as .rti/.obj and parsed back flattens to the
    same bytes as the in-memory fast path (numbers are printed %.17g)."""
    import ctypes as C
    lib = pkg.load_host()
    err = C.create_string_buffer(256)
    rti, obj = tmp_path / "syn.rti", tmp_path / "syn.obj"
    assert lib.as2_write_synthetic(str(rti).encode(), str(obj).encode(), 12, 9, 184, err, 256) == 0, err.value
    a = pkg.flat_arrays(pkg.HostScene.load(rti).flat)
    b = pkg.flat_arrays(pkg.HostScene.synthetic(12, 9, 184).flat)
    assert a["num_faces"] == 12 * 12 * 2 and a["num_geometries"] == 10
    for key, val in a.items():
        if isinstance(val, np.ndarray):
            assert np.array_equal(b[key], val), key
        else:
            assert b[key] == val, key
    sha = hashlib.sha256(rti.read_bytes() + obj.read_bytes()).hexdigest()
    assert sha == hashlib.sha256(rti.read_bytes() + obj.read_bytes()).hexdigest()


def _decode_png_bytes(data):
    """Minimal PNG reader for the writer's own subset (8-bit RGB, filter 0): checks every chunk CRC and the
    zlib stream's adler32 (zlib.decompress does), so a stitching error in the striped encoder cannot hide."""
    import struct
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, idat, w, h = 8, b"", 0, 0
    while pos < len(data):
        (n,) = struct.unpack(">I", data[pos:pos + 4])
        typ, body = data[pos + 4:pos + 8], data[pos + 8:pos + 8 + n]
        (crc,) = struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(typ + body) == crc, typ
        if typ == b"IHDR":
            w, h, depth, ctype, comp, flt, lace = struct.unpack(">IIBBBBB", body)
            assert (depth, ctype, comp, flt, lace) == (8, 2, 0, 0, 0)
        elif typ == b"IDAT":
            idat += body
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), dtype=np.uint8).reshape(h, 1 + 3 * w)
    assert (raw[:, 0] == 0).all()
    return raw[:, 1:].reshape(h, w, 3)


@pytest.mark.parametrize("shape", [(1, 1), (3, 5), (64, 64), (257, 130), (1000, 333)])
@pytest.mark.parametrize("threads", [1, 2, 3, 8, 64])
def test_png_striped_encoder_is_a_valid_stream(pkg, shape, threads):
    """SURVEY section 8 f-2: the rows are deflated in parallel stripes stitched into ONE zlib stream."""
    rng = np.random.default_rng(shape[0] * 1000 + threads)
    img = rng.integers(0, 256, size=(shape[0], shape[1], 3), dtype=np.uint8)
    img[shape[0] // 2:, :, :] = 17          # a compressible half, so stripes differ in ratio
    data = pkg.encode_png(img, threads)
    assert np.array_equal(_decode_png_bytes(data), img)
    if threads == 1:
        from PIL import Image
        import io
        assert np.array_equal(np.array(Image.open(io.BytesIO(data)).convert("RGB")), img)


def test_png_striped_encoder_matches_pil_on_a_rendered_like_frame(pkg, tmp_path):
    yy, xx = np.mgrid[0:540, 0:960]
    img = np.stack([(xx * 255 // 959), (yy * 255 // 539), ((xx + yy) % 256)], axis=-1).astype(np.uint8)
    path = tmp_path / "g.png"
    pkg.write_png(path, img)                  # default thread count of the box
    assert np.array_equal(decode_png(path), img)


# ---- SURVEY section 8 f-1: the chunked (multi-threaded) .obj parser ---------------------------------
def _chunked(monkeypatch, threads, chunk_bytes):
    monkeypatch.setenv("AS2_PARSE_THREADS", str(threads))
    monkeypatch.setenv("AS2_PARSE_CHUNK_BYTES", str(chunk_bytes))


@pytest.mark.parametrize("threads", [2, 3, 7, 16])
@pytest.mark.parametrize("scene", ["inputs/input-02.rti", "excess_inputs/bunny4.rti", "excess_inputs/test.rti"])
def test_chunked_obj_parse_equals_serial_and_reference(pkg, live_reference, monkeypatch, scene, threads):
    """The chunked parse flattens to the bytes of the live reference's object graph where that is built, else to
    the bytes of the one-thread parse."""
    path = scene_path(scene)
    if not path.exists():
        pytest.skip(f"{scene} not shipped")
    if live_reference is not None:
        theirs = pkg.flat_arrays(live_reference.flatten(live_reference.load(path)))
    else:
        _chunked(monkeypatch, 1, 4096)
        theirs = pkg.flat_arrays(pkg.HostScene.load(path).flat)
    _chunked(monkeypatch, threads, 4096)
    ours = pkg.flat_arrays(pkg.HostScene.load(path).flat)
    for key, val in theirs.items():
        if isinstance(val, np.ndarray):
            assert np.array_equal(ours[key], val), key
        else:
            assert ours[key] == val, key


@pytest.mark.parametrize("threads", [2, 5])
@pytest.mark.parametrize("text,msg", BAD_OBJ + [
    # the reference validates corner k before it parses corner k+1, and reads line by line
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 9 x\n", "line 4: vertex index out of range"),
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\nf 1 2 9\nv 1\n", "line 5: vertex index out of range"),
    ("v 0 0 0\nv 1 0 0\nf 1 2 3\nv 0 1 0\n", "line 3: vertex index out of range"),      # defined too late
    ("v 0 0 0\nv 1 0 0\nv 0 1 0\nv 1\nf 1 2 9\n", "line 4: v requires 3 or 4 parameters"),
])
def test_chunked_obj_errors_match_reference(pkg, live_reference, tmp_path, monkeypatch, text, msg, threads):
    """The chunked parse reports the live reference's error where that is built, else the one-thread parse's."""
    _write(tmp_path, "m.obj", "# pad pad pad pad\n" * 0 + text)
    p = _write(tmp_path, "s.rti", "cam 0 0 5 -1 -1 1 1 -1 1 -1 1 1 1 1 1\nobj m.obj\n")
    if live_reference is not None:
        with pytest.raises(RuntimeError) as theirs:
            live_reference.load(p)
    else:
        _chunked(monkeypatch, 1, 8)
        with pytest.raises(pkg.RtError) as theirs:
            pkg.HostScene.load(p)
    _chunked(monkeypatch, threads, 8)
    with pytest.raises(pkg.RtError) as ours:
        pkg.HostScene.load(p)
    assert msg in str(ours.value)
    assert str(ours.value) == str(theirs.value)


def test_chunked_obj_warnings_come_in_line_order_and_stop_at_the_error(pkg, tmp_path, monkeypatch, capfd):
    body = "v 0 0 0\nv 1 0 0\nv 0 1 0\ng a\nf 1 1 2\ns off\nf 1 2 3\nf 1 2 2\nusemtl m\n"
    _write(tmp_path, "m.obj", body)
    p = _write(tmp_path, "s.rti", "cam 0 0 5 -1 -1 1 1 -1 1 -1 1 1 1 1 1\nobj m.obj\n")
    _chunked(monkeypatch, 4, 8)
    scene = pkg.HostScene.load(p)
    assert pkg.flat_arrays(scene.flat)["num_faces"] == 1
    err = [l for l in capfd.readouterr().err.splitlines() if l.startswith("Warning")]
    assert err == ["Warning: line 4: unknown obj line type g", "Warning: line 5: degenerate face",
                   "Warning: line 6: unknown obj line type s", "Warning: line 8: degenerate face",
                   "Warning: line 9: unknown obj line type usemtl"]
    _write(tmp_path, "m.obj", body + "f 1 2 7\nfoo\n")
    with pytest.raises(pkg.RtError):
        pkg.HostScene.load(p)
    err2 = [l for l in capfd.readouterr().err.splitlines() if l.startswith("Warning")]
    assert err2 == err          # nothing after the failing line 10 is reported
