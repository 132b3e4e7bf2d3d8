"""Host pieces of the folder pipeline's mixed route (no GPU needed): input geometry, the readers, the output writers, the
routing rule and the engine's grouping of a batch into one-width chunks."""
import struct

import numpy as np
import pytest
import torch
from PIL import Image

from oracle import synth


def _write_bmp(path, rgb, top_down=False, bpp=24):
    h, w, _ = rgb.shape
    pitch = (w * bpp // 8 + 3) & ~3
    buf = np.zeros((h, pitch), np.uint8)
    px = (rgb if top_down else rgb[::-1])[:, :, ::-1]
    if bpp == 32:
        px = np.dstack([px, np.full((h, w, 1), 255, np.uint8)])
    buf[:, :w * bpp // 8] = px.reshape(h, -1)
    with open(path, 'wb') as f:
        f.write(b'BM' + struct.pack('<IHHI', 54 + buf.size, 0, 0, 54))
        f.write(struct.pack('<IiiHHIIiiII', 40, w, -h if top_down else h, 1, bpp, 0, buf.size, 2835, 2835, 0, 0))
        f.write(buf.tobytes())


@pytest.mark.parametrize('top_down', [False, True])
def test_bmp_pixel_arrays_are_read_as_the_per_image_route_reads_them(tmp_path, top_down):
    from neuralbarkcalculator_b200 import pipeline
    from neuralbarkcalculator_b200.dataset import read_bmp_pixels
    img = synth.texture_u8(37, 1001, 3)           # 3003 bytes of pixels per row, padded to 3004
    p = str(tmp_path / 'x.bmp')
    _write_bmp(p, img, top_down)
    geo = pipeline.raw_geometry(p)
    buf, H, W, pitch, bgr, bottom_up = read_bmp_pixels(p)
    assert geo == (54, H, W, pitch, bgr, bottom_up) == (54, 37, 1001, 3004, True, not top_down)
    pinned = torch.zeros(H * pitch + 100, dtype=torch.uint8)
    assert pipeline.read_raw(p, geo, pinned, True, 1024) == (0, H)
    assert np.array_equal(pinned[:H * pitch].numpy(), buf)


def test_other_inputs_are_decoded_by_pil_loader(tmp_path):
    """PNG (RGB, grey, RGBA, palette), JPEG and a 32-bit BMP: RGB top-down rows, exactly dataset.pil_loader's pixels."""
    from neuralbarkcalculator_b200 import pipeline
    from neuralbarkcalculator_b200.dataset import pil_loader
    img = synth.texture_u8(30, 41, 5)
    files = {'rgb.png': Image.fromarray(img), 'grey.png': Image.fromarray(img[:, :, 0]),
             'rgba.png': Image.fromarray(np.dstack([img, img[:, :, :1]])), 'pal.png': Image.fromarray(img).quantize(16),
             'j.jpg': Image.fromarray(img), 't.tif': Image.fromarray(img)}
    for name, im in files.items():
        im.save(str(tmp_path / name))
    _write_bmp(str(tmp_path / 'b32.bmp'), img, bpp=32)
    for name in list(files) + ['b32.bmp']:
        p = str(tmp_path / name)
        geo = pipeline.raw_geometry(p)
        assert geo == (None, 30, 41, 123, False, False), name
        buf = torch.zeros(30 * 123, dtype=torch.uint8)
        assert pipeline.read_raw(p, geo, buf, True, 1024) == (0, 30)
        assert np.array_equal(buf.numpy().reshape(30, 41, 3), pil_loader(p)), name


def test_zero_band_span_of_a_decoded_scan(tmp_path):
    """A decoded image of 4 target x 4 target pixels is reduced to the rows between its all-zero bands."""
    from neuralbarkcalculator_b200 import pipeline
    img = np.zeros((64, 64, 3), np.uint8)
    img[13:40] = 7
    p = str(tmp_path / 's.png')
    Image.fromarray(img).save(p)
    geo = pipeline.raw_geometry(p)
    buf = torch.zeros(64 * 64 * 3, dtype=torch.uint8)
    assert pipeline.read_raw(p, geo, buf, True, 16) == (12, 28)
    assert pipeline.read_raw(p, geo, buf, False, 16) == (0, 64)
    assert pipeline.read_raw(p, geo, buf, True, 1024) == (0, 64)      # not a 4x scan for this target


def test_outputs_keep_the_format_their_extension_names(tmp_path):
    from neuralbarkcalculator_b200 import pipeline
    img = synth.texture_u8(20, 30, 1)
    mask = synth.class_mask(20, 30, 2)
    for name, fmt in (('a.png', 'PNG'), ('a.jpg', 'JPEG'), ('a.tif', 'TIFF'), ('a.PNG', 'PNG')):
        p = str(tmp_path / name)
        pipeline.save_image(p, img, 1)
        with Image.open(p) as im:
            assert im.format == fmt
            if fmt != 'JPEG':
                assert np.array_equal(np.asarray(im), img)
        pipeline.save_image(p, mask, 1, lut=pipeline._DUAL_LUT)
        with Image.open(p) as im:
            assert im.mode == 'L'
            if fmt != 'JPEG':
                assert np.array_equal(np.asarray(im), pipeline._DUAL_LUT[mask])


def test_processed_size_follows_the_preprocessor_routing():
    from neuralbarkcalculator_b200 import ops
    assert ops.processed_size(4096, 4096) == (1024, 1024)
    assert ops.processed_size(3000, 2000) == (1024, 1024)
    assert ops.processed_size(1025, 10) == (1024, 1024)
    assert ops.processed_size(1024, 1024) == (1024, 1024)
    assert ops.processed_size(900, 700) == (900, 700)
    assert ops.processed_size(700, 1024) == (700, 1024)


def test_mixed_batches_group_by_width():
    """Full-width images first, then one chunk family per narrower width, chunks never longer than the engine's."""
    from neuralbarkcalculator_b200.engine import PredictEngine
    eng = PredictEngine(None, 'cpu', chunk=3)
    widths = [1024, 700, 1024, 600, 700, 1024, 1024, 700, 700, 1024]
    order, chunks = eng._mixed_chunks(widths)
    assert sorted(order) == list(range(len(widths)))
    assert [widths[i] for i in order] == sorted(widths, key=lambda w: (w != 1024, w))
    assert chunks == [(0, 3, 1024), (3, 5, 1024), (5, 6, 600), (6, 9, 700), (9, 10, 700)]
    assert order[:5] == [0, 2, 5, 6, 9]            # stable: dataset order inside a width


def test_mixed_descs_layout():
    from neuralbarkcalculator_b200 import _lib, ops
    import ctypes as C
    assert C.sizeof(_lib.MixedDesc) == 40
    d = ops.mixed_descs([(1234, 4096, 4096, 12288, True, True, (8, 400)), (None, 30, 41, 123, False, False, (0, 30))])
    assert (d[0].raw, d[0].H, d[0].W, d[0].pitch, d[0].flags, d[0].span_row0, d[0].span_rows) == (1234, 4096, 4096, 12288, 3, 8, 400)
    assert (d[1].raw, d[1].flags) == (None, 0)


def test_mixed_kernel_refuses_bad_descriptors(libnbc):
    """Argument checks run on the host before anything is launched."""
    from neuralbarkcalculator_b200 import _lib, ops
    import ctypes as C
    ws = np.zeros(1 << 16, np.uint8)
    out = np.zeros(16, np.uint8)
    fl = np.zeros(2, np.int32)

    def call(items, target=1024, stride=1 << 30):
        d = ops.mixed_descs(items)
        return libnbc.nbc_preprocess_mixed_batch_u8(d, len(items), target, C.c_void_p(out.ctypes.data), stride,
                                                    C.c_void_p(fl.ctypes.data), C.c_void_p(ws.ctypes.data), ws.size, None)
    assert call([(1, 900, 700, 2100, False, False, (0, 900))]) != 0 and 'workspace' in _lib.last_error()
    big = libnbc.nbc_preprocess_mixed_workspace_bytes(None, 1, 1024)
    assert big > 3 * 1024 * 1024
    ws = np.zeros(big, np.uint8)
    assert call([(1, 900, 700, 2000, False, False, (0, 900))]) != 0 and 'pitch' in _lib.last_error()
    assert call([(1, 900, 700, 2100, False, False, (8, 800))]) != 0 and 'only a 4 * target square' in _lib.last_error()
    assert call([(1, 4096, 4096, 12288, False, False, (2, 400))]) != 0 and 'groups of 4' in _lib.last_error()
    assert call([(1, 900, 700, 2100, False, False, (0, 900))], stride=100) != 0 and 'stride' in _lib.last_error()

