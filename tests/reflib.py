"""ctypes bindings for oracle/_ref/libguetzli_ref.so (the unmodified reference,
test infrastructure only).  See oracle/ref_hooks.cc for what each hook wraps."""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(_HERE, "..", "oracle", "_ref", "libguetzli_ref.so")
_lib = None


def available():
    return os.path.exists(REF_SO)


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(REF_SO)
        _lib.gref_target_for_quality.restype = C.c_double
        _lib.gref_target_for_quality.argtypes = [C.c_double]
        _lib.gref_mask_lut.restype = C.c_double
        _lib.gref_mask_lut.argtypes = [C.c_int, C.c_double]
        _lib.gref_gamma.restype = C.c_double
        _lib.gref_gamma.argtypes = [C.c_double]
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def target_for_quality(q):
    return float(np.float32(lib().gref_target_for_quality(float(q))))


def score_for_quality(q):
    """ButteraugliScoreForQuality in double precision (target_for_quality narrows it to float)."""
    return lib().gref_target_for_quality(float(q))


def process_rgb(rgb, quality=95.0, trace=True, lookahead=3, new_zeroing_model=True, try_420=False, force_420=False,
                clear_metadata=True):
    """-> (ok, jpeg bytes, trace str, counters[3], seconds)"""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = rgb.shape
    out = C.POINTER(C.c_uint8)()
    out_len = C.c_size_t()
    tr = C.c_char_p()
    tr_len = C.c_size_t()
    counters = (C.c_int * 3)()
    secs = C.c_double()
    lib().gref_set_420(int(try_420), int(force_420))
    lib().gref_set_clear_metadata(int(clear_metadata))
    try:
        ok = lib().gref_process_rgb_ex(
            _p(rgb, C.c_uint8), w, h, C.c_float(target_for_quality(quality)), int(lookahead), int(new_zeroing_model),
            C.byref(out), C.byref(out_len),
            C.byref(tr) if trace else None, C.byref(tr_len), counters, C.byref(secs))
    finally:
        lib().gref_set_420(0, 0)
        lib().gref_set_clear_metadata(1)
    data = C.string_at(out, out_len.value)
    lib().gref_free(out)
    t = ""
    if trace:
        t = C.string_at(tr, tr_len.value).decode()
        lib().gref_free(tr)
    return bool(ok), data, t, list(counters), secs.value


def process_jpeg(jpeg_in, quality=95.0, clear_metadata=True, trace=True):
    """guetzli::Process(jpeg bytes) -> (ok, jpeg bytes, trace str, counters[3])"""
    buf = np.frombuffer(bytes(jpeg_in), dtype=np.uint8)
    out, out_len = C.POINTER(C.c_uint8)(), C.c_size_t()
    tr, tr_len = C.c_char_p(), C.c_size_t()
    counters = (C.c_int * 3)()
    ok = lib().gref_process_jpeg(_p(buf, C.c_uint8), C.c_size_t(buf.size), C.c_float(target_for_quality(quality)),
                                 int(clear_metadata), C.byref(out), C.byref(out_len),
                                 C.byref(tr) if trace else None, C.byref(tr_len), counters)
    data = C.string_at(out, out_len.value)
    lib().gref_free(out)
    t = ""
    if trace:
        t = C.string_at(tr, tr_len.value).decode()
        lib().gref_free(tr)
    return bool(ok), data, t, list(counters)


def read_jpeg(jpeg_in):
    """ReadJpeg(JPEG_READ_ALL) -> (ok, dims, quantised coefficients of all components, concatenated)"""
    buf = np.frombuffer(bytes(jpeg_in), dtype=np.uint8)
    dims = (C.c_int * 11)()
    cap = 1 << 24
    out = np.zeros(cap, dtype=np.int16)
    ok = lib().gref_read_jpeg(_p(buf, C.c_uint8), C.c_size_t(buf.size), dims, _p(out, C.c_int16), C.c_size_t(cap))
    d = list(dims)
    n = sum(d[3 + 2 * c] * d[4 + 2 * c] * 64 for c in range(d[2])) if ok else 0
    return bool(ok), d, out[:n].copy()


def butteraugli_interface(rgb0, rgb1):
    """butteraugli::ButteraugliInterface on planar linear float32 [3][h][w] -> (diffmap, score)"""
    a = np.ascontiguousarray(rgb0, dtype=np.float32)
    b = np.ascontiguousarray(rgb1, dtype=np.float32)
    _, h, w = a.shape
    dm = np.zeros((h, w), dtype=np.float32)
    score = C.c_double()
    assert lib().gref_butteraugli_interface(_p(a, C.c_float), _p(b, C.c_float), w, h, _p(dm, C.c_float), C.byref(score))
    return dm, score.value


def nblocks(w, h):
    return ((w + 7) // 8) * ((h + 7) // 8)


def rgb_to_coeffs(rgb):
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = rgb.shape
    out = np.zeros((3, nblocks(w, h), 64), dtype=np.int16)
    assert lib().gref_rgb_to_coeffs(_p(rgb, C.c_uint8), w, h, _p(out, C.c_int16))
    return out


def idct_block(block):
    block = np.ascontiguousarray(block, dtype=np.int16)
    out = np.zeros(64, dtype=np.uint8)
    lib().gref_idct_block(_p(block, C.c_int16), _p(out, C.c_uint8))
    return out


def fdct_block(block):
    block = np.array(block, dtype=np.int16).copy()
    lib().gref_fdct_block(_p(block, C.c_int16))
    return block


def render(coeffs, w, h):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int16)
    srgb = np.zeros((h, w, 3), dtype=np.uint8)
    lin = np.zeros((3, h, w), dtype=np.float32)
    lib().gref_render(_p(coeffs, C.c_int16), w, h, _p(srgb, C.c_uint8), _p(lin, C.c_float))
    return srgb, lin


def apply_global_quant(coeffs, w, h, q):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int16)
    q = np.ascontiguousarray(q, dtype=np.int32)
    out = np.zeros_like(coeffs)
    lib().gref_apply_global_quant(_p(coeffs, C.c_int16), w, h, _p(q, C.c_int32), _p(out, C.c_int16))
    return out


def blur(img, sigma, border_ratio):
    img = np.ascontiguousarray(img, dtype=np.float32)
    h, w = img.shape
    out = np.zeros_like(img)
    lib().gref_blur(_p(img, C.c_float), w, h, C.c_float(sigma), C.c_float(border_ratio), _p(out, C.c_float))
    return out


def opsin(rgb_planes):
    a = np.ascontiguousarray(rgb_planes, dtype=np.float32)
    _, h, w = a.shape
    out = np.zeros_like(a)
    lib().gref_opsin(_p(a, C.c_float), w, h, _p(out, C.c_float))
    return out


def separate(xyb):
    a = np.ascontiguousarray(xyb, dtype=np.float32)
    _, h, w = a.shape
    out = np.zeros((10, h, w), dtype=np.float32)
    lib().gref_separate(_p(a, C.c_float), w, h, _p(out, C.c_float))
    return out


def malta(lum0, lum1, w_0gt1, w_0lt1, norm1, lf, acc=None):
    a = np.ascontiguousarray(lum0, dtype=np.float32)
    b = np.ascontiguousarray(lum1, dtype=np.float32)
    h, w = a.shape
    out = np.zeros_like(a) if acc is None else np.array(acc, dtype=np.float32).copy()
    lib().gref_malta(_p(a, C.c_float), _p(b, C.c_float), w, h, C.c_double(w_0gt1),
                     C.c_double(w_0lt1), C.c_double(norm1), int(lf), _p(out, C.c_float))
    return out


def mask(xyb0, xyb1):
    a = np.ascontiguousarray(xyb0, dtype=np.float32)
    b = np.ascontiguousarray(xyb1, dtype=np.float32)
    _, h, w = a.shape
    m = np.zeros_like(a)
    mdc = np.zeros_like(a)
    lib().gref_mask(_p(a, C.c_float), _p(b, C.c_float), w, h, _p(m, C.c_float), _p(mdc, C.c_float))
    return m, mdc


def diffmap(rgb0_lin, rgb1_lin):
    a = np.ascontiguousarray(rgb0_lin, dtype=np.float32)
    b = np.ascontiguousarray(rgb1_lin, dtype=np.float32)
    _, h, w = a.shape
    out = np.zeros((h, w), dtype=np.float32)
    lib().gref_diffmap(_p(a, C.c_float), _p(b, C.c_float), w, h, _p(out, C.c_float))
    return out


def compare_coeffs(rgb, coeffs, target):
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = rgb.shape
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int16)
    dm = np.zeros((h, w), dtype=np.float32)
    dist = C.c_float()
    lib().gref_compare_coeffs(_p(rgb, C.c_uint8), w, h, C.c_float(target),
                              _p(coeffs, C.c_int16), _p(dm, C.c_float), C.byref(dist))
    return dm, dist.value


def block_mask(rgb):
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = rgb.shape
    out = np.zeros((3, h, w), dtype=np.float32)
    lib().gref_block_mask(_p(rgb, C.c_uint8), w, h, _p(out, C.c_float))
    return out


def block_corner_mask(rgb):
    """block_mask at the top-left pixel of every 8x8 block -> [nblocks][3]"""
    m = block_mask(rgb)
    return np.stack([m[c][::8, ::8].reshape(-1) for c in range(3)], axis=1)


def heatmap(distmap):
    """butteraugli_main's CreateHeatMapImage of a [h][w] diffmap -> [h][w][3] uint8"""
    d = np.ascontiguousarray(distmap, dtype=np.float32)
    h, w = d.shape
    out = np.zeros((h, w, 3), dtype=np.uint8)
    lib().gref_heatmap(_p(d, C.c_float), w, h, _p(out, C.c_uint8))
    return out


def huffman_depths(counts, limits):
    """CreateHuffmanTree's code lengths for every row of counts [t][n] with the length limit limits[t]"""
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    t, n = counts.shape
    out = np.zeros((t, n), dtype=np.uint8)
    for i in range(t):
        lib().gref_huffman_depths(_p(counts[i], C.c_uint32), n, int(limits[i]), _p(out[i], C.c_uint8))
    return out


def zeroing_orders(rgb, orig_coeffs, q, target):
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, _ = rgb.shape
    nb = nblocks(w, h)
    coeffs = np.ascontiguousarray(orig_coeffs, dtype=np.int16)
    q = np.ascontiguousarray(q, dtype=np.int32)
    offs = np.zeros(nb + 1, dtype=np.int32)
    idx = np.zeros(189 * nb, dtype=np.uint8)
    err = np.zeros(189 * nb, dtype=np.float32)
    n = lib().gref_zeroing_orders(_p(rgb, C.c_uint8), w, h, C.c_float(target),
                                  _p(coeffs, C.c_int16), _p(q, C.c_int32),
                                  _p(offs, C.c_int32), _p(idx, C.c_uint8), _p(err, C.c_float))
    return offs, idx[:n].copy(), err[:n].copy()


def block_weights(w, h, target, direction, rblock, target_mul, distmap):
    d = np.ascontiguousarray(distmap, dtype=np.float32)
    out = np.zeros(nblocks(w, h), dtype=np.float32)
    lib().gref_block_weights(w, h, C.c_float(target), direction, rblock,
                             C.c_double(target_mul), _p(d, C.c_float), _p(out, C.c_float))
    return out


def write_jpeg(coeffs, w, h, q):
    coeffs = np.ascontiguousarray(coeffs, dtype=np.int16)
    q = np.ascontiguousarray(q, dtype=np.int32)
    out = C.POINTER(C.c_uint8)()
    out_len = C.c_size_t()
    assert lib().gref_write_jpeg(_p(coeffs, C.c_int16), w, h, _p(q, C.c_int32),
                                 C.byref(out), C.byref(out_len))
    data = C.string_at(out, out_len.value)
    lib().gref_free(out)
    return data


def blur_kernel(sigma):
    out = np.zeros(256, dtype=np.float32)
    n = C.c_int()
    lib().gref_blur_kernel(C.c_float(sigma), _p(out, C.c_float), C.byref(n))
    return out[:n.value].copy()


def srgb_lut():
    out = np.zeros(256, dtype=np.float64)
    lib().gref_srgb_lut(_p(out, C.c_double))
    return out


def color_tables():
    t = [np.zeros(256, dtype=np.int32) for _ in range(4)]
    rl = np.zeros(1024, dtype=np.uint8)
    lib().gref_color_tables(*[_p(x, C.c_int32) for x in t], _p(rl, C.c_uint8))
    return t[0], t[1], t[2], t[3], rl
