"""numpy statement of the packed-code format of include/mhaq_fq.h ("Packed codes"), used by the
CPU format tests and as the reference the GPU packer is compared with."""
import numpy as np

WIDTHS = (1, 2, 4, 8, 16)


def row_bytes(n_inner: int, bits: int) -> int:
    """round_up(ceil(n_inner * bits / 8), 16)."""
    return ((n_inner * bits + 7) // 8 + 15) // 16 * 16


def saturate(codes: np.ndarray, bits: int):
    """(uint codes clamped to [0, 2^bits - 1] with NaN -> 0, number of codes that needed it)."""
    c = np.asarray(codes, dtype=np.float64)
    top = (1 << bits) - 1
    bad = ~((c >= 0) & (c <= top))
    return np.clip(np.nan_to_num(c, nan=0.0), 0, top).astype(np.uint32), int(bad.sum())


def pack(codes: np.ndarray, bits: int) -> np.ndarray:
    """uint codes [n_rows, n_inner] (each < 2^bits) -> uint8 [n_rows, row_bytes]."""
    codes = np.asarray(codes, dtype=np.uint32)
    n_rows, n_inner = codes.shape
    out = np.zeros((n_rows, row_bytes(n_inner, bits)), np.uint8)
    if bits == 16:
        out[:, :2 * n_inner] = codes.astype("<u2").view(np.uint8).reshape(n_rows, 2 * n_inner)
    else:
        # code j -> bits [j*b, (j+1)*b) of the row, least-significant bit first
        bitplane = ((codes[..., None] >> np.arange(bits, dtype=np.uint32)) & 1).astype(np.uint8)
        packed = np.packbits(bitplane.reshape(n_rows, n_inner * bits), axis=1, bitorder="little")
        out[:, :packed.shape[1]] = packed
    return out


def unpack(data: np.ndarray, bits: int, n_inner: int) -> np.ndarray:
    """uint8 [n_rows, row_bytes] -> uint codes [n_rows, n_inner]."""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    n_rows = data.shape[0]
    if bits == 16:
        return data[:, :2 * n_inner].copy().view("<u2").astype(np.uint32)
    b = np.unpackbits(data, axis=1, bitorder="little")[:, :n_inner * bits].reshape(n_rows, n_inner, bits)
    return (b.astype(np.uint32) << np.arange(bits, dtype=np.uint32)).sum(-1).astype(np.uint32)
