"""The weight fingerprint of the render session (`spb_session_begin`, csrc/decode_stack.cu) stated in numpy, and the table the
kernel reads.  tests/test_render_session_gpu.py compares the kernel against `fingerprint`."""
import numpy as np
import torch

M64 = (1 << 64) - 1


def fingerprint(arrays) -> int:
    """sum over the 32-bit words w_i of all arrays (in order, i counted across them) of splitmix64((i << 32) | w_i), mod 2^64."""
    words = np.concatenate([np.ascontiguousarray(a).reshape(-1).view(np.uint32) for a in arrays]) if len(arrays) else np.zeros(0, np.uint32)
    i = np.arange(words.size, dtype=np.uint64)
    z = ((i << np.uint64(32)) | words.astype(np.uint64)) + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    z = z ^ (z >> np.uint64(31))
    return int(z.sum(dtype=np.uint64))


def _splitmix64(x: int) -> int:
    z = (x + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def test_fingerprint_statement_equals_python_integers():
    # numpy's uint64 arithmetic wraps exactly like the unbounded integers reduced mod 2^64
    rng = np.random.default_rng(3)
    arrays = [rng.standard_normal(n).astype(np.float32) for n in (1, 7, 256, 1000)]
    words = np.concatenate([a.view(np.uint32) for a in arrays]).tolist()
    want = sum(_splitmix64((i << 32) | w) for i, w in enumerate(words)) & M64
    assert fingerprint(arrays) == want
    assert sum(_splitmix64((i << 32) | w) for i, w in enumerate(words)) > M64      # the sum does wrap around
    assert fingerprint([]) == 0


def test_fingerprint_sees_bit_patterns_and_positions():
    rng = np.random.default_rng(4)
    a = rng.standard_normal(4096).astype(np.float32)
    base = fingerprint([a])
    # bit patterns, not values: -0.0 and 0.0, two NaN payloads, one ulp
    z = a.copy(); z[5] = 0.0
    n = z.copy(); n[5] = -0.0
    assert fingerprint([z]) != fingerprint([n])
    q1 = a.copy(); q1[9] = np.frombuffer(np.uint32(0x7FC00000).tobytes(), np.float32)[0]
    q2 = a.copy(); q2[9] = np.frombuffer(np.uint32(0x7FC00001).tobytes(), np.float32)[0]
    assert fingerprint([q1]) != fingerprint([q2])
    u = a.copy(); u[100] = np.nextafter(u[100], np.float32(np.inf))
    assert fingerprint([u]) != base
    # positions: two values trading places, and the same words split over tensors differently (index counted across the table)
    s = a.copy(); s[[10, 20]] = s[[20, 10]]
    assert fingerprint([s]) != base
    assert fingerprint([a[:1000], a[1000:1003], a[1003:]]) == base
    assert fingerprint([a[1000:], a[:1000]]) != base


def test_fingerprint_table_layout():
    from scoreperformer_b200 import kernels as K
    ts = [torch.zeros(3, 5), torch.zeros(7, dtype=torch.float64), torch.zeros(2, 2, dtype=torch.bfloat16)]
    table = K.fingerprint_table(ts)
    assert table.dtype == torch.int64 and table.shape == (3, 3)
    assert table[:, 0].tolist() == [t.data_ptr() for t in ts]
    assert table[:, 1].tolist() == [15, 14, 2] and table[:, 2].tolist() == [0, 15, 29]
    for bad in (torch.zeros(4, 4).t(), torch.zeros(3, dtype=torch.bfloat16), torch.zeros(8, dtype=torch.uint8)[1:5]):
        try:
            K.fingerprint_table([bad])
        except ValueError:
            continue
        raise AssertionError(f"accepted {bad.dtype} {tuple(bad.shape)} stride {bad.stride()}")
