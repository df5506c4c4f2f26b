"""What the training-convolution tests share (conv_transpose2d, conv1x1, conv3x3): the per-element gate against fp64,
the fp64 emulation of the scaled fp16 planes, the Python mirror of the library's wgrad slice rule, guarded buffers for
the memory contract of the C ABI, and running a step on a side stream or replaying it from a CUDA graph."""
import pytest
import torch

GATE_MAX = 2e-5          # max error / max |reference| (test_gpu_deconv_train.py)
# Per element: |got - ref| <= GATE_C * m + 2^-126, m = the same sum over |operands| (sum |x||w| (+ |b|) for y, |dy||w|
# for dx, |x||dy| for dW, |dy| for db).  Measured on an NVIDIA B200 (1000 W power limit) over every case of
# test_gpu_deconv_train_domain.py: worst (|err| - 2^-126) / m = 3.5e-7 for y, 2.2e-7 for dx, 3.3e-7 for dW, so
# 2^-18 = 3.8e-6 leaves a 10.9x margin.  Losing the lo plane of an fp16 hi/lo operand costs ~2^-12 (the host tests show
# that this gate catches it).
GATE_C = 2.0 ** -18
TINY = 2.0 ** -126       # the fp32 subnormal range: nothing below the smallest normal is resolved by an fp32 output


def gate(name, got, ref, mag, max_gate=True, nonfinite=None, worst=None):
    """Assert the per-element gate on every element finite in ref, and that every non-finite element of ref is
    non-finite in got.  `nonfinite` (optional): where got may be non-finite although ref is not.  Returns
    max (|err| - 2^-126) / m and max |err| / max |ref| over the gated elements, and keeps the largest of the first in
    worst[name] (worst: a module's dict, see report_worst)."""
    got = got.detach().double()
    assert got.shape == ref.shape, name
    fin = torch.isfinite(ref)
    assert not bool(torch.isfinite(got[~fin]).any()), f"{name}: finite where the reference is not"
    if nonfinite is not None:
        fin = fin & ~nonfinite
    got, ref, mag = got[fin], ref[fin], mag[fin]
    err = (got - ref).abs()
    ok = err <= GATE_C * mag + TINY                        # NaN fails
    if not bool(ok.all()):
        i = int((~ok).nonzero()[0])
        raise AssertionError(f"{name}: {int((~ok).sum())} of {ok.numel()} elements outside the per-element gate, "
                             f"first: got {float(got[i])!r} ref {float(ref[i])!r} m {float(mag[i])!r}")
    ratio = float(((err - TINY).clamp_min(0) / mag.clamp_min(1e-300)).max()) if err.numel() else 0.0
    if worst is not None:
        worst[name] = max(worst[name], ratio)
    rel = float(err.max() / ref.abs().max().clamp_min(1e-300)) if err.numel() else 0.0
    if max_gate:
        assert rel <= GATE_MAX, (name, rel)
    return ratio, rel


def report_worst(worst, module):
    """An autouse fixture for `module` that prints, after its tests, the largest error / m its gate saw per pass."""
    @pytest.fixture(scope="module", autouse=True)
    def _report_worst():
        yield
        print(f"\nworst per-element error / m over {module}: " + ", ".join(f"{k} {v:.3e}" for k, v in worst.items()))
    return _report_worst


def wgrad_slices(k_pixels, m, n, taps):
    """Python mirror of the library's wgrad slice rule (csrc/gemm_tc.cu: wgrad_slices as make_train_conv calls it): the
    number of K slices of a weight gradient over k_pixels pixels with M = m, N = n and `taps` taps."""
    kb = k_pixels // 64
    tiles = -(-m // 128) * -(-n // 128) * taps
    s = 1
    while tiles * s < 2 * 148 and kb % (2 * s) == 0 and kb // (2 * s) >= 16:
        s *= 2
    return s


def f16_planes(t, keep_lo):
    """fp64 emulation of the scaled fp16 planes of a tensor (layout.cu: nchw_to_rows_f16p): s = 2^min(13 - ilogb(amax),
    127), hi = rn_f16(x s), lo = rn_f16((x s - hi) 2^11); decoded as (hi + lo 2^-11) / s, or hi / s alone."""
    _, e = torch.frexp(t.abs().max())
    s = 2.0 ** min(13 - (int(e) - 1), 127)
    X = t * s
    hi = X.half().double()
    if not keep_lo:
        return hi / s
    return (hi + ((X - hi) * 2048).half().double() / 2048) / s


# ---- memory contract of the C ABI: exact byte counts, guard bytes around every buffer, stale workspace contents ----
GUARD = 4096             # bytes before and after every buffer; a multiple of 256 keeps the interior 256-byte aligned
SENTINEL = 0x5A


class Region:
    """`nbytes` inside a larger uint8 buffer: GUARD sentinel bytes on each side, the interior filled with `fill`
    (a byte value, "random", or None for the sentinel)."""

    def __init__(self, nbytes, fill=None, gen=None):
        self.nbytes = nbytes
        self.buf = torch.full((GUARD + nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        if fill == "random":
            self.inner.copy_(torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda", generator=gen))
        elif fill is not None:
            self.inner.fill_(fill)
        assert self.buf.data_ptr() % 256 == 0

    @property
    def inner(self):
        return self.buf[GUARD:GUARD + self.nbytes]

    def f32(self, shape):
        return self.inner.view(torch.float32).view(shape)

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENTINEL).all()) and bool((self.buf[GUARD + self.nbytes:] == SENTINEL).all())


def f32_region(shape):
    n = 1
    for d in shape:
        n *= d
    r = Region(4 * n)
    return r, r.f32(shape)


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


# ---- streams, CUDA graphs ----
def on_side_stream(fn, *args):
    """fn(*args) on a new stream that first waits for the current one, which then waits for it."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out = fn(*args)
    torch.cuda.current_stream().wait_stream(s)
    return out


def graph_replay(step, statics, new_values):
    """Run step() once on a side stream (warm-up outside the capture), capture it in a CUDA graph, copy new_values into
    the static tensors it reads and replay the graph -> the outputs step() returned inside the capture."""
    on_side_stream(step)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step()
    with torch.no_grad():
        for t, v in zip(statics, new_values):
            t.copy_(v)
    g.replay()
    torch.cuda.synchronize()
    return out
