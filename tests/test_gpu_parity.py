"""GPU (`-m gpu`): the parity tests proper.  The hand-written sm_100a kernels, called through the
C ABI (include/b200fft.h) via the FftPlanner / Fft mirror, against the CPU oracle on the same seeded
inputs -- the reference's acceptance test (tests/accuracy.rs:124-187: every len 1..1000, forward and
inverse, f32 and f64, three process variants, vs the Bluestein-over-Radix4 control) plus the
BASELINE.json configs, with the reference's criterion (mean |a-b| < 0.1) AND the strict tolerance
stated in tests/util.py::strict_bound (relative L2 <= 4 eps log2 N vs an f64 truth, and never worse
than 2x the oracle's own error).  Full-size configs are checked through size-independent properties
(round trip, Parseval, linearity) with spot transforms compared to the oracle."""
import threading

import numpy as np
import pytest

import oracle
import rustfft_b200 as rb
import plan_kinds
from protocol import check_error_behaviour, check_fft_algorithm, check_planner_cache
from util import EPS, rel_l2, signal, strict_bound, truth

pytestmark = pytest.mark.gpu
DIRS = [rb.FftDirection.Forward, rb.FftDirection.Inverse]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    assert torch.cuda.is_available(), "-m gpu tests need a B200"
    return torch


@pytest.fixture(scope="module", params=[np.complex64, np.complex128], ids=["f32", "f64"])
def planner(request, torch_cuda):
    # default library = rustfft_b200/libb200fft.so; raises if it is missing (no fallback)
    return rb.FftPlanner(request.param, device=0), request.param


def test_native_library_is_the_one_running(torch_cuda):
    import os
    import subprocess
    import sys

    from util import ROOT

    lib = rb.default_library()
    assert lib.path.endswith("rustfft_b200/libb200fft.so") and lib.device_count() >= 1
    # the mapping check runs in a process of its own: the CPU tests of the same session load the emulation library into this one
    code = ("import rustfft_b200 as rb\n"
            "lib = rb.default_library()\n"
            "assert lib.path.endswith('rustfft_b200/libb200fft.so') and lib.device_count() >= 1\n"
            "maps = open('/proc/self/maps').read()\n"
            "assert 'libb200fft.so' in maps and 'libb200fft_emu' not in maps\n"
            "print('NATIVE-OK')\n")
    e = dict(os.environ)
    e["PYTHONPATH"] = ROOT + os.pathsep + os.path.join(ROOT, "tests")
    r = subprocess.run([sys.executable, "-c", code], env=e, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "NATIVE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_accuracy_every_len_1_to_1000(planner):
    """tests/accuracy.rs:124-187."""
    pl, dtype = planner
    for n in range(1, 1001):
        for d in DIRS:
            check_fft_algorithm(pl, n, d, dtype)


@pytest.mark.parametrize("lg", list(range(10, 21)))
def test_config2_power_of_two_sweep_vs_oracle(torch_cuda, lg):
    """BASELINE config 2 (f32 forward 2^10..2^20): a few transforms against the scalar-planner oracle
    (Radix4, src/algorithm/radix4.rs) and the f64 truth."""
    pl = rb.FftPlanner(np.complex64)
    n = 1 << lg
    check_fft_algorithm(pl, n, DIRS[0], np.complex64, control_kind=oracle.PLANNER, chunks=3 if lg < 18 else 1)
    check_fft_algorithm(pl, n, DIRS[1], np.complex64, control_kind=oracle.PLANNER, chunks=1)


@pytest.mark.parametrize("lg", [10, 13, 16, 18, 20])
def test_config2_full_batch_properties(torch_cuda, lg):
    """batch = 4096 on the device path: inverse(forward(x))/N == x, Parseval, linearity in the batch,
    and first / last / middle transforms against the oracle."""
    torch = torch_cuda
    n, batch = 1 << lg, 4096
    pl = rb.FftPlanner(np.complex64)
    f, fi = pl.plan_fft_forward(n), pl.plan_fft_inverse(n)
    g = torch.Generator(device="cuda").manual_seed(lg)
    x = torch.rand(batch * n, 2, device="cuda", generator=g) * 10
    x = torch.view_as_complex(x).contiguous()
    y = torch.empty_like(x)
    f.process_device(x, out=y)
    ex = torch.sum(x.real.double() ** 2 + x.imag.double() ** 2)
    ey = torch.sum(y.real.double() ** 2 + y.imag.double() ** 2) / n
    assert abs((ey / ex).item() - 1) < 1e-5  # Parseval
    for b in (0, batch // 2 + 1, batch - 1):
        xb = x[b * n:(b + 1) * n].cpu().numpy()
        yb = y[b * n:(b + 1) * n].cpu().numpy()
        assert rel_l2(yb, truth(xb, n, False)) <= strict_bound(n, np.complex64)
        assert rel_l2(yb, oracle.fft(xb, n)) <= 2 * strict_bound(n, np.complex64)
    fi.process_device(y)  # in place
    y /= n
    num = torch.sqrt(torch.sum((y.real - x.real).double() ** 2 + (y.imag - x.imag).double() ** 2))
    assert (num / torch.sqrt(ex)).item() <= 2 * strict_bound(n, np.complex64)
    del y
    torch.cuda.empty_cache()


def test_config3_f64_1234_roundtrip_batch_1024(torch_cuda):
    """BASELINE config 3: f64 forward + inverse round trip, N = 1234, batch = 1024."""
    n, batch = 1234, 1024
    pl = rb.FftPlanner(np.complex128)
    f, fi = pl.plan_fft_forward(n), pl.plan_fft_inverse(n)
    x = signal(n * batch, np.complex128, seed=3)
    y = x.copy()
    f.process(y)
    for b in (0, 511, 1023):
        got, xb = y[b * n:(b + 1) * n], x[b * n:(b + 1) * n]
        want = oracle.fft(xb, n)  # RadixN{[2], Raders(617)} in the scalar planner
        assert rel_l2(got, truth(xb, n, False)) <= strict_bound(n, np.complex128)
        assert np.all(np.isfinite(want.view(np.float64)))
    fi.process(y)
    assert rel_l2(y / n, x) <= 2 * strict_bound(n, np.complex128)


def test_config4_prime_65537_batch_512(torch_cuda):
    """BASELINE config 4: f32 prime N = 65537 (Rader in both reference planners), batch = 512."""
    n, batch = 65537, 512
    pl = rb.FftPlanner(np.complex64)
    f = pl.plan_fft_forward(n)
    assert f.describe().startswith("Rader{n=65537")
    x = signal(n * batch, np.complex64, seed=4)
    y = x.copy()
    f.process(y)
    for b in (0, 255, 511):
        xb = x[b * n:(b + 1) * n]
        ref = truth(xb, n, False)
        want = oracle.fft(xb, n)
        assert rel_l2(y[b * n:(b + 1) * n], ref) <= strict_bound(n, np.complex64)
        assert rel_l2(y[b * n:(b + 1) * n], want) <= 2 * strict_bound(n, np.complex64)


@pytest.mark.parametrize("lg", [21, 22, 23, 24])
def test_power_of_two_up_to_2_24(planner, lg):
    """Beyond the BASELINE sweep: 2048/4096-point tiles (the reference benches up to 4 194 304,
    benches/bench_compare_scalar_sse_avx.rs:123-124)."""
    pl, dtype = planner
    n = 1 << lg
    f = pl.plan_fft_forward(n)
    assert f.describe().startswith("FourStep{")
    x = signal(2 * n, dtype, seed=lg)
    y = x.copy()
    f.process(y)
    assert rel_l2(y, truth(x, n, False)) <= strict_bound(n, dtype)
    pl.plan_fft_inverse(n).process(y)
    assert rel_l2(y / n, x) <= 2 * strict_bound(n, dtype)


@pytest.mark.parametrize("n", [2049, 4099, 10007, 44100, 112501, 300000, 1000003])
def test_large_non_power_of_two(planner, n):
    """Bluestein over a four-step inner FFT (beyond the reference's accuracy test range, which stops at
    1000; 112501 is one of its 32-bit-overflow Rader primes, raders_algorithm.rs:311-322)."""
    pl, dtype = planner
    check_fft_algorithm(pl, n, DIRS[0], dtype, control_kind=oracle.PLANNER, chunks=2)
    check_fft_algorithm(pl, n, DIRS[1], dtype, control_kind=oracle.PLANNER, chunks=1)


@pytest.mark.parametrize("check", plan_kinds.ALL, ids=[c.__name__[6:] for c in plan_kinds.ALL])
def test_round2_plan_kinds(planner, check):
    """General Rader, MixedRadix{r0 x Rader}, Good-Thomas, Bluestein over smooth lengths, caller-owned recipes (tests/plan_kinds.py)."""
    pl, dtype = planner
    check(pl, dtype)


def test_compiled_tile_lengths_in_both_roles(torch_cuda):
    """Every compiled composite tile length (SmoothTileGeo) as the column pass and as the row pass of a two-pass plan, many transforms."""
    pl = rb.FftPlanner(np.complex64)
    ls = [64, 100, 125, 128, 196, 200, 225, 250, 256, 375, 400, 500, 512, 625, 1000, 1024]
    for a, b in zip(ls[:-1], ls[1:]):
        for d in DIRS:
            f = check_fft_algorithm(pl, a * b, d, np.complex64, control_kind=oracle.PLANNER, chunks=40 if a * b < 100000 else 3,
                                    recipe=rb.Recipe.mixed_radix(a, b))
            assert f.describe() == "SmoothFourStep{%dx%d,compiled}" % (a, b)


@pytest.mark.parametrize("n", [4225, 5000, 6000, 10000, 17017, 29791, 44100, 48000, 100000, 196608, 1000000])
def test_smooth_composites_two_pass(planner, n):
    """Composite lengths above the one-pass limit, prime factors <= 31: SmoothFourStep (two passes, run-time radix
    lists) -- the reference plans them as MixedRadix / GoodThomas trees (src/plan.rs:508-607)."""
    pl, dtype = planner
    chunks = 60 if n <= 50000 else 3
    f = check_fft_algorithm(pl, n, DIRS[0], dtype, control_kind=oracle.PLANNER, chunks=chunks)
    assert f.describe().startswith("SmoothFourStep{")
    check_fft_algorithm(pl, n, DIRS[1], dtype, control_kind=oracle.PLANNER, chunks=2)


@pytest.mark.parametrize("n", [360, 1000, 1200, 1536, 2000, 2401, 3600, 4000, 143, 961, 1196, 1131, 3683])
def test_smooth_lengths_native(planner, n):
    """Prime factors <= 31: one-pass run-time-radix kernel (the reference: RadixN / MixedRadix / butterflies
    2..32, plan.rs:508-634).  3683 = 29 * 127 has a larger factor and goes through Bluestein."""
    pl, dtype = planner
    f = check_fft_algorithm(pl, n, DIRS[0], dtype, control_kind=oracle.PLANNER, chunks=300)
    if n != 3683 and (n <= 2048 or dtype == np.complex64):
        assert f.describe().startswith("Smooth{")
    check_fft_algorithm(pl, n, DIRS[1], dtype, control_kind=oracle.PLANNER, chunks=3)


def test_device_path_equals_host_path_and_workspace_variants(torch_cuda):
    torch = torch_cuda
    pl = rb.FftPlanner(np.complex64)
    for n, batch in [(1024, 33), (1 << 14, 5), (1 << 15, 300), (1 << 16, 5), (257, 9), (1000, 17), (997, 17), (65537, 80), (5000, 3)]:
        f = pl.plan_fft_forward(n)
        x = signal(n * batch, np.complex64, seed=n)
        host = x.copy()
        f.process(host)
        d = torch.from_numpy(x).cuda()
        out = torch.full_like(d, float("nan"))
        f.process_device(d, out=out)
        assert np.array_equal(out.cpu().numpy(), host), n
        assert np.array_equal(d.cpu().numpy(), x), "out-of-place must leave the input intact"
        f.process_device(d)  # in place
        assert np.array_equal(d.cpu().numpy(), host), n
        nbytes = f.workspace_bytes(batch)
        if nbytes:
            ws = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")  # dirty workspace
            d2 = torch.from_numpy(x).cuda()
            f.process_device(d2, workspace=ws)
            assert np.array_equal(d2.cpu().numpy(), host), n
            with pytest.raises(rb.FftError, match="workspace too small"):
                f.process_device(d2, workspace=ws[: nbytes // 2])


@pytest.mark.parametrize("env", [
    {"B200FFT_PIPELINE": "1"},                      # persistent TMA (cp.async.bulk + mbarrier) kernels
    {"B200FFT_RADIX32": "0"},                       # radix <= 16 geometries
    {"B200FFT_FUSED": "0"},                         # two-pass plans as chunked launch pairs (TMA tiles) instead of the fused kernel
    {"B200FFT_FUSED": "0", "B200FFT_OVERLAP": "0"},  # ... chunks on one stream
    {"B200FFT_FUSED": "0", "B200FFT_STREAMS": "4", "B200FFT_CHUNK_MB": "8"},  # ... many small chunks over four streams
    {"B200FFT_HOST_PIPE": "2"},                     # two-stream host-slice path
    {"B200FFT_FUSED": "0", "B200FFT_TMA_TILES": "0"},  # two-pass tiles through LDG/STG instead of TMA tensor copies
    {"B200FFT_FUSED_W": "2"},                       # fused kernel with the smallest ring (every tile waits)
    {"B200FFT_FUSED_LOOKAHEAD": "40"},              # ... with a short look-ahead
    {"B200FFT_FUSED_LOOKAHEAD": "5000"},            # ... and a deep one
    {"B200FFT_FUSED_TILED": "1"},                   # ... with the tile-major ring (pass A stores from its registers)
    {"B200FFT_FUSED_BDIRECT": "63"},                # ... with pass B storing its results from the registers (no TMA store)
    {"B200FFT_FLOW": "1"},                          # two-pass plans as one launch of the (round-1) dataflow kernel
    {"B200FFT_FLOW": "1", "B200FFT_FLOW_W": "2"},   # ... with the smallest ring (every tile waits)
], ids=["tma-pipelined", "radix16", "chunked", "chunked-one-stream", "chunked-four-streams-small-chunks", "host-two-stream", "chunked-ldg-tiles",
        "fused-ring2", "fused-short-lookahead", "fused-deep-lookahead", "fused-tile-major-ring", "fused-direct-pass-b-output", "flow", "flow-ring2"])
def test_alternative_code_paths_in_a_fresh_process(torch_cuda, env):
    import os
    import subprocess
    import sys

    from util import ROOT

    e = dict(os.environ)
    e.update(env)
    e["PYTHONPATH"] = ROOT + os.pathsep + os.path.join(ROOT, "tests")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "variant_check.py")], env=e, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "VARIANT-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_sharded_scatter_fft_gather_two_gpus(torch_cuda):
    """BASELINE config 5's data path on hardware: NCCL scatter of batch shards -> FFT per GPU -> gather, two ranks under torchrun
    (skipped on a one-GPU box; tests/test_sharding_gloo.py covers the host logic on the CPU)."""
    import os
    import subprocess
    import sys

    from util import ROOT

    if torch_cuda.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    e = dict(os.environ)
    e["PYTHONPATH"] = ROOT + os.pathsep + os.path.join(ROOT, "tests")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29731", os.path.join(ROOT, "tests", "sharded_gpu_check.py")], env=e, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "SHARDED-OK world=2" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


@pytest.mark.parametrize("rdtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_real_fft_wrappers(torch_cuda, rdtype):
    """r2c / c2r of even lengths on top of the complex plans: host entry points (tests/real_fft_cases.py) and the device ones."""
    import real_fft_cases

    torch = torch_cuda
    pl = rb.RealFftPlanner(rdtype)
    real_fft_cases.check_real_fft(pl, rdtype)
    n, batch = 4096, 300
    f = pl.plan_fft(n)
    x = (np.random.default_rng(1).random(n * batch) * 10).astype(rdtype)
    X = np.zeros(batch * (n // 2 + 1), np.complex64 if rdtype == np.float32 else np.complex128)
    f.forward(x, X)
    dx = torch.from_numpy(x).cuda()
    dX = torch.empty(batch * (n // 2 + 1), dtype=torch.complex64 if rdtype == np.float32 else torch.complex128, device="cuda")
    f.forward(dx, dX)
    assert np.array_equal(dX.cpu().numpy(), X)
    back = torch.empty_like(dx)
    f.inverse(dX, back)
    assert rel_l2(back.cpu().numpy() / n, x) <= 2 * strict_bound(n, X.dtype)


def test_fft_2d(planner, torch_cuda):
    """2-D plans (tests/fft2d_cases.py): host entry point against numpy fft2, device entry point equal to it bit for bit."""
    import fft2d_cases

    torch = torch_cuda
    pl, dtype = planner
    fft2d_cases.check_fft2d(pl, dtype)
    h, w, batch = 270, 480, 5
    f = pl.plan_fft_2d(h, w)
    x = signal(batch * h * w, dtype, seed=2)
    y = x.copy()
    f.process(y)
    d = torch.from_numpy(x).cuda()
    out = torch.empty_like(d)
    f.process_device(d, out=out)
    assert np.array_equal(out.cpu().numpy(), y)


def test_host_pipeline_many_chunks(torch_cuda):
    """Host-slice path with more 64 MiB staging chunks than ring slots (4): 6.x chunks, pageable and pinned."""
    torch = torch_cuda
    pl = rb.FftPlanner(np.complex64)
    n, batch = 4096, 6 * 2048 + 77
    f = pl.plan_fft_forward(n)
    x = signal(n * batch, np.complex64, seed=12)
    a = x.copy()
    f.process(a)  # pageable
    pin_in = torch.from_numpy(x).pin_memory()
    pin_out = torch.empty_like(pin_in).pin_memory()
    f.process_outofplace_with_scratch(pin_in.numpy(), pin_out.numpy())
    assert np.array_equal(a, pin_out.numpy())
    for t in (0, 2047, 2048, 8191, batch - 1):
        assert rel_l2(a[t * n:(t + 1) * n], truth(x[t * n:(t + 1) * n], n, False)) <= strict_bound(n, np.complex64)


def test_error_behaviour_and_cache(planner):
    pl, dtype = planner
    check_error_behaviour(pl, dtype)
    check_planner_cache(pl)


def test_shared_plan_from_many_threads(torch_cuda):
    """examples/concurrency.rs:17-29: one Arc<dyn Fft> used by several threads at once."""
    torch = torch_cuda
    pl = rb.FftPlanner(np.complex64)
    f = pl.plan_fft_forward(1 << 15)  # FourStep: needs a per-call workspace
    n = 1 << 15
    xs = [signal(n * 8, np.complex64, seed=t) for t in range(6)]
    outs = [None] * 6

    def work(t):
        with torch.cuda.stream(torch.cuda.Stream()):
            d = torch.from_numpy(xs[t]).cuda()
            for _ in range(5):
                o = torch.empty_like(d)
                f.process_device(d, out=o)
            torch.cuda.current_stream().synchronize()
            outs[t] = o.cpu().numpy()

    ths = [threading.Thread(target=work, args=(t,)) for t in range(6)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    for t in range(6):
        want = xs[t].copy()
        f.process(want)
        assert np.array_equal(outs[t], want), t


def test_ragged_batches_and_tails(torch_cuda):
    """batch sizes that do not fill the last CTA (F transforms per CTA) or the last L2 chunk."""
    pl = rb.FftPlanner(np.complex64)
    for n, batches in [(8, [1, 127, 129]), (64, [1, 15, 17]), (256, [1, 7, 9]), (1 << 13, [1, 3]), (1 << 15, [1, 3]),
                       (100, [1, 15, 17])]:
        f = pl.plan_fft_forward(n)
        for b in batches:
            x = signal(n * b, np.complex64, seed=b)
            y = x.copy()
            f.process(y)
            assert rel_l2(y, truth(x, n, False)) <= strict_bound(n, np.complex64), (n, b)
