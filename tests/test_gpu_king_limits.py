"""The KING accumulator at the limits include/vcfx_cuda.h promises: counts in the upper half of uint32, cohorts larger than
C2, streams other than torch's current one, a second device, and sizes the library must refuse.

Expected counts come from float64 products of 0/1 planes (numpy, or torch on the GPU for the large cases), never from the
library; counts must be equal and kinship bit-equal, as in test_gpu_king.py, whose helpers these tests reuse.
test_emu_king_limits.py runs the refusals under the warp emulator.
"""
import time

import numpy as np
import pytest

import test_gpu_king as K

pytestmark = pytest.mark.gpu

E_INVALID, E_NOMEM = -1, -4
UINT32_MAX = 0xFFFFFFFF
MAX_SAMPLES = 128 << 14          # s_pad may not pass 2^21: the MMA kernel's tile word holds the tile row in 14 bits
SLEEP = 1 << 27                  # torch.cuda._sleep cycles: tens of milliseconds, far longer than a call into the library


# ----------------------------------------------------------------------------- helpers
def torch_planes_counts(x, n, want=None, step=8192):
    """CC, HH, AB, HC (float64 [n, n] CUDA tensors, added to `want`) of .bed codes x [rows, >= n] (a uint8 CUDA tensor),
    from float64 torch.matmul of the planes over row blocks: exact, every count is far below 2^53."""
    import torch
    if want is None:
        want = [torch.zeros((n, n), dtype=torch.float64, device=x.device) for _ in range(4)]
    for r0 in range(0, x.shape[0], step):
        b = x[r0:r0 + step, :n]
        a, h, bb = (b == 3).double(), (b == 2).double(), (b == 0).double()
        c = (b != 1).double()
        for w, (p, q) in zip(want, ((c, c), (h, h), (a, bb), (h, c))):
            w += p.T @ q
    return want


def torch_pack(v, gen):
    """.bed rows of .bed codes v [rows, n] (uint8 CUDA tensor); the padding bits of each row's last byte are random."""
    import torch
    rows, n = v.shape
    nb = (n + 3) // 4
    full = torch.randint(0, 4, (rows, 4 * nb), generator=gen, device=v.device, dtype=torch.uint8)
    full[:, :n] = v
    q = full.view(rows, nb, 4)
    return q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)


def counts_both(k):
    """counts() as device tensors (the int32 view and its mask) and as host arrays: both as int64 numpy, checked equal."""
    d = k.counts(device=True)
    h = k.counts(device=False)
    assert d.cc.is_cuda and not h.cc.is_cuda and d.rows == h.rows
    got = [t.cpu().numpy() for t in (d.cc, d.hh, d.ab, d.hc)]
    for name, g, t in zip(("CC", "HH", "AB", "HC"), got, (h.cc, h.hh, h.ab, h.hc)):
        assert np.array_equal(g, t.numpy()), f"{name}: counts(device=True) != counts(device=False)"
    return d, got


def packed_codes(rng, rows, n):
    """Seeded .bed codes [rows, n] with an all-missing sample, an all-homozygous sample and two duplicates, packed with
    garbage padding bits: (codes, rows)."""
    v = K.random_codes(rng, rows, n)
    v[:, 1] = 1
    v[:, 2] = np.where(rng.integers(0, 2, rows) == 1, 3, 0)
    v[:, n - 1] = v[:, 0]
    return v, K.pack_codes(v, rng)


# ----------------------------------------------------------------------------- A. the upper half of uint32
def test_king_counts_up_to_uint32_max(cuda_api):
    """Exactly UINT32_MAX rows: one device slab added 4,095 times and a prefix of it once.  Sample 0 is het, sample 1 hom
    A2 and sample 2 hom A1 on every row, so CC, HH, HC [0][0] and AB[1][2] reach 2^32 - 1; sample 3 is missing on every
    other row.  255 samples: one padding sample per row, whose bits are random."""
    import torch
    n = 255
    with cuda_api.King(n) as k:
        slab = k.slab_rows
        assert slab == 1 << 20                       # 1 GiB of planes / (4 planes x 256 padded samples)
        q, tail = divmod(UINT32_MAX, slab)
        gen = torch.Generator(device="cuda").manual_seed(255)
        v = torch.randint(0, 4, (slab, n), generator=gen, device="cuda", dtype=torch.uint8)
        v[:, 0] = 2
        v[:, 1] = 3
        v[:, 2] = 0
        v[::2, 3] = 1
        rows = torch_pack(v, gen)
        prefix = [w.round().to(torch.int64).cpu().numpy() for w in torch_planes_counts(v[:tail], n, step=1 << 17)]
        last = [w.round().to(torch.int64).cpu().numpy() for w in torch_planes_counts(v[tail:], n)]
        block = [p + r for p, r in zip(prefix, last)]
        del v
        half = (1 << 31) // slab + 1                 # slabs whose total first passes 2^31
        t0 = time.perf_counter()
        for i in range(q):
            k.add(rows)
            if i + 1 == half:
                c, got = counts_both(k)
                assert c.rows == half * slab > 1 << 31
                K.check(cuda_api, c, got, [half * b for b in block], f"{half} slabs")
        k.add(rows[:tail])
        c, got = counts_both(k)
        torch.cuda.synchronize()
        print(f"\n{UINT32_MAX:,} rows of {n} samples ({q} slabs + {tail} rows): {time.perf_counter() - t0:.1f} s")
        assert c.rows == UINT32_MAX
        want = [q * b + p for b, p in zip(block, prefix)]
        assert want[0][0, 0] == want[1][0, 0] == want[3][0, 0] == want[2][1, 2] == UINT32_MAX
        K.check(cuda_api, c, got, want, "UINT32_MAX rows")
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            k.add(rows[:1])                          # one row more: refused, nothing added
        assert e.value.code == E_INVALID
        c, again = counts_both(k)
        assert c.rows == UINT32_MAX and all(np.array_equal(a, b) for a, b in zip(again, got))


# ----------------------------------------------------------------------------- B. cohorts past C2
@pytest.mark.parametrize("n", (4097, 10000, 16385))
def test_king_large_cohorts_against_matmul(cuda_api, n):
    """Two slabs and 129 rows (three launches, the last with a partial K block) of seeded codes with an all-missing
    sample, an all-homozygous sample and duplicates, against float64 torch.matmul of the planes."""
    import torch
    s_pad = (n + 255) // 256 * 256
    need = 16 * s_pad * s_pad + 150 * n * n + (4 << 30)        # counts, their int32 / int64 copies, the reference, planes
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"{n} samples need about {need / 1e9:.0f} GB of device memory, {free / 1e9:.0f} GB are free")
    gen = torch.Generator(device="cuda").manual_seed(n)
    with cuda_api.King(n) as k:
        rows = 2 * k.slab_rows + 129
        v = torch.randint(0, 4, (rows, n), generator=gen, device="cuda", dtype=torch.uint8)
        v[:, 1] = 1
        v[:, 2] = torch.where(torch.rand(rows, generator=gen, device="cuda") < 0.5, 3, 0).to(torch.uint8)
        v[:, n - 1] = v[:, 0]
        v[:, n // 2] = v[:, 3]
        k.add(torch_pack(v, gen))
        c = k.counts()
    assert c.rows == rows
    want = torch_planes_counts(v, n)
    del v
    for name, g, w in zip(("CC", "HH", "AB", "HC"), (c.cc, c.hh, c.ab, c.hc), want):
        assert torch.equal(g, w.round().to(torch.int64)), f"n{n}: {name}"
    cc, hh, ab, hc = want
    del cc
    num = hc + hc.T - 2 * hh + 4 * (ab + ab.T)
    del hh, ab
    den = torch.minimum(hc, hc.T)
    kw = 0.5 - num / (4.0 * den)
    del num
    kin = c.kinship()
    nan = den == 0
    assert torch.equal(torch.isnan(kin), nan), f"n{n}: NA pattern"
    assert torch.equal(kin[~nan].view(torch.int64), kw[~nan].view(torch.int64)), f"n{n}: kinship not bit-equal"
    assert nan[1].all() and nan[:, 2].all() and kin[0, n - 1] == 0.5 and kin[3, n // 2] == 0.5


# ----------------------------------------------------------------------------- C. streams and devices
def test_king_on_its_own_stream(cuda_api):
    """A King on a side stream, fed a non-contiguous device view: the contiguous copy add() makes is written late (torch's
    current stream is asleep), and its memory is asked for again at once (the same size, filled on the current stream);
    then once more with the King's stream asleep, so the library reads late.  counts(device=True) is then called while
    the current stream still has to fill a freed block of the output's size.  Every count must be exact."""
    import torch
    n, rows = 513, 6000
    rng = np.random.default_rng(513)
    v, packed = packed_codes(rng, rows, n)
    big = np.zeros((2 * rows, packed.shape[1]), dtype=np.uint8)
    big[::2] = packed                                # (no device temporary of the rows' size that stale memory could match)
    big = torch.from_numpy(big).cuda()
    side = torch.cuda.Stream()
    k = cuda_api.King(n, stream=side.cuda_stream)
    try:
        torch.cuda.synchronize()
        torch.cuda._sleep(SLEEP)
        k.add(big[::2])
        junk = torch.empty((rows, packed.shape[1]), dtype=torch.uint8, device="cuda")
        junk.fill_(0x55)
        del junk
        with torch.cuda.stream(side):
            torch.cuda._sleep(SLEEP)
        k.add(big[::2])
        junk = torch.empty((rows, packed.shape[1]), dtype=torch.uint8, device="cuda")
        junk.fill_(0x55)
        del junk
        torch.cuda._sleep(SLEEP)
        junk = torch.empty((4, n, n), dtype=torch.int32, device="cuda")
        junk.fill_(7)
        del junk
        c = k.counts(device=True)
        got = [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)]
        assert c.rows == 2 * rows
        K.check(cuda_api, c, got, [2 * w for w in K.expected_counts(v)], "side stream")
    finally:
        k.close()


def test_king_two_streams_interleaved(cuda_api):
    """Two Kings on two side streams, their adds (contiguous slices and strided views of device rows) interleaved."""
    import torch
    rng = np.random.default_rng(77)
    cases = []
    for n in (300, 131):
        v, packed = packed_codes(rng, 4000, n)
        wide = np.zeros((2 * len(packed), packed.shape[1]), dtype=np.uint8)
        wide[1::2] = packed
        s = torch.cuda.Stream()
        cases.append((v, torch.from_numpy(wide).cuda(), s, cuda_api.King(n, stream=s.cuda_stream)))
    try:
        for a, b in ((0, 1000), (1000, 1001), (1001, 2500), (2500, 4000)):
            for i, (v, wide, s, k) in enumerate(cases):
                view = wide[1::2][a:b]
                k.add(view if i == 0 else view.clone())
        for v, wide, s, k in cases:
            c = k.counts(device=True)
            got = [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)]
            assert c.rows == 4000
            K.check(cuda_api, c, got, K.expected_counts(v), f"n{v.shape[1]} on its own stream")
    finally:
        for case in cases:
            case[3].close()


def test_king_second_device_keeps_current_device(cuda_api):
    """King(n, device=1) with rows on cuda:1 gives exact counts, and torch's current device is the same before and after
    every call; Kings on devices 0 and 1 used in turn are each exact."""
    import torch
    if cuda_api.device_count() < 2 or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(5)
    n = 260
    v, packed = packed_codes(rng, 3000, n)
    want = K.expected_counts(v)
    dev = torch.cuda.current_device()
    k = cuda_api.King(n, device=1)
    assert torch.cuda.current_device() == dev, "after create"
    k.add(torch.from_numpy(packed).to("cuda:1"))
    assert torch.cuda.current_device() == dev, "after add"
    c = k.counts()
    assert torch.cuda.current_device() == dev, "after counts"
    assert c.cc.device == torch.device("cuda:1")
    K.check(cuda_api, c, [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)], want, "device 1")
    k.close()
    assert torch.cuda.current_device() == dev, "after close"
    kings = [cuda_api.King(n, device=d) for d in (0, 1)]
    try:
        for a, b in ((0, 1200), (1200, 3000)):
            for d, k in enumerate(kings):
                k.add(torch.from_numpy(packed[a:b]).to(f"cuda:{d}"))
        for d, k in enumerate(kings):
            c = k.counts()
            K.check(cuda_api, c, [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)], want, f"device {d}, interleaved")
    finally:
        for k in kings:
            k.close()
    assert torch.cuda.current_device() == dev


# ----------------------------------------------------------------------------- D. refusals and recovery
def test_king_create_refuses_sizes_it_cannot_index(cuda_api):
    """Sample counts whose padded size does not fit the tile word, and those that do not fit uint32 at all, are refused
    at once, before anything is allocated; the accumulator goes on working."""
    for n in (MAX_SAMPLES + 1, 0xFFFFFF00, 0xFFFFFF01, UINT32_MAX):
        t0 = time.perf_counter()
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            K.new_king(cuda_api, n)
        assert e.value.code == E_INVALID, n
        assert time.perf_counter() - t0 < 5, n
    for n in (2 ** 32 + 5, 2 ** 40):
        with pytest.raises(ValueError):
            K.new_king(cuda_api, n)
    K.run_codes(cuda_api, K.random_codes(np.random.default_rng(3), 300, 7), "after the refusals")


def test_king_and_scan_work_after_an_allocation_failure(cuda_api, oracle):
    """A create whose counts do not fit the device fails with VCFX_E_NOMEM and gives its memory back, and so does a scan
    context whose output slot does not fit; the failures leave nothing behind that a later call could report: a fresh
    King is exact and allele_freq_calc equals the oracle.  The largest size the tile word takes is not refused either:
    its counts do not fit the device."""
    import torch
    from vcfx_b200 import synth
    data = synth.make_vcf(3, 400, 300, seed=11)
    _, total = torch.cuda.mem_get_info()
    for n in (120000, MAX_SAMPLES):
        s_pad = (n + 255) // 256 * 256
        assert 16 * s_pad * s_pad > total
        torch.cuda.synchronize()
        free0, _ = torch.cuda.mem_get_info()
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            cuda_api.King(n)
        assert e.value.code == E_NOMEM, n
        free1, _ = torch.cuda.mem_get_info()
        assert abs(free1 - free0) < 64 << 20, f"n{n}: {(free0 - free1) / 2 ** 20:.0f} MiB not given back"
        assert cuda_api.allele_freq_calc(data).out == oracle.allele_freq(data, 0).out, f"scan after King({n})"
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            cuda_api.King(n)
        K.run_codes(cuda_api, K.random_codes(np.random.default_rng(n), 700, 300), f"King after King({n})", device=True)
    with cuda_api.Context(cuda_api.OP_ALLELE_FREQ, out_bytes=total) as ctx:
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            ctx.acquire()                            # the output slot is as large as the device
        assert e.value.code == E_NOMEM
    assert cuda_api.allele_freq_calc(data).out == oracle.allele_freq(data, 0).out, "scan after a failed slot"
    with pytest.raises(cuda_api.VcfxCudaError):
        cuda_api.King(120000)
    K.run_codes(cuda_api, K.random_codes(np.random.default_rng(1), 700, 129), "King after a failed slot")
