"""KING-robust relatedness counts (vcfx_cuda_king_*, api.King, api.king) on the tensor cores.

The expected counts do not come from the library: codes come from the oracle's dosage text (as test_gpu_dosage_bed.py
reads them) or from a seeded generator, numpy turns them into the four 0/1 planes (A hom REF, H het, B hom ALT, C called)
and multiplies them (float64 BLAS, exact for integers below 2^53).  All four count matrices must be equal and kinship
bit-equal to numpy's float64 of the same expression (NaN for NA).  test_emu_king.py runs the small cases under the warp
emulator, where the MMA reads its operands through the same descriptors.
"""
import functools

import numpy as np
import pytest

import test_gpu_dosage_bed as B
import test_gpu_dosage_matrix as D
import test_gpu_parity as G
import test_gpu_resident as R
from vcfx_b200 import synth

pytestmark = pytest.mark.gpu

E_INVALID = -1
SAMPLES = (1, 2, 3, 4, 5, 127, 128, 129, 255, 256, 257, 2504)
ROWS = (0, 1, 127, 128, 129)


@pytest.fixture
def resident():
    return functools.partial(R.run_resident, R.TorchMem())


# ----------------------------------------------------------------------------- helpers
def emulated(api):
    return "emu" in api.lib_path().name


def new_king(api, n):
    """A King on torch's current stream, or (emulator, no torch device) on the default stream."""
    return api.King(n, stream=0) if emulated(api) else api.King(n)


def counts_np(api, k):
    c = k.counts(device=not emulated(api))
    assert c.cc.is_cuda != emulated(api)
    return c, [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)]


def add_device(api, k, rows):
    """rows (numpy uint8 [n, B]) as device memory: a CUDA tensor, or (emulator) host memory passed as on_device."""
    rows = np.ascontiguousarray(rows, dtype=np.uint8)
    if emulated(api):
        k._add(rows.ctypes.data, rows.shape[0], True)
    else:
        import torch
        k.add(torch.from_numpy(rows).cuda())


def bed_codes(dosage_codes):
    """dosage codes (2 / 1 / 0, -1 NA, -2 no column) -> .bed codes (00 / 10 / 11 / 01 as 0 / 2 / 3 / 1)."""
    d = np.asarray(dosage_codes)
    v = np.ones(d.shape, dtype=np.uint8)
    v[d == 2] = 0
    v[d == 1] = 2
    v[d == 0] = 3
    return v


def pack_codes(v, garbage=None):
    """.bed rows of .bed codes [rows, n]; garbage: random bits for the padding of each row's last byte."""
    rows, n = v.shape
    nb = (n + 3) // 4
    full = np.zeros((rows, 4 * nb), dtype=np.uint8)
    full[:, :n] = v
    if garbage is not None and n % 4:
        full[:, n:] = garbage.integers(0, 4, size=(rows, 4 * nb - n), dtype=np.uint8)
    q = full.reshape(rows, nb, 4)
    return (q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6)).astype(np.uint8)


def expected_counts(v, step=1 << 16):
    """CC, HH, AB, HC of .bed codes [rows, n] as int64, from float64 products of the planes over row blocks."""
    n = v.shape[1]
    out = [np.zeros((n, n), dtype=np.int64) for _ in range(4)]
    for r0 in range(0, v.shape[0], step):
        x = v[r0:r0 + step]
        a, h, b = (x == 3).astype(np.float64), (x == 2).astype(np.float64), (x == 0).astype(np.float64)
        c = (x != 1).astype(np.float64)
        for o, (p, q) in zip(out, ((c, c), (h, h), (a, b), (h, c))):
            o += np.rint(p.T @ q).astype(np.int64)
    return out


def expected_kinship(cc, hh, ab, hc):
    het1, het2 = hc, hc.T
    num = (het1 + het2 - 2 * hh + 4 * (ab + ab.T)).astype(np.float64)
    den = np.minimum(het1, het2)
    with np.errstate(divide="ignore", invalid="ignore"):
        k = 0.5 - num / (4.0 * den.astype(np.float64))
    k[den == 0] = np.nan
    return k


def check(api, c, got, want, tag):
    for name, g, w in zip(("CC", "HH", "AB", "HC"), got, want):
        assert g.shape == w.shape, (tag, name)
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            i, j = bad[0]
            raise AssertionError(f"{tag}: {name} differs at {len(bad)} places, first ({i}, {j}): {g[i, j]} != {w[i, j]}")
    k = c.kinship().cpu().numpy()
    kw = expected_kinship(*want)
    assert np.array_equal(np.isnan(k), np.isnan(kw)), tag
    assert np.array_equal(k.view(np.int64)[~np.isnan(kw)], kw.view(np.int64)[~np.isnan(kw)]), f"{tag}: kinship not bit-equal"


def run_codes(api, v, tag, garbage=None, device=False, pieces=1):
    """One King over the .bed codes v, added in `pieces` calls from the host or from device memory; checked."""
    k = new_king(api, v.shape[1])
    try:
        rows = pack_codes(v, garbage)
        cuts = np.linspace(0, len(rows), pieces + 1).astype(int)
        for a, b in zip(cuts[:-1], cuts[1:]):
            if device:
                add_device(api, k, rows[a:b])
            else:
                k.add(rows[a:b])
        c, got = counts_np(api, k)
        assert c.rows == len(rows), tag
        check(api, c, got, expected_counts(v), tag)
        return got
    finally:
        k.close()


def random_codes(rng, rows, n):
    return rng.integers(0, 4, size=(rows, n), dtype=np.uint8)


# ----------------------------------------------------------------------------- 1. shapes
@pytest.mark.parametrize("n", SAMPLES)
@pytest.mark.parametrize("rows", ROWS)
def test_king_sample_and_row_counts(cuda_api, n, rows):
    if emulated(cuda_api) and n > 257:
        pytest.skip("2,504 samples stay on the GPU")
    rng = np.random.default_rng(1000 * n + rows)
    run_codes(cuda_api, random_codes(rng, rows, n), f"n{n} rows{rows}", garbage=rng)


@pytest.mark.parametrize("n", (5, 257))
def test_king_slab_borders(cuda_api, n):
    """Rows at one slab - 1, one slab, one slab + 1 and several slabs: each full slab is a launch of its own."""
    with new_king(cuda_api, n) as k:
        slab = k.slab_rows
    assert slab % 128 == 0
    rng = np.random.default_rng(n)
    for rows in (slab - 1, slab, slab + 1, 3 * slab + 5):
        run_codes(cuda_api, random_codes(rng, rows, n), f"n{n} rows{rows} slab{slab}", garbage=rng, pieces=3)


def test_king_padding_bits_are_ignored(cuda_api):
    """Whatever the padding bits of a row's last byte hold, the counts are those of 00 padding."""
    rng = np.random.default_rng(7)
    for n in (1, 2, 3, 5, 6, 7, 129, 255):
        v = random_codes(rng, 200, n)
        clean = run_codes(cuda_api, v, f"n{n} clean")
        dirty = run_codes(cuda_api, v, f"n{n} garbage", garbage=rng)
        for a, b in zip(clean, dirty):
            assert np.array_equal(a, b), n


def test_king_na_and_duplicates(cuda_api):
    """An all-missing sample and an all-hom sample have HET = 0 against everyone (NA); duplicated samples give exactly 0.5."""
    rng = np.random.default_rng(11)
    v = random_codes(rng, 300, 9)
    v[:, 1] = 1                          # all missing
    v[:, 2] = np.where(rng.integers(0, 2, 300) == 1, 3, 0)     # hom REF or hom ALT only
    v[:, 5] = v[:, 4]                    # duplicates
    v[:, 8] = v[:, 0]
    k = new_king(cuda_api, 9)
    k.add(pack_codes(v))
    c, got = counts_np(cuda_api, k)
    check(cuda_api, c, got, expected_counts(v), "na/dup")
    kin = c.kinship().cpu().numpy()
    assert np.isnan(kin[1]).all() and np.isnan(kin[:, 2]).all()
    assert kin[4, 5] == 0.5 and kin[0, 8] == 0.5 and kin[3, 3] == 0.5
    k.close()


def test_king_several_adds_and_device_rows(cuda_api):
    """Several add calls give the counts of one call; rows in device memory give the counts of host rows; counts() may be
    called in between and the accumulator goes on."""
    rng = np.random.default_rng(3)
    v = random_codes(rng, 1000, 130)
    one = run_codes(cuda_api, v, "one call")
    for pieces in (2, 7):
        for device in (False, True):
            got = run_codes(cuda_api, v, f"{pieces} pieces device={device}", device=device, pieces=pieces)
            assert all(np.array_equal(a, b) for a, b in zip(one, got))
    with new_king(cuda_api, 130) as k:
        k.add(pack_codes(v[:400]))
        c, got = counts_np(cuda_api, k)
        check(cuda_api, c, got, expected_counts(v[:400]), "first part")
        add_device(cuda_api, k, pack_codes(v[400:]))
        c, got = counts_np(cuda_api, k)
        assert c.rows == 1000
        check(cuda_api, c, got, one, "after a counts() call")


def test_king_refusals(cuda_api):
    with new_king(cuda_api, 10) as k:
        with pytest.raises(ValueError):
            k.add(np.zeros((4, 2), dtype=np.uint8))                 # 10 samples take 3 bytes
        with pytest.raises(ValueError):
            k.add(np.zeros((4, 3), dtype=np.int8))
        bed = cuda_api.DosageBed([], 9, None, None, None, None, cuda_api.Totals())
        with pytest.raises(ValueError):
            k.add(bed)
        k.add(pack_codes(np.full((5, 10), 2, dtype=np.uint8)))
        big = np.zeros((1, 3), dtype=np.uint8)
        with pytest.raises(cuda_api.VcfxCudaError) as e:
            k._add(big.ctypes.data, (1 << 32) - 5, False)             # past UINT32_MAX rows in all: refused, nothing added
        assert e.value.code == E_INVALID
        k._add(big.ctypes.data, 0, False)
        c, got = counts_np(cuda_api, k)
        assert c.rows == 5 and got[0][0, 0] == 5 and got[1][0, 0] == 5
    with pytest.raises(ValueError):
        cuda_api.King(0)


# ----------------------------------------------------------------------------- 2. the .bed corpora
def corpus_cases():
    cases = [(f"shape{s} {V}x{S}", functools.partial(G.shape_input, s, V, S)) for s, V, S in G.SHAPES]
    cases += [(f"fuzz{seed}", functools.partial(G.adversarial_input, seed)) for seed in range(0, 40, 3)]
    cases += [(f"degenerate{i}", (lambda d=d: d)) for i, d in enumerate(G.DEGENERATE)]
    cases += [(f"ds S{S}", functools.partial(D.ds_lattice_input, S)) for S in (1, 2, 127, 128, 129, 257)]
    cases += [(f"sweep S{S}", functools.partial(G.sweep_input, 2, S)) for S in (119, 255, 256, 257)]
    return cases


CORPUS = corpus_cases()


def run_corpus(api, O, resident, data, tag):
    for mode in B.MODES:
        if O.dosage(data, mode).first_bad_line:
            with pytest.raises(api.VcfxCudaError, match=r"VCF header \(#CHROM\) not found"):
                api.dosage_bed(data, mode)
            continue
        W = D.widest(data)
        if W == 0 or (emulated(api) and W > 257):
            continue
        v = bed_codes(B.oracle_codes(O, data, mode, W)[0])
        want = expected_counts(v)
        beds = [api.dosage_bed(data, mode, width=W, chunk_bytes=D.small_chunk(data))]
        if data and resident is not None:
            got = resident(api, api.OP_DOSAGE, mode, data, out_cap=B.out_cap_for(data, W), ctx_kw=B.bed_kw(api, W))
            beds.append(B.from_resident(api, got, W))
        for how, bed in zip(("4 KiB chunks", "resident"), beds):
            with new_king(api, W) as k:
                k.add(bed)
                c, got = counts_np(api, k)
            assert c.rows == len(v)
            check(api, c, got, want, f"{tag} mode{mode} {how}")


@pytest.mark.parametrize("case", range(len(CORPUS)), ids=[c[0] for c in CORPUS])
def test_king_corpora(cuda_api, oracle, resident, case):
    tag, make = CORPUS[case]
    run_corpus(cuda_api, oracle, resident, make(), tag)


def test_king_end_to_end_and_device_bed(cuda_api, oracle):
    """api.king on VCF bytes, and api.dosage_bed_device's packed rows straight into a King."""
    import torch
    data = G.shape_input(2, 300, 300)
    host = cuda_api.dosage_bed(data)
    want = expected_counts(bed_codes(B.oracle_codes(oracle, data, 0, host.width)[0]))
    c = cuda_api.king(data)
    assert c.samples == host.samples and c.rows == 300
    check(cuda_api, c, [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)], want, "api.king")
    d_in = torch.zeros(len(data) + cuda_api.DEVICE_PAD, dtype=torch.uint8, device="cuda")
    d_in[:len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    bed = cuda_api.dosage_bed_device(d_in, len(data))
    with cuda_api.King(bed.width) as k:
        k.add(bed.packed)
        k.add(bed)                                   # (a DosageBed with device rows)
        c = k.counts()
    check(cuda_api, c, [t.cpu().numpy() for t in (c.cc, c.hh, c.ab, c.hc)], [2 * w for w in want], "device rows twice")


# ----------------------------------------------------------------------------- 3. statistics and scale (GPU only)
def test_king_simulated_pedigree(cuda_api):
    """A seeded pedigree as a sanity check of the estimator only: parent-offspring and full sibs near 0.25, unrelated
    founders near 0, a duplicate at 0.5."""
    rng = np.random.default_rng(2024)
    V, F = 20000, 16
    p = rng.uniform(0.05, 0.95, V)
    hap = (rng.random((F, 2, V)) < p).astype(np.uint8)          # founders' haplotypes: 1 = ALT
    kids = []
    for f in range(0, 8, 2):                                     # four couples, two children each
        for _ in range(2):
            a = hap[f, rng.integers(0, 2, V), np.arange(V)]
            b = hap[f + 1, rng.integers(0, 2, V), np.arange(V)]
            kids.append(np.stack([a, b]))
    all_hap = np.concatenate([hap, np.array(kids)])
    dos = all_hap.sum(axis=1).T                                  # [V, samples] dosage
    dos = np.concatenate([dos, dos[:, :1]], axis=1)              # sample 24 duplicates sample 0
    with cuda_api.King(dos.shape[1]) as k:
        k.add(pack_codes(bed_codes(dos)))
        kin = k.counts().kinship().cpu().numpy()
    po = [kin[2 * (j // 2) + parent, F + j] for j in range(8) for parent in (0, 1)]
    sibs = [kin[F + 2 * c, F + 2 * c + 1] for c in range(4)]
    unrel = [kin[i, j] for i in range(F) for j in range(i + 1, F)]            # (founders, spouses included)
    assert all(0.2 < x < 0.3 for x in po), po
    assert all(0.15 < x < 0.35 for x in sibs), sibs
    assert max(abs(x) for x in unrel) < 0.06, max(unrel)
    assert kin[0, 24] == 0.5


def test_king_c2_shape_against_matmul(cuda_api):
    """2,504 samples x 427,409 variants from synth through dosage_bed_device, counted by the MMA kernel in several slabs,
    against float64 torch.matmul of planes unpacked on the GPU."""
    import torch
    data = synth.make_vcf(2, 427409, 2504, seed=7)
    d_in = torch.zeros(len(data) + cuda_api.DEVICE_PAD, dtype=torch.uint8, device="cuda")
    d_in[:len(data)] = torch.frombuffer(data, dtype=torch.uint8).cuda()
    bed = cuda_api.dosage_bed_device(d_in, len(data))
    del d_in
    n = bed.width
    assert n == 2504 and bed.packed.shape[0] == 427409
    with cuda_api.King(n) as k:
        assert k.slab_rows < 427409
        k.add(bed)
        c = k.counts()
    want = [torch.zeros((n, n), dtype=torch.float64, device="cuda") for _ in range(4)]
    shifts = torch.arange(0, 8, 2, device="cuda", dtype=torch.uint8)
    for r0 in range(0, 427409, 32768):
        x = ((bed.packed[r0:r0 + 32768, :, None] >> shifts) & 3).reshape(-1, 4 * bed.packed.shape[1])[:, :n]
        a, h, b = (x == 3).double(), (x == 2).double(), (x == 0).double()
        cc = (x != 1).double()
        for w, (p, q) in zip(want, ((cc, cc), (h, h), (a, b), (h, cc))):
            w += p.T @ q
    for name, g, w in zip(("CC", "HH", "AB", "HC"), (c.cc, c.hh, c.ab, c.hc), want):
        assert torch.equal(g, w.round().to(torch.int64)), name
