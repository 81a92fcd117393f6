"""The ordering layer (K1c / K1d) at every launch path against NumPy's stable argsort.

The radix argsort picks its code path from n and from sx_sort_set_tuning, and nothing reports which one ran:

  * n <= 8192: one CTA, every pass in shared memory (rs_small_sort_kernel);
  * up to 64 tiles of 4096 keys: one cooperative launch of 512-thread tiles;
  * up to one resident CTA per SM (148 x 8192 keys on a B200): one cooperative launch of 1024-thread tiles;
  * above that, or with sx_sort_set_tuning(0): upsweep / scan / downsweep launches per pass, 256, 384, 512 or
    1024 threads per tile (512 by default, 1024 from 2^26 keys, where the grid cap also changes to 888 CTAs).

A wrong order still gives a spanning tree, just not the reference's, so every output here is compared exactly
with a literal reference:

  * sort:   np.argsort(key, kind="stable"); sorted keys are the bits of key[ref] with -0.0 read as +0.0 and every
            NaN as 0x7FFFFFFFFFFFFFFF (sort_key_to_f64(f64_to_sort_key(v)), sx_common.cuh), compared bit for bit;
  * queue:  ref[::-1];
  * Kruskal order: np.argsort(-key, kind="stable") (oracle.kruskal_order), only for keys without NaN -- NaN
            weights are rejected before a Kruskal order is built (tree_BI.py);
  * heads and prefixes: the first entries of that order, with the length the 24-bit threshold rule gives;
  * histogram: np.bincount(image >> 52, minlength=4096).

Key families, each seeded: full 64-bit patterns (every byte of every pass varies, NaNs of both signs), special
values (signed zeros, subnormals, +-DBL_MAX, +-inf, quiet and signalling NaNs of both signs) among random ones,
64 repeated full-precision values, a constant, sorted and reverse-sorted input, and keys that vary only in their
top two bytes or only in their low six.  Sizes sit on the edges of every path: one tile either side of a tile
boundary, the grid sizes where a downsweep CTA goes from one tile to two, a partial last tile with three tiles per
CTA, the cooperative limits and the 2^26 switch.  A profiler trace proves which kernel each path table entry runs.

sx_sort_set_tuning is process-wide; the `sort_path` fixture restores both defaults after every test.  The tests
without the `gpu` marker check the generators, the references and the path table itself.
"""
import ctypes
import functools
import re

import numpy as np
import pytest

from oracle import network_oracle as orc

SMALL_MAX = 8192              # kSmallSortMax: one CTA up to this many keys
ITEMS = 8                     # kRsItems: keys per thread, tile = 8 x threads
MAX_GRID = 148 * 6            # kRsMaxGrid: grid cap of the launch-per-pass path from 2^26 keys
BIG = 1 << 26                 # from here: 1024-thread tiles by default and the 888-CTA grid cap
COOP512_MAX_TILES = 64        # the cooperative launch takes 1024-thread tiles above 64 tiles of 4096 keys
KO_TILE = 4096                # kKoTile: positions per block of sx_kruskal_order
PF_BND_FACTOR = 4             # kPfBndFactor: boundary list of sx_kruskal_prefix holds 4 x T_cap arcs
TUNING_THREADS_DEFAULT, TUNING_COOP_DEFAULT = 2, 1

SIGN = np.uint64(1 << 63)
ALL = np.uint64(0xFFFFFFFFFFFFFFFF)
NAN_OUT = np.uint64(0x7FFFFFFFFFFFFFFF)   # sort_key_to_f64(~0): the bits every NaN comes out as


# ==== references ============================================================================================
def sort_image(v):
    """f64_to_sort_key (sx_common.cuh): ascending uint64 == NumPy's ascending order, -0.0 == +0.0, NaN last."""
    b = np.ascontiguousarray(v, dtype=np.float64).view(np.uint64).copy()
    b[(b << np.uint64(1)) == 0] = 0
    nan = (b & ~SIGN) > np.uint64(0x7FF0000000000000)
    out = np.where((b >> np.uint64(63)) == 1, ~b, b | SIGN)
    out[nan] = ALL
    return out


def image_to_bits(k):
    """sort_key_to_f64, as bits."""
    k = np.asarray(k, dtype=np.uint64)
    return np.where((k >> np.uint64(63)) == 1, k & ~SIGN, ~k)


def sorted_bits_ref(key, ref):
    """The sorted keys sx_argsort_f64 writes: key[ref] with -0.0 as +0.0 and every NaN as 0x7FF...F."""
    s = key[ref]
    bits = s.view(np.uint64).copy()
    bits[(bits << np.uint64(1)) == 0] = 0
    bits[np.isnan(s)] = NAN_OUT
    return bits


def u64_sorted_bits(key_bits):
    """sx_argsort_u64 sorts whole bytes, at least two: the low 8 * max(2, ceil(key_bits / 8)) bits."""
    return 8 * max(2, -(-key_bits // 8))


def u64_mask(key_bits):
    b = u64_sorted_bits(key_bits)
    return ALL if b == 64 else np.uint64((1 << b) - 1)


def prefix_count(asc24, T):
    """Arcs sx_kruskal_prefix returns: every arc whose 24-bit image prefix is >= that of the T-th heaviest (all of
    them when T > n).  asc24: the prefixes, ascending."""
    n = asc24.size
    if T > n:
        return n, 0
    thr = asc24[n - T]
    return n - int(np.searchsorted(asc24, thr, side="left")), int(thr)


# ==== the path table ========================================================================================
def rs_plan(n, threads):
    """rs_plan in sx_sort.cu for an explicit downsweep shape: (tiles, tiles per CTA, grid)."""
    sms = num_sms()
    tile = threads * ITEMS
    tiles = max(1, -(-n // tile))
    cap = ((1 if threads == 1024 else 2) * sms) if n < BIG else MAX_GRID
    cap = min(cap, MAX_GRID)
    tpb = -(-tiles // cap)
    return tiles, tpb, -(-tiles // tpb)


def resident_limit():
    """Largest n of the 1024-thread cooperative launch: one 8192-key tile per SM (one CTA fits an SM)."""
    return num_sms() * 1024 * ITEMS


def expected_path(n, coop, threads):
    """("small", 1024) | ("coop", 512 / 1024) | ("downsweep", threads) for sx_sort_set_tuning(coop), (threads)."""
    if n <= SMALL_MAX:
        return "small", 1024
    ct = 1024 if -(-n // 4096) > COOP512_MAX_TILES else 512
    if coop and (ct == 512 or n <= resident_limit()):      # at most 64 tiles of 512 threads: always resident
        return "coop", ct
    return "downsweep", threads if threads != 2 else (1024 if n >= BIG else 512)


# path name -> (sx_sort_set_tuning(0 / 1), sx_sort_set_tuning(threads))
PATHS = {
    "small": (1, 2), "coop512": (1, 2), "coop1024": (1, 2),
    "ds256": (0, 256), "ds384": (0, 384), "ds512": (0, 512), "ds1024": (0, 1024),
    "default": (1, 2),
}
DS_LABELS = ["kt-1", "kt", "kt+1", "grid*t-1", "grid*t", "grid*t+1", "3grid*t-12345"]
SIZE_LABELS = {
    "small": ["1", "2", "3", "33", "1025", "4097", "8191", "8192"],
    "coop512": ["8193", "100001", "262143", "262144"],
    "coop1024": ["262145", "500001", "resident-1", "resident"],
    "ds256": DS_LABELS, "ds384": DS_LABELS, "ds512": DS_LABELS, "ds1024": DS_LABELS,
    "default": ["2^26-1", "2^26+12345"],
}


def path_size(path, label):
    """The size behind a label, on this device (grid caps and the resident limit follow its SM count)."""
    if path.startswith("ds"):
        threads = int(path[2:])
        t = threads * ITEMS
        kt = (SMALL_MAX // t + 1) * t                 # first tile multiple above the single-CTA limit
        g = min(MAX_GRID, (1 if threads == 1024 else 2) * num_sms()) * t
        return {"kt-1": kt - 1, "kt": kt, "kt+1": kt + 1, "grid*t-1": g - 1, "grid*t": g, "grid*t+1": g + 1,
                "3grid*t-12345": 3 * g - 12345}[label]
    if label.startswith("resident"):
        return resident_limit() + (-1 if label.endswith("-1") else 0)
    if label.startswith("2^26"):
        return BIG - 1 if label == "2^26-1" else BIG + 12345
    return int(label)


_SMS = [None]


def num_sms():
    """SM count of the device (148 on a B200); the CPU tests use 148."""
    if _SMS[0] is None:
        try:
            import torch
            _SMS[0] = torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148
        except ImportError:
            _SMS[0] = 148
    return _SMS[0]


# ==== key families ==========================================================================================
def random_bits(rng, n):
    return np.frombuffer(rng.bytes(8 * n), dtype=np.uint64).copy()


def as_f64(bits):
    return np.ascontiguousarray(bits, dtype=np.uint64).view(np.float64)


SPECIAL_BITS = np.array([
    0x0000000000000000, 0x8000000000000000,            # +0, -0
    0x0000000000000001, 0x8000000000000001,            # +-smallest subnormal
    0x000FFFFFFFFFFFFF, 0x800ABCDEF0123457,            # other subnormals
    0x7FEFFFFFFFFFFFFF, 0xFFEFFFFFFFFFFFFF,            # +-DBL_MAX
    0x7FF0000000000000, 0xFFF0000000000000,            # +-inf
    0x7FF8000000000000, 0xFFF8000000000000,            # quiet NaN, both signs
    0x7FF0000000000001, 0xFFF4000000000000,            # signalling NaN, both signs
    0x7FFFFFFFFFFFFFFF, 0xFFFFFFFFFFFFFFFF,            # all-ones NaN payloads
], dtype=np.uint64)


def gen_full(rng, n):
    """Random 64-bit patterns: every byte of every pass varies; NaN patterns of both signs planted."""
    b = random_bits(rng, n)
    if n >= 8:
        b[rng.integers(0, n, 2)] = [0x7FF123456789ABCD, 0xFFF0000000000BAD]
    return as_f64(b)


def gen_special(rng, n):
    """Random finite values of many magnitudes with the special values scattered through them (1 in 8)."""
    v = rng.standard_normal(n) * 10.0 ** rng.uniform(-300, 300, n)
    b = v.view(np.uint64)
    pos = np.flatnonzero(rng.random(n) < 0.125)
    b[pos] = SPECIAL_BITS[rng.integers(0, SPECIAL_BITS.size, pos.size)]
    if n >= SPECIAL_BITS.size:                           # every special value at least once
        b[rng.choice(n, SPECIAL_BITS.size, replace=False)] = SPECIAL_BITS
    return v


def gen_ties(rng, n):
    """About 64 distinct full-precision values of both signs, repeated."""
    vals = rng.standard_normal(64) * 2.0 ** rng.integers(-900, 900, 64)
    return vals[rng.integers(0, 64, n)]


def gen_constant(rng, n):
    return np.full(n, -1.2345678901234567e-3)            # negative, no zero byte: every pass complements


def gen_sorted(rng, n):
    v = np.sort(gen_special(rng, n))                     # NaNs last, as NumPy sorts them
    if n >= 4:
        v[1:n // 2:5] = v[0:n // 2 - 1:5]                 # ties
    return v


def gen_reversed(rng, n):
    return gen_sorted(rng, n)[::-1].copy()


def gen_high16(rng, n):
    """Equal in bytes 0-5, varying in bytes 6-7 (sign, exponent, top mantissa bits)."""
    return as_f64(np.uint64(0x0000A5C3E1F0B4D7) | (random_bits(rng, n) & np.uint64(0xFFFF000000000000)))


def gen_low48(rng, n):
    """Varying in bytes 0-5, equal in bytes 6-7 (negative: every digit is complemented)."""
    return as_f64(np.uint64(0xC123000000000000) | (random_bits(rng, n) & np.uint64(0x0000FFFFFFFFFFFF)))


FAMILIES = {"full": gen_full, "special": gen_special, "ties": gen_ties, "constant": gen_constant,
            "sorted": gen_sorted, "reversed": gen_reversed, "high16": gen_high16, "low48": gen_low48}
LARGE_FAMILIES = ["full", "special", "ties", "constant"]     # sizes of millions: the families that differ most
BIG_FAMILIES = ["full", "constant"]                          # the 2^26 sizes: NumPy's sort takes ~20 s per case


def family_seed(family, n):
    return (list(FAMILIES).index(family) + 1) * 1_000_003 + n


def make_keys(family, n):
    return FAMILIES[family](np.random.default_rng(family_seed(family, n)), n)


def without_nan(key, rng):
    """NaN-free copy: each NaN replaced by a random finite value (the prefix and Kruskal order take no NaN)."""
    key = key.copy()
    nan = np.isnan(key)
    key[nan] = rng.standard_normal(int(nan.sum()))
    return key


@functools.lru_cache(maxsize=6)
def sort_case(family, n):
    """Keys and their references, shared by every path that sorts the same size."""
    key = make_keys(family, n)
    ref = np.argsort(key, kind="stable")
    kref = None if np.isnan(key).any() else orc.kruskal_order(key)
    return key, ref, kref


def byte_values(bits):
    """Distinct values of each of the 8 bytes."""
    return [np.unique((bits >> np.uint64(8 * i)) & np.uint64(0xFF)).size for i in range(8)]


# ==== CPU tests: references, generators, path table =========================================================
def test_reference_image_and_sorted_bits():
    """sort_image is monotone and matches NumPy's order (NaN last, -0.0 == +0.0); the sorted-key reference is
    image_to_bits(sort_image(v)) -- the round trip the kernels write."""
    for fam in FAMILIES:
        key = make_keys(fam, 5000)
        img = sort_image(key)
        ref = np.argsort(key, kind="stable")
        assert np.all(img[ref][1:] >= img[ref][:-1])
        assert np.array_equal(np.argsort(img, kind="stable"), ref)
        assert np.array_equal(sorted_bits_ref(key, ref), image_to_bits(img[ref]))
    special = as_f64(SPECIAL_BITS)
    img = sort_image(special)
    assert img[0] == img[1] == SIGN                               # +0 and -0 share one image
    assert np.all(img[np.isnan(special)] == ALL)                  # every NaN last
    assert image_to_bits(ALL) == NAN_OUT
    # bin 2048: +-0 and the two positive subnormals; bin 2047: the negative ones; bin 4095: +inf and the 6 NaNs
    assert np.array_equal(np.bincount((img >> np.uint64(52)).astype(np.int64), minlength=4096)[[2047, 2048, 4095]],
                          [2, 4, 7])


@pytest.mark.parametrize("n", [33, 5000, 100001])
def test_generator_plants_what_it_claims(n):
    full = make_keys("full", n).view(np.uint64)
    assert min(byte_values(sort_image(full.view(np.float64)))) >= 2          # a nonconstant digit in every pass
    assert min(byte_values(full)) >= 2                                      # and in the raw first-pass byte
    fnan = np.isnan(full.view(np.float64))
    assert (fnan & (full >> np.uint64(63) == 1)).any() and (fnan & (full >> np.uint64(63) == 0)).any()

    sp = make_keys("special", n)
    if n >= SPECIAL_BITS.size:
        assert set(SPECIAL_BITS.tolist()) <= set(sp.view(np.uint64).tolist())
        sb = sp.view(np.uint64)
        sub = (np.abs(sp) < 2.2250738585072014e-308) & (sp != 0)
        assert np.unique(sb[sub] & ~SIGN).size >= 3                         # the smallest and other subnormals
        ordinary = np.isfinite(sp) & (sp != 0)
        assert ordinary.sum() > n // 2
        if n >= 5000:                                                       # of many magnitudes
            assert np.unique(np.floor(np.log10(np.abs(sp[ordinary])))).size > 500

    ties = make_keys("ties", n)
    u = np.unique(ties)
    assert 2 <= u.size <= 64 and (n < 1000 or u.size == 64)
    assert np.mean((u.view(np.uint64) & np.uint64(0xFFFF)) != 0) > 0.9      # full precision
    assert (u < 0).any() and (u > 0).any()

    assert np.unique(make_keys("constant", n)).size == 1
    s, r = make_keys("sorted", n), make_keys("reversed", n)
    sf = s[~np.isnan(s)]
    assert np.all(sf[1:] >= sf[:-1]) and np.all(np.isnan(s[sf.size:])) and np.unique(sf).size < sf.size
    rf = r[~np.isnan(r)]
    assert np.all(rf[1:] <= rf[:-1]) and np.all(np.isnan(r[:r.size - rf.size]))

    hi = make_keys("high16", n).view(np.uint64)
    assert byte_values(hi)[:6] == [1] * 6 and min(byte_values(hi)[6:]) >= 2
    lo = make_keys("low48", n).view(np.uint64)
    assert byte_values(lo)[6:] == [1, 1] and min(byte_values(lo)[:6]) >= 2
    assert np.all(lo.view(np.float64) < 0)


def test_path_table():
    """The sizes behind every label take the path they are named for, and sit where they claim (tile and
    tiles-per-CTA boundaries, a partial last tile) -- on a 148-SM device."""
    for path, labels in SIZE_LABELS.items():
        coop, threads = PATHS[path]
        for lab in labels:
            n = path_size(path, lab)
            kind, th = expected_path(n, coop, threads)
            if path == "small":
                assert kind == "small"
            elif path.startswith("coop"):
                assert (kind, th) == ("coop", int(path[4:])), (path, lab, n)
            elif path.startswith("ds"):
                assert (kind, th) == ("downsweep", int(path[2:])), (path, lab, n)
                t = th * ITEMS
                tiles, tpb, grid = rs_plan(n, th)
                if lab.startswith("kt"):
                    assert SMALL_MAX < n and (n % t in (t - 1, 0, 1))
                elif lab == "grid*t+1":
                    assert tpb == 2
                elif lab.startswith("grid*t"):
                    assert tpb == 1
                else:
                    assert tpb == 3 and n % t != 0
            else:
                assert kind == "downsweep" and th == (512 if n < BIG else 1024)
    if num_sms() == 148:
        assert resident_limit() == 1212416
        assert rs_plan(BIG - 1, 512)[1:] == (56, 293) and rs_plan(BIG + 12345, 1024)[1:] == (10, 820)
    assert expected_path(resident_limit() + 1, 1, 2) == ("downsweep", 512)
    assert expected_path(64 * 4096, 1, 2) == ("coop", 512) and expected_path(64 * 4096 + 1, 1, 2) == ("coop", 1024)


def test_u64_mask_rule():
    """Whole bytes, at least two: 1 and 8 bits sort 16, 9 sorts 16, 17 sorts 24, 63 and 64 sort all 64."""
    assert [u64_sorted_bits(b) for b in (1, 8, 9, 16, 17, 32, 33, 56, 63, 64)] == [16, 16, 16, 16, 24, 32, 40, 56, 64, 64]


def test_prefix_reference_counts():
    """prefix_count against a direct restatement: threshold = 24-bit prefix of the T-th heaviest weight."""
    rng = np.random.default_rng(4)
    w = without_nan(make_keys("special", 3001), rng)
    p = np.sort(sort_image(w) >> np.uint64(40))
    desc = np.sort(sort_image(w))[::-1] >> np.uint64(40)
    for T in (1, 2, 100, 1500, 3000, 3001, 3006):
        c, thr = prefix_count(p, T)
        if T <= w.size:
            assert thr == desc[T - 1] and c == int((desc >= desc[T - 1]).sum()) and c >= T
        else:
            assert c == w.size
        ko = orc.kruskal_order(w)
        if c < w.size:                                     # the cut falls between two different prefixes
            assert (sort_image(w[ko[c]]) >> np.uint64(40)) < (sort_image(w[ko[c - 1]]) >> np.uint64(40))


# ==== GPU fixtures and helpers ==============================================================================
@pytest.fixture(scope="module")
def dev():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from smart_crossover import device
    return device


@pytest.fixture
def lib(dev):
    from smart_crossover._native import lib as native
    return native


@pytest.fixture
def sort_path(request, lib):
    """sx_sort_set_tuning for one path of the table; both defaults (2, then 1) restored afterwards."""
    coop, threads = PATHS[request.param]
    try:
        assert lib.sx_sort_set_tuning(threads) == 0 and lib.sx_sort_set_tuning(coop) == 0
        yield request.param
    finally:
        assert lib.sx_sort_set_tuning(TUNING_THREADS_DEFAULT) == 0
        assert lib.sx_sort_set_tuning(TUNING_COOP_DEFAULT) == 0


def cu(a, dtype=None):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t.to(dtype) if dtype is not None else t).cuda()


def u32(t):
    return t.cpu().numpy().view(np.uint32).astype(np.int64)


def f64_bits(t):
    return t.cpu().numpy().view(np.uint64)


def check_sort(dev, key, ref, kref, key_t=None):
    """sx_argsort_f64 (order, sorted keys), sx_queue_from_order and, without NaN, sx_kruskal_order."""
    order, skey = dev.argsort_f64(cu(key) if key_t is None else key_t)
    got = u32(order)
    bad = np.flatnonzero(got != ref)
    assert bad.size == 0, f"order differs at {bad.size} positions, first {bad[:5]}: {got[bad[:5]]} vs {ref[bad[:5]]}"
    sb = sorted_bits_ref(key, ref)
    gb = f64_bits(skey)
    bad = np.flatnonzero(gb != sb)
    assert bad.size == 0, f"sorted keys differ at {bad.size} positions, first {bad[:5]}"
    assert np.array_equal(dev.queue_from_order(order).cpu().numpy(), ref[::-1])
    if kref is not None:
        assert np.array_equal(u32(dev.kruskal_order(skey, order)), kref)


SORT_KERNEL_RE = [
    ("small", re.compile(r"rs_small_sort_kernel")),
    ("coop", re.compile(r"rs_coop_sort_kernel<\s*(?:true|false|\d)\s*,\s*(\d+)\s*>|rs_coop_sort_kernelILb[01]ELi(\d+)E")),
    ("downsweep", re.compile(r"rs_downsweep_kernel<\s*(\d+)\s*,|rs_downsweep_kernelILi(\d+)E")),
]


def sort_kernels_run(fn):
    """{(path, threads)} of the radix-sort kernels launched by fn(), from a torch.profiler CUDA trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    seen = set()
    for e in prof.events():
        for kind, rx in SORT_KERNEL_RE:
            m = rx.search(e.name)
            if m:
                seen.add((kind, 1024 if kind == "small" else int(next(g for g in m.groups() if g))))
    return seen


# ==== 1. the sort at every path =============================================================================
def _sort_params():
    out = []
    for path, labels in SIZE_LABELS.items():
        for lab in labels:
            fams = BIG_FAMILIES if path == "default" else LARGE_FAMILIES if lab == "3grid*t-12345" else list(FAMILIES)
            out += [pytest.param(path, lab, f, id=f"{path}-{lab}-{f}") for f in fams]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("sort_path,label,family", _sort_params(), indirect=["sort_path"])
def test_argsort_every_path(dev, sort_path, label, family):
    n = path_size(sort_path, label)
    key, ref, kref = sort_case(family, n)
    check_sort(dev, key, ref, kref)


@pytest.mark.gpu
@pytest.mark.parametrize("sort_path,label", [
    ("small", "8192"), ("coop512", "8193"), ("coop512", "262144"), ("coop1024", "262145"), ("coop1024", "resident"),
    ("default", "resident+1"), ("ds256", "kt+1"), ("ds384", "kt+1"), ("ds512", "kt+1"), ("ds1024", "kt+1"),
    ("default", "2^26-1"), ("default", "2^26"),
], indirect=["sort_path"])
def test_path_is_the_intended_kernel(dev, sort_path, label):
    """The kernel each row of the path table names is the one that runs, and no other sort kernel does."""
    import torch
    coop, threads = PATHS[sort_path]
    n = {"resident+1": resident_limit() + 1, "2^26": BIG}.get(label) or path_size(sort_path, label)
    want = expected_path(n, coop, threads)
    key =torch.arange(n, 0, -1, device="cuda", dtype=torch.float64)          # reverse-sorted: easy to check
    got = sort_kernels_run(lambda: dev.argsort_f64(key))
    assert got == {want}, f"n = {n}: expected {want}, ran {got}"
    order, skey = dev.argsort_f64(key)
    assert torch.equal(order.to(torch.int64), torch.arange(n - 1, -1, -1, device="cuda"))


# ==== 2. sx_argsort_u64 =====================================================================================
U64_BITS = [1, 8, 9, 16, 17, 32, 33, 56, 63, 64]
U64_PATHS = {"small": "4097", "coop512": "100001", "coop1024": "500001", "ds256": "grid*t+1", "ds1024": "kt+1"}


def u64_case(n, key_bits):
    rng = np.random.default_rng(77 * n + key_bits)
    key = random_bits(rng, n)                                  # bits above the sorted range: random
    mask = u64_mask(key_bits)
    src, dst = rng.integers(0, n, n // 4), rng.integers(0, n, n // 4)
    key[dst] = (key[dst] & ~mask) | (key[src] & mask)          # ties in the sorted bits, different high bits
    key[::3] |= SIGN                                           # the top bit set
    return key, np.argsort(key & mask, kind="stable")


@pytest.mark.gpu
@pytest.mark.parametrize("key_bits", U64_BITS)
@pytest.mark.parametrize("sort_path", list(U64_PATHS), indirect=True)
def test_argsort_u64_key_bits(dev, lib, sort_path, key_bits):
    """Stable argsort of the key masked to the bits the code sorts; the sorted keys carry the unmasked key."""
    import torch
    from smart_crossover._native import check
    n = path_size(sort_path, U64_PATHS[sort_path])
    key, ref = u64_case(n, key_bits)
    kt = cu(key.view(np.int64))
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    skey = torch.empty(n, dtype=torch.int64, device="cuda")
    ws = torch.empty(lib.sx_argsort_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    check(lib.sx_argsort_u64(dev._ptr(kt), n, key_bits, dev._ptr(order), dev._ptr(skey), dev._ptr(ws), ws.numel(),
                             dev._stream()), "sx_argsort_u64")
    got = u32(order)
    bad = np.flatnonzero(got != ref)
    assert bad.size == 0, f"order differs at {bad.size} positions, first {bad[:5]}"
    assert np.array_equal(skey.cpu().numpy().view(np.uint64), key[ref])


# ==== 3. sx_kruskal_order and sx_kruskal_order_head ========================================================
ZERO = "zero"


def layout(name):
    """(run lengths, run values) of the ascending keys.  A value "zero" is a run of mixed -0.0 / +0.0."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "edges":                 # runs starting at 4095, 4096, 4097 of every block; runs of 4096 / 4097
        lens = [4095, 1, 1] + [4094, 1, 1] * 3 + [4096, 4097, 4096, 4097, 3]
    elif name == "block_aligned":       # runs starting and ending exactly on block boundaries
        lens = [4096, 4096, 8192, 4097, 4095, 1, 4096, 2]
    elif name == "long_run":            # one run across more than 1024 blocks: the carry scan walks 2 per thread
        lens = [3, 1, 1, 1025 * KO_TILE + 100, 2, 1]
    elif name == "zeros_infs":          # runs of -inf, of mixed-sign zeros and of +inf, across blocks
        return [3000, 5, 5000, 1, 4100], [-np.inf, -1.0, ZERO, 2.0 ** -1074, np.inf]
    elif name.startswith("n"):          # n = 1, 2, 4095, 4096, 4097 with random runs
        n = int(name[1:])
        lens = []
        while sum(lens) < n:
            lens.append(int(min(rng.geometric(0.05), n - sum(lens))))
    else:
        raise KeyError(name)
    vals = np.unique(rng.standard_normal(len(lens) + 8) * 1e3)[:len(lens)]
    return lens, list(vals)


def order_case(name):
    """(key, order_asc, sorted keys as the kernel reads them): key[order_asc] ascending, ids ascending in a run."""
    lens, vals = layout(name)
    rng = np.random.default_rng(len(lens))
    parts = []
    for ln, v in zip(lens, vals):
        if isinstance(v, str):
            parts.append(np.where(rng.random(ln) < 0.5, -0.0, 0.0))
        else:
            parts.append(np.full(ln, v, dtype=np.float64))
    asc_vals = np.concatenate(parts)
    n = asc_vals.size
    perm = rng.permutation(n)
    key = np.empty(n)
    key[perm] = asc_vals
    order = np.argsort(key, kind="stable")
    return key, order, key[order]


KO_LAYOUTS = ["n1", "n2", "n4095", "n4096", "n4097", "edges", "block_aligned", "long_run", "zeros_infs"]


def test_order_layouts_are_what_they_claim():
    key, order, skey = order_case("edges")
    heads = np.flatnonzero(np.r_[True, skey[1:] != skey[:-1]])
    assert {4095, 4096, 4097, 8191, 8192, 8193} <= set(heads.tolist())
    runs = np.diff(np.r_[heads, skey.size])
    assert {4096, 4097} <= set(runs.tolist())
    key, order, skey = order_case("block_aligned")
    heads = set(np.flatnonzero(np.r_[True, skey[1:] != skey[:-1]]).tolist())
    assert {4096, 8192, 16384} <= heads
    key, order, skey = order_case("long_run")
    runs = np.diff(np.r_[np.flatnonzero(np.r_[True, skey[1:] != skey[:-1]]), skey.size])
    assert runs.max() > 1024 * KO_TILE and -(-skey.size // KO_TILE) > 1024
    key, order, skey = order_case("zeros_infs")
    z = skey == 0
    assert np.signbit(skey[z]).any() and (~np.signbit(skey[z])).any()
    assert np.isneginf(skey).sum() == 3000 and np.isposinf(skey).sum() == 4100
    for nm in ("n1", "n2", "n4095", "n4096", "n4097"):
        assert order_case(nm)[0].size == int(nm[1:])
    # the head cuts start at every residue mod 4: ko_scatter_kernel's vector loads (start % 4 == 0) and scalar ones
    for nm in ("n4097", "edges"):
        skey = order_case(nm)[2]
        assert {(skey.size - m) % 4 for T, m in head_cases(skey)} == {0, 1, 2, 3}


@pytest.mark.gpu
@pytest.mark.parametrize("name", KO_LAYOUTS)
def test_kruskal_order_layouts(dev, name):
    """sx_kruskal_order on hand-built ascending keys == np.argsort(-key, kind="stable")."""
    key, order, skey = order_case(name)
    got = u32(dev.kruskal_order(cu(skey), cu(order.astype(np.uint32).view(np.int32))))
    ref = orc.kruskal_order(key)
    bad = np.flatnonzero(got != ref)
    assert bad.size == 0, f"{bad.size} positions differ, first {bad[:5]}: {got[bad[:5]]} vs {ref[bad[:5]]}"


def order_head(dev, lib, skey_t, order_t, T, T_cap):
    """sx_kruskal_order_head with T and T_cap passed as given (no clipping); None for -1."""
    import torch
    from smart_crossover._native import check
    n = order_t.numel()
    out = torch.full((T_cap,), -1, dtype=torch.int32, device="cuda")
    ws = torch.empty(lib.sx_kruskal_order_workspace_bytes(T_cap) + 256, dtype=torch.uint8, device="cuda")
    nh = ctypes.c_int64(0)
    check(lib.sx_kruskal_order_head(dev._ptr(skey_t), dev._ptr(order_t), n, T, T_cap, dev._ptr(out),
                                    ctypes.byref(nh), dev._ptr(ws), ws.numel(), dev._stream()), "sx_kruskal_order_head")
    return None if nh.value < 0 else u32(out[:nh.value])


def head_cases(skey):
    """(T, m): m = n - first position of the run holding position n - T.  Covers T = 1, n, n + 3 and, for every
    start % 4 (the vector load path needs start % 4 == 0: keys and ids 16-byte aligned), a cut inside a run."""
    n = skey.size
    heads = np.flatnonzero(np.r_[True, skey[1:] != skey[:-1]])
    ends = np.r_[heads[1:], n]
    cases = {(1, n - heads[-1]), (n, n), (n + 3, n)}
    for r in range(4):
        for h, e in zip(heads, ends):
            if h % 4 == r and h > 0:
                cases.add((n - (h + (e - h) // 2), n - h))        # n - T in the middle of the run at h
                break
    return sorted(cases)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n1", "n2", "n4097", "edges", "block_aligned", "zeros_infs", "long_run"])
def test_kruskal_order_head(dev, lib, name):
    """T = 1, n, n + 3 and cuts at every start % 4; T_cap = the covering run size succeeds, one less reports -1."""
    key, order, skey = order_case(name)
    ref = orc.kruskal_order(key)
    skey_t, order_t = cu(skey), cu(order.astype(np.uint32).view(np.int32))
    for T, m in head_cases(skey):
        got = order_head(dev, lib, skey_t, order_t, T, max(T, m))
        assert got is not None and got.size == m and np.array_equal(got, ref[:m]), (T, m)
        if m - 1 >= T:
            assert order_head(dev, lib, skey_t, order_t, T, m - 1) is None, (T, m)


# ==== 4. sx_kruskal_prefix and sx_hist12_f64 ===============================================================
PF_N = [60000, 60001]
PF_FAMILIES = list(FAMILIES)


@functools.lru_cache(maxsize=4)
def prefix_case(family, n):
    w = without_nan(make_keys(family, n), np.random.default_rng(n))
    img = sort_image(w)
    return w, np.sort(img >> np.uint64(40)), np.bincount((img >> np.uint64(52)).astype(np.int64), minlength=4096), \
        orc.kruskal_order(w)


def prefix_grid(n):
    """(T, T_cap) pairs: T in {1, small, n/2, n - 1, n, n + 5}, T_cap in {T, 4T, n} (T_cap >= T)."""
    out = []
    for T in (1, 100, n // 2, n - 1, n, n + 5):
        out += [(T, c) for c in sorted({T, 4 * T, n}) if c >= T]
    return out


def test_prefix_grid_takes_both_sides_of_the_crowded_fallback():
    """For every family, the grid hits both sides of the crowded-bin fallback (boundary bin holds more than
    4 T_cap arcs: two more passes over all weights) and of the -1 report."""
    for fam in PF_FAMILIES:
        w, asc24, hist, _ = prefix_case(fam, PF_N[0])
        crowded, fail = set(), set()
        for T, T_cap in prefix_grid(w.size):
            c, thr = prefix_count(asc24, T)
            crowded.add(T <= w.size and hist[thr >> 12] > PF_BND_FACTOR * T_cap)
            fail.add(c > T_cap)
        assert crowded == {False, True}, fam
        assert fail == {False, True} or fam == "full", fam           # distinct full-bit weights never tie


def kruskal_prefix(dev, lib, w_t, n, T, T_cap, hist_t=None):
    import torch
    from smart_crossover._native import check
    out = torch.full((T_cap,), -1, dtype=torch.int32, device="cuda")
    ws = torch.empty(lib.sx_kruskal_prefix_workspace_bytes(T_cap), dtype=torch.uint8, device="cuda")
    nh = ctypes.c_int64(0)
    check(lib.sx_kruskal_prefix(dev._ptr(w_t), n, T, T_cap, dev._ptr(hist_t), dev._ptr(out), ctypes.byref(nh),
                                dev._ptr(ws), ws.numel(), dev._stream()), "sx_kruskal_prefix")
    return None if nh.value < 0 else u32(out[:nh.value])


def device_weights(w, offset):
    """w on the device, at a 16-byte aligned address (offset 0) or 8 bytes past one (offset 1)."""
    import torch
    buf = torch.full((w.size + 1,), np.nan, dtype=torch.float64, device="cuda")
    view = buf[offset:offset + w.size]
    view.copy_(torch.from_numpy(w))
    assert view.data_ptr() % 16 == 8 * offset
    return view


def check_prefix(dev, lib, w, w_t, asc24, korder, T, T_cap, hist_t=None):
    n = w.size
    c, _ = prefix_count(asc24, T)
    got = kruskal_prefix(dev, lib, w_t, n, T, T_cap, hist_t)
    if c > T_cap:
        assert got is None, f"T={T} T_cap={T_cap}: {c} arcs at or above the threshold, expected -1"
        return None
    assert got is not None, f"T={T} T_cap={T_cap}: reported -1 for {c} arcs"
    assert min(T, n) <= got.size <= T_cap
    assert got.size == c, (T, T_cap, got.size, c)
    bad = np.flatnonzero(got != korder[:c])
    assert bad.size == 0, f"T={T} T_cap={T_cap}: {bad.size} positions differ, first {bad[:5]}"
    if c < n:                                           # nothing left out is heavier than the lightest arc kept
        assert w[korder[c]] < w[got[-1]]
    return got.size


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset8"])
@pytest.mark.parametrize("n", PF_N)
@pytest.mark.parametrize("family", PF_FAMILIES)
def test_kruskal_prefix_grid(dev, lib, family, n, offset):
    """Every (T, T_cap) of the grid, with and without a caller-supplied histogram."""
    w, asc24, hist, korder = prefix_case(family, n)
    w_t = device_weights(w, offset)
    hist_t = cu(hist.astype(np.uint32).view(np.int32))
    for T, T_cap in prefix_grid(n):
        a = check_prefix(dev, lib, w, w_t, asc24, korder, T, T_cap)
        b = check_prefix(dev, lib, w, w_t, asc24, korder, T, T_cap, hist_t)
        assert a == b


def dense_weights(n):
    """Full-bit finite weights: T = n / 2 puts about half of them above the threshold bin, more hits per CTA and
    load batch than a shared-memory stage of the split pass holds."""
    return without_nan(make_keys("full", n), np.random.default_rng(5))


def one_bin_weights(n):
    """Every weight in one level-0 bin: the boundary list is the whole input; T = 0.9 n makes the filter dense."""
    return 1.0 + np.random.default_rng(6).random(n)


def prefix_tie_weights(n, ties=20000):
    """`ties` weights with one 24-bit prefix that differ in the low 40 bits (and some exactly equal), a few above
    them and the rest below: the head is longer than T and must still be sorted exactly."""
    rng = np.random.default_rng(7)
    w = rng.random(n) * 0.5                                   # below
    pos = rng.choice(n, ties + 10, replace=False)
    base = np.float64(0.75).view(np.uint64) & np.uint64(0xFFFFFF0000000000)
    low = random_bits(rng, ties) & np.uint64(0x000000FFFFFFFFFF)
    low[3::4] = low[0::4]                                     # exact ties among them
    w[pos[:ties]] = as_f64(base | low)
    w[pos[ties:]] = 0.9 + rng.random(10) * 0.01               # above
    return w


PF_TAIL_CASES = {
    "dense_split": (lambda: dense_weights(300001), lambda n: n // 2, lambda n: n),
    "dense_filter": (lambda: one_bin_weights(300000), lambda n: (9 * n) // 10, lambda n: n),
    "prefix_ties": (lambda: prefix_tie_weights(200001), lambda n: 100, lambda n: 30000),
    "small_tail": (lambda: dense_weights(300001), lambda n: 1000, lambda n: 4000),
}


def test_prefix_tail_cases_are_what_they_claim():
    w = dense_weights(300001)
    img = sort_image(w)
    c, thr = prefix_count(np.sort(img >> np.uint64(40)), w.size // 2)
    above = int(((img >> np.uint64(52)) > np.uint64(thr >> 12)).sum())
    assert above > 0.45 * w.size and c > SMALL_MAX
    w = one_bin_weights(300000)
    assert np.unique(sort_image(w) >> np.uint64(52)).size == 1
    w = prefix_tie_weights(200001)
    asc24 = np.sort(sort_image(w) >> np.uint64(40))
    c, thr = prefix_count(asc24, 100)
    same = w[(sort_image(w) >> np.uint64(40)) == np.uint64(thr)]
    assert c >= 20000 and same.size >= 20000 and np.unique(same).size < same.size
    assert np.unique(same.view(np.uint64) & np.uint64(0xFFFFFFFFFF)).size > 10000


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PF_TAIL_CASES))
@pytest.mark.parametrize("sort_path", ["default", "ds256", "ds1024"], indirect=True)
def test_kruskal_prefix_tail_on_every_sort_path(dev, lib, sort_path, case):
    """Dense selections (stage overflow straight to global), a head of 20000 arcs tied on the 24-bit prefix, and
    the candidate tail's two sorts (u64 ids, then f64 weights) on the path its size and the tuning pick -- checked
    in a profiler trace."""
    make, Tf, Cf = PF_TAIL_CASES[case]
    w = make()
    n = w.size
    T, T_cap = Tf(n), Cf(n)
    img = sort_image(w)
    asc24 = np.sort(img >> np.uint64(40))
    korder = orc.kruskal_order(w)
    c, _ = prefix_count(asc24, T)
    w_t = cu(w)
    got = check_prefix(dev, lib, w, w_t, asc24, korder, T, T_cap)
    assert got == c
    coop, threads = PATHS[sort_path]
    want = expected_path(c, coop, threads)
    ran = sort_kernels_run(lambda: kruskal_prefix(dev, lib, w_t, n, T, T_cap))
    assert ran == {want}, f"{c} candidates: expected {want}, ran {ran}"


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["special", "full"])
@pytest.mark.parametrize("n,offset", [(1, 0), (2, 1), (7, 1), (100001, 0), (100001, 1), (100000, 1)])
def test_hist12_special_values(dev, lib, family, n, offset):
    """sx_hist12_f64 adds the 4096-bin histogram of the top 12 image bits to the caller's: -0.0 in +0.0's bin
    (2048), NaNs of both signs in bin 4095; odd n and an 8-byte offset pointer."""
    from smart_crossover._native import check
    key = make_keys(family, n)
    img = sort_image(key)
    ref = np.bincount((img >> np.uint64(52)).astype(np.int64), minlength=4096)
    rng = np.random.default_rng(n)
    pre = rng.integers(0, 1000, 4096).astype(np.uint32)
    hist_t = cu(pre.view(np.int32))
    w_t = device_weights(key, offset)
    check(lib.sx_hist12_f64(dev._ptr(w_t), n, dev._ptr(hist_t), dev._stream()), "sx_hist12_f64")
    got = hist_t.cpu().numpy().view(np.uint32).astype(np.int64)
    assert np.array_equal(got, pre.astype(np.int64) + ref)
    if n > 1000 and family == "special":
        zeros = int((key == 0).sum())
        assert zeros >= 2 and ref[2048] >= zeros and ref[4095] >= int(np.isnan(key).sum()) > 0
