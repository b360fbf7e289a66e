"""The one-launch proxy forward (dprt_proxy_infer: one mlp_kernel launch for every scene object of a stage) on row layouts
the test chooses, against per-object references.

The queries are installed through dprt_upload (BUF_NN_QUERY / BUF_NN_INPUT), bucketed with dprt_bucket_queries (which = 1)
and evaluated with dprt_proxy_infer. Each layout is a list of live rows per scene object. The networks differ from object
to object in depth (4 or 6 residual blocks), trunk width (256, or 128 embedded in the 256-wide kernel) and head (LeakyReLU
or Sigmoid), and some objects have no vis or no depth network. The largest layout is sized from the device's SM count so
that every CTA of the launch runs several work units and each of its units belongs to another object than the one before.

Checks:
  * bucketing: offsets, packed records and packed features equal a numpy stable partition bit for bit;
  * every object's rows equal, bit for bit, dprt_mlp_infer of that object's network on the same rows (the single-object
    launch, pinned to the reference module and the oracle by test_gpu_mlp.py): a row's arithmetic must not depend on the
    tile, slot or CTA that holds it;
  * every object's rows are within the stated tolerance of the network's PyTorch module in float64 (1e-3 for fp16
    operands, 4e-3 for bf16) and, for fp16 operands, of oracle.mlp_forward. Neighbouring networks are chosen so that their
    float64 outputs differ by more than 10x that tolerance on the layout's rows, so a swap of networks cannot pass;
  * rows of an object without a network stay exactly 0, and no half outside the prediction range is written.
The tests without the gpu mark check the references themselves (the numpy partition against the oracle's, the float64
modules against the oracle, and the separation of neighbouring networks) on the very layouts the GPU tests use.
"""
import ctypes
import functools
import zlib

import numpy as np
import pytest

from helpers import D, assert_bits_equal, assert_records_equal, dprt

WIDTH, HEIGHT, MC = 512, 512, 3               # MC * WIDTH * HEIGHT = 786 432 query slots for which = 1
TOL = {1: 1e-3, 0: 4e-3}                       # mlp_dtype 1 = fp16 operands, 0 = bf16 (tests/test_gpu_mlp.py)
SENTINEL = 0x7E5A                              # an fp16 NaN: never a prediction
B200_SMS = 148
TILE = 128

# name: (trunk width, residual blocks, Sigmoid head, torch seed)
CATALOGUE = {
    "4Res256": (256, 4, False, 11),
    "Sig4Res128": (128, 4, True, 15),
    "6Res256": (256, 6, False, 12),
    "Sig4Res256": (256, 4, True, 14),
    "4Res128": (128, 4, False, 13),
}
CYCLE = tuple(CATALOGUE)                       # objects take the networks in this order

# Objects without a network for a kind. At S = 32 every object has a vis network (all 32 slots of the vis table hold one).
MISSING = {8: {0: (4, 6), 1: (2, 6)}, 32: {0: (), 1: (2, 15, 31)}}


def networks(S, kind):
    """Network name (or None) of every scene object for one kind: 0 = vis, 1 = depth."""
    shift = 0 if kind == 0 else 2
    return [None if i in MISSING[S][kind] else CYCLE[(i + shift) % len(CYCLE)] for i in range(S)]


# ---- networks and their references ---------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _module(name):
    import torch
    width, nres, sig, seed = CATALOGUE[name]
    torch.manual_seed(seed)
    return dprt.proxy.make_proxy(width, nres, sigmoid=sig).eval()


@functools.lru_cache(maxsize=None)
def blob(name):
    return dprt.proxy.pack_module(_module(name))


@functools.lru_cache(maxsize=None)
def feature_pool():
    """fp16 feature rows in [0, 1]: the 32 corners of the unit cube (both ends of every feature), then uniform rows.
    Every query slot takes one pool row, so the references are evaluated once per network."""
    corners = ((np.arange(32)[:, None] >> np.arange(5)) & 1).astype(np.float16)
    rest = np.random.default_rng(20241016).random((4096 - 32, 5)).astype(np.float16)
    return np.concatenate([corners, rest]).view(np.uint16)


@functools.lru_cache(maxsize=None)
def reference64(name):
    """The network's PyTorch module in float64 on the pool's fp16 features."""
    import copy

    import torch
    m = copy.deepcopy(_module(name)).double()
    x = torch.from_numpy(feature_pool().view(np.float16).astype(np.float64))
    with torch.no_grad():
        return m(x).numpy()[:, 0]


@functools.lru_cache(maxsize=None)
def reference_oracle(name):
    from oracle import oracle as O
    return O.mlp_forward(blob(name), feature_pool())[0]


# ---- layouts ---------------------------------------------------------------------------------------------------------
def _both_models(S):
    return [i for i in range(S) if networks(S, 0)[i] and networks(S, 1)[i]]


def _large(S, sms):
    """About 5 x sms tile pairs spread over all objects, none with more than sms pairs, tile counts odd and even."""
    per = 5 * sms * 2 * TILE // S
    return [per + (i % 3) * TILE - (i % 2) * (TILE - 1) + 7 * i for i in range(S)]


def layout(name, S, sms=B200_SMS):
    c = [0] * S
    if name == "one_object":
        c[_both_models(S)[len(_both_models(S)) // 2]] = 4999
    elif name == "empty_first_middle_last":
        c = [0 if i in (0, S // 2, S - 1) else 64 + (97 * i) % 400 for i in range(S)]
    elif name == "ragged":
        sizes = (1, 129, 127, 255, 257, 256, 383, 128)       # tiles 1 2 1 2 3 2 3 1
        c = [sizes[(i + i // len(sizes)) % len(sizes)] for i in range(S)]
    elif name == "modelless_between":
        for kind in (0, 1):
            for k in MISSING[S][kind]:
                if 0 < k < S - 1:
                    c[k - 1], c[k], c[k + 1] = 300, 200 + 57 * k, 129
    elif name == "modelless_only":           # an object without any network if there is one, else one without a depth network
        missing = [i for i in range(S) if networks(S, 0)[i] is None or networks(S, 1)[i] is None]
        c[min(missing, key=lambda i: (networks(S, 0)[i] is not None) + (networks(S, 1)[i] is not None))] = 1000
    elif name == "large":
        c = _large(S, sms)
    elif name == "no_live_rows":
        pass
    else:
        raise KeyError(name)
    return c


LAYOUTS = ("one_object", "empty_first_middle_last", "ragged", "modelless_between", "modelless_only", "large", "no_live_rows")
SCENE_SIZES = (8, 32)


def make_queries(counts, S, inside_only, seed):
    """Query slots for which = 1: the live records (hitAABBID = object + 1; isInside = 1 when inside_only) interleaved with
    records bucketing must drop (hitAABBID 0, negative or > S; for inside_only also valid ids with isInside = 0).
    Returns (records, pool row of every slot, pathSize); pixelIndex = slot index."""
    rng = np.random.default_rng(seed)
    live = np.repeat(np.arange(1, S + 1, dtype=np.int64), counts)
    n_noise = max(97, live.size // 4)
    bad_ids = np.array([0, -1, S + 1, S + 2, 127, 128, 255, 1000, 2 ** 31 - 1, -2 ** 31], np.int64)
    noise = rng.choice(bad_ids, n_noise)
    inside = np.concatenate([np.ones(live.size, np.uint8) if inside_only else rng.integers(0, 2, live.size).astype(np.uint8),
                             rng.integers(0, 2, n_noise).astype(np.uint8)])
    ids = np.concatenate([live, noise])
    if inside_only:                                   # valid objects, but not inside the proxy AABB
        outside = rng.integers(1, S + 1, n_noise // 2)
        ids = np.concatenate([ids, outside]); inside = np.concatenate([inside, np.zeros(outside.size, np.uint8)])
    path_size = -(-ids.size // MC)
    n = MC * path_size
    ids = np.concatenate([ids, np.zeros(n - ids.size, np.int64)]); inside = np.concatenate([inside, np.zeros(n - inside.size, np.uint8)])
    perm = rng.permutation(n)
    ids, inside = ids[perm], inside[perm]
    q = np.frombuffer(rng.integers(0, 256, n * D.QUERY_DTYPE.itemsize, dtype=np.uint8).tobytes(), D.QUERY_DTYPE).copy()
    q["throughput"] = rng.random((n, 3)).astype(np.float32)
    q["normalizedT"] = rng.random(n).astype(np.float32)
    q["pixelIndex"] = np.arange(n)
    q["hitAABBID"] = ids.astype(np.int32)
    q["isInside"] = inside
    pool_row = rng.integers(0, feature_pool().shape[0], n)
    return q, pool_row, path_size


def stable_partition(q, S, inside_only):
    """Bucket-major, original order inside a bucket, dead entries dropped: (offsets [S + 1], slot of every packed row)."""
    ids = q["hitAABBID"].astype(np.int64)
    keep = (ids >= 1) & (ids <= S)
    if inside_only:
        keep &= q["isInside"] != 0
    slots = np.nonzero(keep)[0]
    slots = slots[np.argsort(ids[slots], kind="stable")]
    offsets = np.concatenate([[0], np.cumsum(np.bincount(ids[slots] - 1, minlength=S))]).astype(np.int32)
    return offsets, slots


def case(name, S, inside_only, sms=B200_SMS):
    counts = layout(name, S, sms)
    q, pool_row, path_size = make_queries(counts, S, inside_only, zlib.crc32(f"{name}/{S}/{inside_only}".encode()))
    offsets, slots = stable_partition(q, S, inside_only)
    assert np.array_equal(np.diff(offsets), counts)
    return counts, q, pool_row, path_size, offsets, slots


def tile_pairs(counts, nets):
    return [(-(-c // TILE) + 1) // 2 if (c > 0 and net) else 0 for c, net in zip(counts, nets)]


def cta_units(pairs, sms):
    """Object of every work unit each CTA runs: mlp_kernel walks u = blockIdx.x, u + gridDim.x, ... over the tile pairs."""
    obj = np.repeat(np.arange(len(pairs)), pairs)
    grid = min(len(obj), sms)
    return [obj[b::grid] for b in range(grid)]


def neighbour_separation(counts, nets, offsets, slots, pool_row):
    """For consecutive objects (in row order) that both have rows and a network: the largest difference between their
    float64 references over the two objects' rows. Returns [(object a, object b, difference)]."""
    live = [i for i in range(len(counts)) if counts[i] > 0 and nets[i]]
    out = []
    for a, b in zip(live, live[1:]):
        rows = pool_row[np.concatenate([slots[offsets[a]:offsets[a + 1]], slots[offsets[b]:offsets[b + 1]]])]
        out.append((a, b, float(np.abs(reference64(nets[a])[rows] - reference64(nets[b])[rows]).max())))
    return out


# ---- checks that need no GPU -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", SCENE_SIZES)
def test_layouts_cover_the_edges(S):
    assert any(networks(S, 0)[i] is None for i in range(S)) or S == 32
    assert any(networks(S, 1)[i] is None for i in range(S))
    if S == 32:
        assert all(networks(S, 0))                                 # every slot of the vis table holds a network
    for kind in (0, 1):
        pairs = [(CATALOGUE[a], CATALOGUE[b]) for a, b in zip(networks(S, kind), networks(S, kind)[1:]) if a and b]
        assert all(a != b for a, b in pairs)
        for field in range(3):                                     # width, residual blocks, head
            assert any(a[field] != b[field] for a, b in pairs)
    e = layout("empty_first_middle_last", S)
    assert e[0] == 0 and e[S // 2] == 0 and e[-1] == 0 and sum(e) > 0
    assert set(layout("ragged", S)) == {1, 127, 128, 129, 255, 256, 257, 383}
    for kind in (0, 1):
        nets, c = networks(S, kind), layout("modelless_between", S)
        assert not MISSING[S][kind] or any(nets[k] is None and nets[k - 1] and nets[k + 1] and min(c[k - 1:k + 2]) > 0
                                           for k in range(1, S - 1))
    assert sum(layout("no_live_rows", S)) == 0
    for name in LAYOUTS:
        for inside_only in (0, 1):
            assert case(name, S, inside_only)[3] <= WIDTH * HEIGHT      # pathSize: MC * pathSize slots fit the query buffers


@pytest.mark.parametrize("S", SCENE_SIZES)
def test_large_layout_crosses_objects_in_every_cta(S):
    check_large_layout(S, B200_SMS)


def check_large_layout(S, sms):
    counts = layout("large", S, sms)
    assert any((-(-c // TILE)) % 2 for c in counts) and any((-(-c // TILE)) % 2 == 0 for c in counts)
    for kind in (0, 1):
        pairs = tile_pairs(counts, networks(S, kind))
        assert sum(pairs) >= 3 * sms
        for units in cta_units(pairs, sms):
            assert units.size >= 3
            assert np.all(units[1:] != units[:-1])       # every unit after the first belongs to another object


@pytest.mark.parametrize("S", SCENE_SIZES)
@pytest.mark.parametrize("inside_only", [0, 1])
def test_numpy_partition_matches_oracle(oracle, S, inside_only):
    cfg = dprt.make_config(WIDTH, HEIGHT, mc=MC, scene_size=S, proxy_mode=1)
    world = oracle.World(cfg, 2)
    x = feature_pool()
    for name in ("ragged", "modelless_between", "large", "no_live_rows"):
        counts, q, pool_row, path_size, offsets, slots = case(name, S, inside_only)
        world.set_path_size(0, path_size)
        world.upload(0, D.BUF_NN_QUERY, q)
        world.upload(0, D.BUF_NN_INPUT, x[pool_row].reshape(-1))
        total = world.bucket_queries(0, 1, inside_only)
        assert total == slots.size == offsets[-1]
        assert_bits_equal(world.download(0, D.BUF_SCENE_OFFSET, S + 1), offsets, f"{name}: offsets")
        assert_records_equal(world.download(0, D.BUF_NN_PACKED_QUERY, total), q[slots], f"{name}: packed queries")
        assert_bits_equal(world.download(0, D.BUF_NN_PACKED_INPUT, 5 * total), x[pool_row[slots]].reshape(-1), f"{name}: packed features")
    world.close()


@pytest.mark.parametrize("name", CYCLE)
def test_float64_references_match_oracle(oracle, name):
    assert np.abs(reference64(name) - reference_oracle(name)).max() <= 1e-3


@pytest.mark.parametrize("S", SCENE_SIZES)
@pytest.mark.parametrize("mlp_dtype", [1, 0])
def test_neighbouring_networks_are_told_apart(S, mlp_dtype):
    for name in LAYOUTS:
        for inside_only in (0, 1):
            counts, q, pool_row, path_size, offsets, slots = case(name, S, inside_only)
            for kind in (0, 1):
                for a, b, d in neighbour_separation(counts, networks(S, kind), offsets, slots, pool_row):
                    assert d > 10 * TOL[mlp_dtype], (name, inside_only, kind, a, b, d)


# ---- the grouped forward on the GPU ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def contexts(gpu_required):
    made = {}

    def get(S, mlp_dtype):
        if (S, mlp_dtype) not in made:
            cfg = dprt.make_config(WIDTH, HEIGHT, mc=MC, scene_size=S, proxy_mode=1, mlp_dtype=mlp_dtype)
            R = dprt.Renderer(cfg, rank=0, world=2)
            for i in range(S):
                vis, dep = networks(S, 0)[i], networks(S, 1)[i]
                R.upload_proxy(i, dprt.make_object_desc(1, [0, 0, 0], [1, 1, 1], is_proxy=1),
                               blob(vis) if vis else None, blob(dep) if dep else None)
            made[(S, mlp_dtype)] = R
        return made[(S, mlp_dtype)]

    yield get
    for R in made.values():
        R.close()


def _buffer_count(R, buf):
    nbytes = ctypes.c_size_t()
    assert R.lib.dprt_buffer_bytes(R.h, buf, ctypes.byref(nbytes)) == 0
    return nbytes.value // D.BUFFER_DTYPES[buf].itemsize


def _fill_pred(R, size):
    R.upload(D.BUF_PRED, np.full(size, SENTINEL, np.uint16))


def _check_outside(pred, off, total, what):
    outside = np.ones(pred.size, bool)
    outside[off:off + total] = False
    bad = np.nonzero(pred[outside] != SENTINEL)[0]
    assert bad.size == 0, f"{what}: {bad.size} halves outside [{off}, {off + total}) were written"


@pytest.mark.gpu
@pytest.mark.parametrize("inside_only", [0, 1])
@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("S,mlp_dtype", [(8, 1), (8, 0), (32, 1), (32, 0)])
def test_grouped_forward_matches_per_object_references(contexts, oracle, S, mlp_dtype, name, inside_only):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if name == "large":
        check_large_layout(S, sms)
    R = contexts(S, mlp_dtype)
    counts, q, pool_row, path_size, offsets, slots = case(name, S, inside_only, sms)
    x = feature_pool()[pool_row].reshape(-1)
    n = MC * path_size
    assert n <= _buffer_count(R, D.BUF_NN_QUERY) and 5 * n <= _buffer_count(R, D.BUF_NN_INPUT)
    size = _buffer_count(R, D.BUF_PRED)

    # bucketing
    R.set_path_size(path_size)
    R.upload(D.BUF_NN_QUERY, q)
    R.upload(D.BUF_NN_INPUT, x)
    total = R.bucket_queries(1, inside_only)
    assert total == slots.size == offsets[-1]
    assert_bits_equal(R.download(D.BUF_SCENE_OFFSET, S + 1), offsets, "offsets")
    assert_records_equal(R.download(D.BUF_NN_PACKED_QUERY, total), q[slots], "packed queries")
    packed_x = R.download(D.BUF_NN_PACKED_INPUT, 5 * total)
    assert_bits_equal(packed_x, x.reshape(-1, 5)[slots].reshape(-1), "packed features")
    assert_records_equal(R.download(D.BUF_NN_QUERY, n), q, "queries after bucketing")
    assert_bits_equal(R.download(D.BUF_NN_INPUT, 5 * n), x, "features after bucketing")
    packed_x = packed_x.reshape(-1, 5)

    tol = TOL[mlp_dtype]
    expected = {}
    for kind in (0, 1):
        nets = networks(S, kind)
        rows_with_model = sum(c for c, net in zip(counts, nets) if net)
        for a, b, d in neighbour_separation(counts, nets, offsets, slots, pool_row):
            assert d > 10 * tol, f"kind {kind}: objects {a} and {b} are not told apart on this layout ({d:.2e})"
        # what every object's rows must be: the single-object launch on the same rows, bit for bit
        expect = expected[kind] = np.zeros(total, np.uint16)
        for i in range(S):
            a, b = offsets[i], offsets[i + 1]
            if b > a and nets[i]:
                expect[a:b] = R.mlp_infer(i, kind, packed_x[a:b])
        for off in (0, total):
            what = f"kind {kind} pred_offset {off}"
            _fill_pred(R, size)
            s0 = R.stats()
            R.proxy_infer(kind, off)
            s1 = R.stats()
            assert s1["kernel_launches"] - s0["kernel_launches"] == (1 if rows_with_model else 0), what
            assert s1["nn_queries"] - s0["nn_queries"] == rows_with_model, what
            pred = R.download(D.BUF_PRED)
            _check_outside(pred, off, total, what)
            y = pred[off:off + total]
            failed = []                    # every failing check of every object, so that a report shows which checks see a fault
            for i in range(S):
                a, b = offsets[i], offsets[i + 1]
                if b == a:
                    continue
                if nets[i] is None:
                    if y[a:b].any():
                        failed.append(f"object {i} has no network: {np.count_nonzero(y[a:b])}/{b - a} rows are not 0")
                    continue
                diff = np.count_nonzero(y[a:b] != expect[a:b])
                if diff:
                    failed.append(f"object {i} ({nets[i]}): {diff}/{b - a} rows differ from its single-object launch")
                yf = y[a:b].view(np.float16).astype(np.float64)
                rows = pool_row[slots[a:b]]
                refs = [("float64 module", reference64(nets[i]))] + ([("oracle", reference_oracle(nets[i]))] if mlp_dtype == 1 else [])
                for ref_name, ref in refs:
                    err = np.abs(yf - ref[rows])
                    if not err.max() <= tol:
                        failed.append(f"object {i} ({nets[i]}): max |gpu - {ref_name}| = {err.max():.2e} "
                                      f"({np.count_nonzero(~(err <= tol))}/{b - a} rows above {tol})")
            assert not failed, f"{what}:\n  " + "\n  ".join(failed)
            # the same layout again: the same bits
            R.proxy_infer(kind, off)
            assert_bits_equal(R.download(D.BUF_PRED, total, offset=off), y, f"{what}: second launch")

    # a prediction range outside BUF_PRED is rejected before anything is written
    _fill_pred(R, size)
    for bad in (-1, size - total + 1):
        with pytest.raises(dprt.DprtError):
            R.proxy_infer(0, bad)
    assert not np.any(R.download(D.BUF_PRED) != SENTINEL), "a rejected call wrote BUF_PRED"
    # the range may end exactly at the end of the buffer
    R.proxy_infer(0, size - total)
    pred = R.download(D.BUF_PRED)
    _check_outside(pred, size - total, total, "range at the end of BUF_PRED")
    assert_bits_equal(pred[size - total:], expected[0], "range at the end of BUF_PRED")
