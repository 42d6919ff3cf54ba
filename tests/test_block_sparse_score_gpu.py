"""GPU: block-sparse FP4 cover scoring.  Candidates and columns reordered, all-zero K blocks skipped; the gains must be
bit-identical to the dense natural-order scorer and to the popcount scorer, and the reordered planes must equal a column
gather of the natural planes, also after bmf_cover_apply_f4_mapped has patched them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from oracle import asso_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def nat():
    from pybmf_b200 import _native, device
    _native.require_gpu()
    return _native, device


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def order_reference(B, cand_pad, ld4):
    """numpy restatement of engine.block_sparse_order: (pi, col_pos, cum, lists)."""
    n = B.shape[0]
    pop = B.sum(axis=1)
    minc = np.where(pop > 0, B.argmax(axis=1), n)
    group = np.where(pop >= 2, 0, np.where(pop == 1, 1, 2))
    pi = np.lexsort((np.arange(n), minc, group))
    pos = np.empty(n, np.int64)
    pos[pi] = np.arange(n)
    first = np.full(n, np.iinfo(np.int32).max, np.int64)
    rows, cols = np.nonzero(B)
    np.minimum.at(first, cols, pos[rows])
    sigma = np.lexsort((np.arange(n), first))
    col_pos = np.empty(n, np.int64)
    col_pos[sigma] = np.arange(n)
    P = np.zeros((cand_pad, 2 * ld4), bool)
    P[:n, :n] = B[pi][:, sigma].astype(bool)
    mt, kb = cand_pad // 256, 2 * ld4 // 256
    nz = P.reshape(mt, 256, kb, 256).any(axis=(1, 3))
    lists = np.argsort(~nz, axis=1, kind="stable")
    cum = np.concatenate([[0], np.cumsum(nz.sum(axis=1))])
    return pi, col_pos, cum, lists


def planted_basis(rng, n, groups, width, extra=0.0):
    """Basis rows: `groups` planted column groups shared by the candidates of each group, the rest single-column."""
    B = np.zeros((n, n), np.uint8)
    B[np.arange(n), np.arange(n)] = 1
    for g in range(groups):
        cols = rng.choice(n, size=width, replace=False)
        members = rng.choice(n, size=max(2, width // 4), replace=False)
        B[np.ix_(members, cols)] = 1
    if extra:
        B |= (rng.rand(n, n) < extra).astype(np.uint8)
    return B


def _basis_cases():
    rng = np.random.RandomState(11)
    n = 1500
    empty_tiles = planted_basis(rng, n, 6, 40)
    empty_tiles[600:1200] = 0                                   # zero rows: whole candidate tiles without any block
    return {"planted": planted_basis(rng, n, 8, 60),
            "dense": (rng.rand(700, 700) < 0.3).astype(np.uint8),
            "singletons": np.eye(1300, dtype=np.uint8),
            "empty_tiles": empty_tiles}


BASES = _basis_cases()


def _build(device, B):
    from pybmf_b200 import engine
    n = B.shape[0]
    words = device.words_for(n)
    cand_pad, ld4 = device.round_up(n, 256), device.round_up(n, 256) // 2
    b_d = _dev(device.dense_to_words(B))
    pop = np.zeros(cand_pad, np.int32)
    pop[:n] = B.sum(axis=1)
    plane = device.empty((cand_pad, ld4), torch.uint8)
    cand_id, col_pos, table = engine.block_sparse_order(b_d, _dev(pop), n, words, cand_pad, ld4, plane)
    return b_d, pop, plane, cand_id, col_pos, table, words, cand_pad, ld4


@pytest.mark.parametrize("case", sorted(BASES))
def test_order_and_table_match_numpy(nat, case):
    _native, device = nat
    B = BASES[case]
    n = B.shape[0]
    _b, _p, plane, cand_id, col_pos, table, _w, cand_pad, ld4 = _build(device, B)
    pi, cpos, cum, lists = order_reference(B, cand_pad, ld4)
    mt, kb = cand_pad // 256, ld4 // 128
    assert np.array_equal(cand_id.cpu().numpy()[:n], pi)
    assert np.array_equal(cand_id.cpu().numpy()[n:], np.arange(n, cand_pad))
    assert np.array_equal(col_pos.cpu().numpy(), cpos)
    t = table.cpu().numpy()
    assert np.array_equal(t[:mt + 1], cum)
    got_lists = t[mt + 1:].reshape(mt, kb)
    for m in range(mt):
        assert np.array_equal(got_lists[m, :cum[m + 1] - cum[m]], lists[m, :cum[m + 1] - cum[m]])
    # the candidate plane is the natural plane gathered by (pi, sigma)
    nat_plane = device.empty((cand_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4", _b, None, n, n, _w, 2, 0, 0, nat_plane, cand_pad, ld4)
    assert torch.equal(_unpack(plane)[:n, :n], _unpack(nat_plane)[:n][pi][:, np.argsort(cpos)])
    assert not _unpack(plane)[n:].any()
    if case == "dense":
        assert cum[-1] == mt * kb
    if case == "empty_tiles":
        assert (np.diff(cum) == 0).any()


def _unpack(plane):
    p = plane.cpu().numpy()
    out = np.empty((p.shape[0], 2 * p.shape[1]), np.uint8)
    out[:, 0::2], out[:, 1::2] = p & 15, p >> 4
    return torch.from_numpy(out)


@pytest.mark.parametrize("case", sorted(BASES))
def test_block_sparse_gains_bit_identical(nat, case):
    _native, device = nat
    from pybmf_b200 import engine
    B = BASES[case]
    n = B.shape[0]
    m = 3000
    rng = np.random.RandomState(n)
    X = (rng.rand(m, n) < 0.05).astype(np.uint8)
    C = (X & (rng.rand(m, n) < 0.3)).astype(np.uint8)
    wa, wb = 1, 1
    lib = _native.load()
    c_one, c_cov = lib.bmf_e2m1_code(wa + wb), lib.bmf_e2m1_code(wa)
    b_d, pop, cplane, cand_id, col_pos, table, words, cand_pad, ld4 = _build(device, B)
    rows_pad = device.round_up(m, engine.F4_ROW_PAD)
    x_d, c_d = _dev(device.dense_to_words(X)), _dev(device.dense_to_words(C))
    rplane = device.empty((rows_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4_mapped", x_d, c_d, m, n, words, c_one, 0, c_cov, None, col_pos, rplane, rows_pad, ld4)
    nat_r = device.empty((rows_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4", x_d, c_d, m, n, words, c_one, 0, c_cov, nat_r, rows_pad, ld4)
    inv = np.argsort(col_pos.cpu().numpy())
    assert torch.equal(_unpack(rplane)[:, :n], _unpack(nat_r)[:, :n][:, inv])
    nat_c = device.empty((cand_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4", b_d, None, n, n, words, 2, 0, 0, nat_c, cand_pad, ld4)
    pop_d = _dev(pop)
    dense = device.zeros((cand_pad,), torch.int64)
    _native.call("bmf_cover_score_f4", nat_c, cand_pad, nat_r, rows_pad, ld4, pop_d, wa, dense)
    sparse = device.zeros((cand_pad,), torch.int64) + 7
    _native.call("bmf_cover_score_f4_blocks", cplane, cand_pad, rplane, rows_pad, ld4, pop_d, wa, table, cand_id, sparse)
    tp, fp, _ = O.confusion(X, C, axis=1)
    popc = device.zeros((cand_pad,), torch.int64)
    _native.call("bmf_cover_score_popc", x_d, c_d, m, n, words, b_d, _dev(np.ones(n, np.uint8)),
                 _dev(tp.astype(np.int32)), _dev(fp.astype(np.int32)), wa, wb, 0.5, 0.5, popc, None)
    assert torch.equal(sparse, dense)
    assert torch.equal(sparse[:n], popc[:n])
    assert np.array_equal(sparse.cpu().numpy()[:n], O.integer_gains(X, C, B, wa, wb))

    # apply a winner with the mapped patch: the plane equals a fresh mapped expansion of the new cover
    j = int(np.argmax(sparse.cpu().numpy()[:n]))
    alive = _dev(np.ones(n, np.uint8))
    tpo, fpo = _dev(tp.astype(np.int32)), _dev(fp.astype(np.int32))
    ub = device.zeros((device.words_for(m),), torch.int64)
    tot = device.zeros((3,), torch.int64)
    _native.call("bmf_cover_apply_f4_mapped", x_d, c_d, m, n, words, b_d, alive, _dev(np.array([j], np.int64)), tpo, fpo,
                 wa, wb, rplane, ld4, c_cov, col_pos, ub, tot)
    fresh = device.empty((rows_pad, ld4), torch.uint8)
    _native.call("bmf_expand_bits_f4_mapped", x_d, c_d, m, n, words, c_one, 0, c_cov, None, col_pos, fresh, rows_pad, ld4)
    assert torch.equal(fresh, rplane)

    # incremental re-score of the next winner over mapped compact rows == a full pass on the updated planes
    full_before = device.zeros((cand_pad,), torch.int64)
    _native.call("bmf_cover_score_f4_blocks", cplane, cand_pad, rplane, rows_pad, ld4, pop_d, wa, table, cand_id,
                 full_before)
    j2 = int(np.argmax(np.where(np.arange(n) == j, -1, full_before.cpu().numpy()[:n])))
    comp_old = device.empty((rows_pad, ld4), torch.uint8)
    comp_new = device.empty((rows_pad, ld4), torch.uint8)
    nused = device.zeros((2,), torch.int32)
    ub2 = device.zeros((device.words_for(m),), torch.int64)
    tot2 = device.zeros((3,), torch.int64)
    _native.call("bmf_cover_apply_compact_mapped", x_d, c_d, m, n, words, b_d, alive, _dev(np.array([j2], np.int64)),
                 tpo, fpo, wa, wb, 1, c_one, 0, c_cov, comp_old, comp_new, ld4, rows_pad, engine.F4_ROW_PAD, nused, ub2,
                 None, 0, 0, None, col_pos, tot2)
    inc = full_before.clone()
    for plane, sign in ((comp_old, -1), (comp_new, 1)):
        _native.call("bmf_cover_rescore_f4_blocks", cplane, cand_pad, plane, rows_pad, ld4, pop_d, wa, table, cand_id,
                     nused, sign, inc)
    _native.call("bmf_expand_bits_f4_mapped", x_d, c_d, m, n, words, c_one, 0, c_cov, None, col_pos, fresh, rows_pad, ld4)
    full_after = device.zeros((cand_pad,), torch.int64)
    _native.call("bmf_cover_score_f4_blocks", cplane, cand_pad, fresh, rows_pad, ld4, pop_d, wa, table, cand_id, full_after)
    assert torch.equal(inc, full_after)


def test_c4_table(nat):
    """At the c4 workload's basis (tau = 0.5) the reorder leaves 1009 of 4900 candidate blocks nonzero."""
    _native, device = nat
    from pybmf_b200 import synth
    from pybmf_b200.engine import CoverEngine
    X = synth.config_c4()
    eng = CoverEngine(X, 0.5, 0.5, scorer="tcgen05", rescore="full")
    eng.build_basis(0.5)
    assert eng.kb_table is not None
    n = eng.n
    B = device.bits_to_host(eng.basis_bits, n)
    pi, cpos, cum, lists = order_reference(B, eng.cand_pad, eng.ld4)
    t = eng.kb_table.cpu().numpy()
    mt = eng.cand_pad // 256
    assert np.array_equal(t[:mt + 1], cum) and cum[-1] == 1009
    assert np.array_equal(eng.cand_id.cpu().numpy()[:n], pi)
    assert np.array_equal(eng.col_pos.cpu().numpy(), cpos)
