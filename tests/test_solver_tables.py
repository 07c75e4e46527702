"""CPU: the solver distance tables (SURVEY 8f row 3). The oracle restatement against the fixture written by the
reference's own InterPieceDistance class (tests/golden/make_golden_tables.py), the host-side pieces of
vited_b200.solver_tables, the object install() builds against the constructor state stored in that fixture, and --
where VITED_REFERENCE names a checkout of the reference project -- the prebuilt object against the reference's own
constructor and dropped into the reference's solver against the solver run with its own callbacks."""
import enum
import os
import sys

import numpy as np
import pytest

from tests.conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import make_golden_tables as mg  # noqa: E402

REF = os.environ.get('VITED_REFERENCE', '')
KEYS = ['asym_dist', 'asym_compat', 'mutual_compat', 'min_dist', 'second_dist', 'candidates', 'best_buddy',
        'start_order', 'start_compat']


def _cases():
    z = np.load(os.path.join(GOLDEN, 'solver_tables.npz'))
    return z, [tuple(int(v) for v in c) for c in z['cases']]


def test_fixture_generator_cases_match_fixture():
    z, cases = _cases()
    assert cases == [tuple(c) for c in mg.CASES]


RULES = {'numpy1': '_np1', 'numpy2': ''}   # scalar rules -> fixture key infix (see make_golden_tables.py)


@pytest.mark.parametrize('rules', sorted(RULES))
@pytest.mark.parametrize('case', mg.CASES, ids=lambda c: f'seed{c[0]}_{c[1]}x{c[2]}')
def test_oracle_tables_match_reference_fixture(case, rules):
    from oracle import vited_oracle as orc
    z, _ = _cases()
    d, order = mg.case_inputs(*case)
    got = orc.solver_tables(d, order, scalar_rules=rules)
    for k in KEYS:
        ref = z[f'{k}{RULES[rules]}_{case[0]}']
        assert got[k].dtype == ref.dtype and got[k].shape == ref.shape, k
        assert np.array_equal(got[k], ref), k          # bit-exact: integers, and floats produced by the same operations


def test_scalar_rules_differ_where_the_fixture_says():
    """float32(0.02 k) * 1000: 19.99.. in float64 (NumPy 1.x, the reference's pinned stack), 20.0 in float32."""
    case = mg.CASES[4]
    z, _ = _cases()
    a, b = z[f'asym_dist_np1_{case[0]}'], z[f'asym_dist_{case[0]}']
    assert (a != b).sum() > 100 and np.abs(a.astype(np.int64) - b.astype(np.int64)).max() == 1


@pytest.mark.parametrize('case', mg.CASES, ids=lambda c: f'seed{c[0]}_{c[1]}x{c[2]}')
def test_start_piece_ordering_host(case):
    from vited_b200 import solver_tables
    z, _ = _cases()
    seed = case[0]
    got = solver_tables.start_piece_ordering(z[f'best_buddy_{seed}'], z[f'mutual_compat_{seed}'])
    assert [(a, b) for (a, b, _) in got] == [tuple(r) for r in z[f'start_order_{seed}'].tolist()]
    assert np.array_equal(np.array([float(c) for (_, _, c) in got]), z[f'start_compat_{seed}'])


def _tables_from_oracle(d, order, rules='numpy2'):
    """(the reference-run comparisons below execute the reference under THIS container's NumPy >= 2)"""
    from oracle import vited_oracle as orc
    from vited_b200 import solver_tables
    t = orc.solver_tables(d, order, scalar_rules=rules)
    n = len(order)
    n_cand = t['candidates'].sum(-1).astype(np.int32)
    cand = np.where(n_cand > 0, t['candidates'].argmax(-1), -1).astype(np.int32)
    tables = solver_tables.PuzzleTables(n=n, asym_dist=t['asym_dist'], min_dist=t['min_dist'], second_dist=t['second_dist'],
                                        n_candidates=n_cand, candidate=cand, asym_compat=t['asym_compat'],
                                        mutual_compat=t['mutual_compat'], best_buddy=t['best_buddy'])
    tables.start_piece_ordering = solver_tables.start_piece_ordering(tables.best_buddy, tables.mutual_compat)
    return tables


class _Side(enum.Enum):
    """What install() uses of the reference's PuzzlePieceSide (paikin_tal_solver/puzzle_piece.py)."""
    top = 0
    right = 1
    bottom = 2
    left = 3

    @staticmethod
    def get_all_sides():
        return [_Side.top, _Side.right, _Side.bottom, _Side.left]

    @property
    def complementary_side(self):
        return _Side((self.value + 2) % 4)


class _PieceInfo:
    """What install() uses of the reference's PieceDistanceInformation: the state its constructor starts from."""

    def __init__(self, id_numb, numb_pieces, puzzle_type):
        self._id, self._numb_pieces, self._puzzle_type = id_numb, numb_pieces, puzzle_type
        self._best_buddy_candidates = [[] for _ in range(4)]
        self._best_buddies = [[] for _ in range(4)]


class _InterPieceDistance:
    pass


@pytest.mark.parametrize('case', mg.CASES, ids=lambda c: f'seed{c[0]}_{c[1]}x{c[2]}')
def test_installed_object_matches_reference_fixture(case):
    """install() leaves an InterPieceDistance in the state the reference's own constructor left it in, as the fixture
    stores that state (tests/golden/make_golden_tables.py, run under NumPy >= 2 scalar rules like the tables here)."""
    from vited_b200 import solver_tables
    z, _ = _cases()
    seed = case[0]
    d, order = mg.case_inputs(*case)
    n = len(order)
    pieces = [mg._Piece(o) for o in order]
    ipd = solver_tables.install(_tables_from_oracle(d, order), pieces, 'type1', _InterPieceDistance, _PieceInfo, _Side)
    assert isinstance(ipd, _InterPieceDistance)
    assert [p.id_number for p in pieces] == list(range(n))
    assert ipd._numb_pieces == n and ipd._puzzle_type == 'type1' and ipd._distance_function is None
    assert [(a, b) for a, b, _ in ipd._start_piece_ordering] == [tuple(r) for r in z[f'start_order_{seed}'].tolist()]
    assert np.array_equal(np.array([float(c) for _, _, c in ipd._start_piece_ordering]), z[f'start_compat_{seed}'])
    assert len(ipd._piece_distance_info) == n
    for i, info in enumerate(ipd._piece_distance_info):
        assert info._id == i and info._numb_pieces == n
        for name, key in (('_asymmetric_distances', 'asym_dist'), ('_asymmetric_compatibilities', 'asym_compat'),
                          ('_mutual_compatibilities', 'mutual_compat')):
            x, y = getattr(info, name), z[f'{key}_{seed}'][i]
            assert x.shape == (4, n, 1) and x.dtype == y.dtype and np.array_equal(x[:, :, 0], y), name
        assert [int(v) for v in info._min_distance] == z[f'min_dist_{seed}'][i].tolist()
        assert [int(v) for v in info._second_best_distance] == z[f'second_dist_{seed}'][i].tolist()
        for s in range(4):
            cs = _Side((s + 2) % 4)
            assert info._best_buddy_candidates[s] == [(int(j), cs) for j in np.nonzero(z[f'candidates_{seed}'][i, s])[0]]
            b = int(z[f'best_buddy_{seed}'][i, s])
            assert info._best_buddies[s] == ([(b, cs)] if b >= 0 else [])


@pytest.mark.skipif(not os.path.isdir(REF), reason='needs a checkout of the reference project (VITED_REFERENCE)')
@pytest.mark.parametrize('case', [mg.CASES[1], mg.CASES[4], mg.CASES[6]], ids=lambda c: f'seed{c[0]}')
def test_installed_object_equals_reference_constructor(case):
    """install() leaves the reference's InterPieceDistance in exactly the state its own constructor does."""
    from vited_b200 import solver_tables
    sys.path.insert(0, REF)
    from paikin_tal_solver.inter_piece_distance import InterPieceDistance, PieceDistanceInformation
    from paikin_tal_solver.puzzle_importer import PuzzleType
    from paikin_tal_solver.puzzle_piece import PuzzlePieceSide
    d, order = mg.case_inputs(*case)
    pieces = [mg._Piece(o) for o in order]
    ipd = solver_tables.install(_tables_from_oracle(d, order), pieces, PuzzleType.type1, InterPieceDistance,
                                PieceDistanceInformation, PuzzlePieceSide)
    ref_pieces = [mg._Piece(o) for o in order]

    def distance_function(piece_i, piece_i_side, piece_j, piece_j_side):
        pred = d[piece_i.origin_piece_id][piece_j.origin_piece_id]
        table = {(PuzzlePieceSide.right, PuzzlePieceSide.left): 0, (PuzzlePieceSide.bottom, PuzzlePieceSide.top): 1,
                 (PuzzlePieceSide.left, PuzzlePieceSide.right): 2, (PuzzlePieceSide.top, PuzzlePieceSide.bottom): 3}
        return pred[table[(piece_i_side, piece_j_side)]] * 1000.

    ref = InterPieceDistance(ref_pieces, distance_function, PuzzleType.type1)
    assert [p.id_number for p in pieces] == [p.id_number for p in ref_pieces]
    assert ipd._numb_pieces == ref._numb_pieces and ipd._puzzle_type == ref._puzzle_type
    assert ipd._distance_function is None and ref._distance_function is None
    assert [(a, b, float(c)) for a, b, c in ipd._start_piece_ordering] == \
           [(a, b, float(c)) for a, b, c in ref._start_piece_ordering]
    for a, b in zip(ipd._piece_distance_info, ref._piece_distance_info):
        for name in ('_asymmetric_distances', '_asymmetric_compatibilities', '_mutual_compatibilities'):
            x, y = getattr(a, name), getattr(b, name)
            assert x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x, y), name
        assert [int(v) for v in a._min_distance] == [int(v) for v in b._min_distance]
        assert [int(v) for v in a._second_best_distance] == [int(v) for v in b._second_best_distance]
        assert [type(v) for v in a._min_distance] == [type(v) for v in b._min_distance]
        assert a._best_buddy_candidates == b._best_buddy_candidates
        assert a._best_buddies == b._best_buddies
        assert a._id == b._id and a._numb_pieces == b._numb_pieces


@pytest.mark.skipif(not os.path.isdir(REF), reason='needs a checkout of the reference project (VITED_REFERENCE)')
def test_reference_solver_runs_unmodified_on_prebuilt_tables(tmp_path, monkeypatch):
    """paikin_tal_driver (solver_driver.py:17-30) with the InterPieceDistance name in solver.py:212 bound to
    solver_tables.factory places every piece exactly where the run with the Python callbacks places it."""
    import cv2
    from vited_b200 import solver_tables, synthetic
    sys.path.insert(0, REF)
    import paikin_tal_solver.solver as ref_solver
    from paikin_tal_solver.inter_piece_distance import InterPieceDistance, PieceDistanceInformation
    from paikin_tal_solver.puzzle_importer import Puzzle
    from paikin_tal_solver.puzzle_piece import PuzzlePieceSide
    from solver_driver import paikin_tal_driver
    monkeypatch.setattr(ref_solver.PaikinTalSolver, '_PRINT_PROGRESS_MESSAGES', False, raising=False)
    rows, cols = 4, 5
    path = str(tmp_path / 'puzzle.png')
    cv2.imwrite(path, synthetic.synthetic_puzzle_image(rows, cols, 64, seed=3))
    d, _ = mg.case_inputs(11, rows, cols, 0, 0)            # true neighbours close, everything else far

    def solve(use_tables):
        puzzle = Puzzle(0, path, 64, starting_piece_id=0, erosion=0.07)
        pieces = puzzle.pieces
        order = np.random.default_rng(5).permutation(len(pieces))
        pieces = [pieces[k] for k in order]
        calls = [0]

        def distance_function(piece_i, piece_i_side, piece_j, piece_j_side):   # evaluation.py:116-131
            calls[0] += 1
            pred = d[piece_i.origin_piece_id][piece_j.origin_piece_id]
            if piece_j_side == PuzzlePieceSide.left and piece_i_side == PuzzlePieceSide.right:
                return pred[0] * 1000.
            if piece_j_side == PuzzlePieceSide.right and piece_i_side == PuzzlePieceSide.left:
                return pred[2] * 1000.
            if piece_j_side == PuzzlePieceSide.top and piece_i_side == PuzzlePieceSide.bottom:
                return pred[1] * 1000.
            if piece_j_side == PuzzlePieceSide.bottom and piece_i_side == PuzzlePieceSide.top:
                return pred[3] * 1000.
            return float('inf')

        if use_tables:
            tables = _tables_from_oracle(d, [p.origin_piece_id for p in pieces])
            monkeypatch.setattr(ref_solver, 'InterPieceDistance',
                                solver_tables.factory(tables, InterPieceDistance, PieceDistanceInformation, PuzzlePieceSide))
        else:
            monkeypatch.setattr(ref_solver, 'InterPieceDistance', InterPieceDistance)
        solved = paikin_tal_driver(pieces, 64, distance_function, puzzle.grid_size)
        return sorted((p.origin_piece_id, tuple(p.location)) for p in solved.pieces), calls[0]

    want, n_calls = solve(False)
    got, n_calls_tables = solve(True)
    assert n_calls == 4 * rows * cols * (rows * cols - 1) and n_calls_tables == 0
    assert got == want
