"""SGF reader (elf_b200/sgf.py) against the reference's reader and its own gtests.

* known answers of ELF's src_cpp/elfgames/go/sgf/sgf_test.cc (9x9, MiniGo-derived game
  records): coordinates, header fields, every move replayable, the "miracle final board";
* field-by-field parity with the compiled reference Sgf class (oracle/_ref, ref_sgf_parse) on those
  records, on synthetic records made from oracle playouts (with blanks, comments, escapes, passes,
  off-board letters) and, from stored results (tests/golden), on a sample of its 19x19 ladder_suite records.
"""
import json
import os
import random

import pytest

from elf_b200 import sgf
from tests import oracles
from tests.test_reference_known_answers import A, OracleGame, RefGame, board_rows, turn

N = 9
PASS = N * N

# sgf_test.cc:34-47
SGF_MAKE = (
    "(;CA[UTF-8]SZ[9]PB[Murakawa Daisuke]PW[Iyama Yuta]KM[6.5]HA[0]RE[W+1.5]GM[1];"
    "B[fd];W[cf];B[eg];W[dd];B[dc];W[cc];B[de];W[cd];B[ed];W[he];B[ce];W[be];B[df];W[bf];"
    "B[hd];W[ge];B[gd];W[gg];B[db];W[cb];B[cg];W[bg];B[gh];W[fh];B[hh];W[fg];B[eh];W[ei];"
    "B[di];W[fi];B[hg];W[dh];B[ch];W[ci];B[bh];W[ff];B[fe];W[hf];B[id];W[bi];B[ah];W[ef];"
    "B[dg];W[ee];B[di];W[ig];B[ai];W[ih];B[fb];W[hi];B[ag];W[ab];B[bd];W[bc];B[ae];W[ad];"
    "B[af];W[bd];B[ca];W[ba];B[da];W[ie])"
)
# sgf_test.cc:64-75 / 118-128 (same record)
SGF_CHINESE = (
    "(;GM[1]FF[4]CA[UTF-8]AP[CGoban:3]ST[2]RU[Chinese]SZ[9]HA[2]RE[Void]KM[5.50]"
    "PW[test_white]PB[test_black]RE[B+39.50];"
    "B[gc];B[cg];W[ee];B[gg];W[eg];B[ge];W[ce];B[ec];W[cc];B[dd];W[de];B[cd];W[bd];B[bc];"
    "W[bb];B[be];W[ac];B[bf];W[dh];B[ch];W[ci];B[bi];W[di];B[ah];W[gh];B[hh];W[fh];B[hg];"
    "W[gi];B[fg];W[dg];B[ei];W[cf];B[ef];W[ff];B[fe];W[bg];B[bh];W[af];B[ag];W[ae];B[ad];"
    "W[ae];B[ed];W[db];B[df];W[eb];B[fb];W[ea];B[fa])"
)
# sgf_test.cc:97-100
SGF_JAPANESE = (
    "(;GM[1]FF[4]CA[UTF-8]AP[CGoban:3]ST[2]RU[Japanese]SZ[9]HA[2]RE[Void]KM[5.50]PW[test_white]"
    "PB[test_black]AB[gc][cg];W[ee];B[dg])"
)
# sgf_test.cc:143-152
FINAL_CHINESE = ["....OX...", ".O.OOX...", "O.O.X.X..", ".OXXX....", "OX...XX..", ".X.XXO...", "X.XOOXXX.",
                 "XXXO.OOX.", ".XOOX.O.."]

CPU_GAMES = [pytest.param(OracleGame, id="oracle"),
             pytest.param(RefGame, id="ref",
                          marks=pytest.mark.skipif(not oracles.have_ref(N), reason="oracle/_ref not built"))]


def replay(g, record):  # the loop of sgf_test.cc:52-58,80-88
    for m in record:
        if turn(g) != m.player:
            g.forward(PASS)  # "to handle handicap"
        assert g.forward(m.action), m


def test_translate_sgf_move():  # sgf_test.cc:24-28
    assert sgf.str2action("db", N) == A(3, 1)
    assert sgf.str2action("aa", N) == A(0, 0)
    assert sgf.str2action("", N) == PASS  # M_PASS == 0 in the reference
    assert sgf.action2str(A(3, 1), N) == "db" and sgf.action2str(PASS, N) == ""
    assert sgf.str2action("tt", 19) == sgf.INVALID and sgf.str2action("ss", 19) == 19 * 18 + 18


@pytest.mark.parametrize("Game", CPU_GAMES)
def test_make_sgf_replays(Game):  # sgf_test.cc:33-59
    rec = sgf.Sgf.loads(SGF_MAKE, N)
    assert len(rec) == 62 and rec.header.komi == 6.5 and rec.header.winner == sgf.S_WHITE
    assert rec.header.win_margin == 1.5 and rec.header.black_name == "Murakawa Daisuke"
    replay(Game(), rec)


@pytest.mark.parametrize("Game", CPU_GAMES)
def test_sgf_props_and_final_board(Game):  # sgf_test.cc:61-91,115-156
    rec = sgf.Sgf.loads(SGF_CHINESE, N)
    assert rec.header.komi == 5.5 and rec.header.handi == 2 and rec.header.size == 9
    assert rec.header.winner == sgf.S_BLACK and rec.header.win_margin == 39.5
    assert rec.header.white_name == "test_white" and rec.header.black_name == "test_black"
    g = Game()
    replay(g, rec)
    assert board_rows(g) == FINAL_CHINESE


@pytest.mark.parametrize("Game", CPU_GAMES)
def test_japanese_handicap(Game):  # sgf_test.cc:95-113: AB[] stones live in the header node and are not moves
    rec = sgf.Sgf.loads(SGF_JAPANESE, N)
    assert rec.actions() == [sgf.str2action("ee", N), sgf.str2action("dg", N)]
    assert rec.players() == [sgf.S_WHITE, sgf.S_BLACK]
    replay(Game(), rec)


def test_compact_record_strings():  # coords2sgfstr / sgfstr2coords, sgf.h:87-125
    from elf_b200.record import moves_to_sgf

    acts = [A(3, 1), PASS, A(0, 0), A(8, 8)]
    s = moves_to_sgf(acts, N)
    assert s == "(;B[db];W[];B[aa];W[ii])"
    assert sgf.sgfstr2actions(s, N) == acts
    assert sgf.sgfstr2actions("", N) == [] and sgf.sgfstr2actions("B[aa]", N) == []


def test_main_line_of_a_tree():
    rec = sgf.Sgf.loads("(;SZ[9];B[aa](;W[bb];B[cc])(;W[dd](;B[ee])(;B[ff])))", N)
    assert [sgf.action2str(a, N) for a in rec.actions()] == ["aa", "bb", "cc"]
    with pytest.raises(ValueError):
        sgf.Sgf.loads("no node here", N)
    with pytest.raises(ValueError):
        sgf.Sgf.loads("(;SZ[9]KM[7.5])", N)  # header only: the reference's load() returns false too


# ---- parity with the compiled reference reader ------------------------------------------------
REF_PARSE = object()


def same_as_reference(text, n, want=REF_PARSE):
    """``want``: what the reference's reader returned for ``text`` (default: ask the compiled reference)"""
    if want is REF_PARSE:
        want = oracles.ref_sgf_parse(text, n)
    try:
        got = sgf.Sgf.loads(text, n)
    except ValueError:
        assert want is None, text[:200]
        return 0
    assert want is not None, text[:200]
    assert got.actions() == want["actions"], text[:200]
    # SgfEntry::player is left uninitialised by the reference for nodes without B/W: compare movers only
    for m, p in zip(got.moves, want["players"]):
        if m.player != sgf.S_OFF_BOARD:
            assert m.player == p
    h = got.header
    assert (h.size, h.handi, h.winner, got.num_moves) == (want["size"], want["handi"], want["winner"],
                                                          want["num_moves"]), text[:200]
    assert abs(h.komi - want["komi"]) < 1e-6 and abs(h.win_margin - want["win_margin"]) < 1e-4
    return len(got)


needs_ref9 = pytest.mark.skipif(not oracles.have_ref(9), reason="oracle/_ref not built")
needs_ref19 = pytest.mark.skipif(not oracles.have_ref(19), reason="oracle/_ref not built")


@needs_ref9
def test_reader_matches_reference_on_its_test_records():
    for text in (SGF_MAKE, SGF_CHINESE, SGF_JAPANESE):
        assert same_as_reference(text, N) > 0


def synth_record(rng, n, lib):
    """a linear record from a random legal game, decorated with what real files contain"""
    o = oracles.Oracle(n, lib)
    letters = "abcdefghijklmnopqrstuvwxyz"
    hdr = "(;GM[1]FF[4]" + rng.choice(["", "\n", " "]) + f"SZ[{n}]KM[{rng.choice(['7.5', '6.5', '0', '5.50', '-3'])}]"
    hdr += rng.choice(["", "HA[0]", "HA[2]", "HA[ 3]"])
    hdr += rng.choice(["", "RE[B+Resign]", "RE[W+2.5]", "RE[b+0.5]", "RE[W+T]", "RE[B+]", "RE[Void]", "RE[]"])
    hdr += rng.choice(["", "PW[a \\] b]PB[x]", "C[root (comment); with ] \\] stuff]".replace(" ] ", " ")])
    body = []
    for t in range(rng.randrange(1, 80)):
        if o.terminated():
            break
        legal = [a for a in range(n * n) if o.legal()[a]]
        r = rng.random()
        if r < 0.06 or not legal:
            a, val = n * n, rng.choice(["", "", " "])
        elif r < 0.09:
            a, val = None, rng.choice(["tt", "zz", "A1", "a", "a "])  # off-board / malformed: never replayed
        else:
            a = rng.choice(legal)
            val = letters[a // n] + rng.choice(["", " ", "\n"]) + letters[a % n]
        who = "B" if o.info()[1] == 1 else "W"
        node = rng.choice([";", ";", "\n;", "; "]) + rng.choice(["", "", " "]) + who + "[" + val + "]"
        node += rng.choice(["", "", f"{who}L[{rng.randrange(900)}]", "C[nice; move (really)]", "C[esc \\] aped]", "N[x]"])
        body.append(node)
        if a is not None:
            assert o.forward(a)
    return hdr + "".join(body) + rng.choice([")", ")\n", ""])


@needs_ref9
@needs_ref19
def test_reader_matches_reference_on_synthetic_records(oracle_lib):
    rng = random.Random(20260922)
    total = 0
    for i in range(300):
        n = 9 if i % 3 else 19
        total += same_as_reference(synth_record(rng, n, oracle_lib), n)
    assert total > 5000


LADDER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sgf_ladder_suite.json")


def test_reader_matches_reference_on_ladder_suite(oracle_lib):
    """a sample of ELF's ladder_suite records (tests/golden) with the reference reader's results stored beside
    them; when the compiled reference is present it is asked again and must still agree with the stored data"""
    records = json.load(open(LADDER))["records"]
    assert len(records) > 25
    for r in records:
        text, f = r["text"], r["name"]
        if oracles.have_ref(19):
            assert oracles.ref_sgf_parse(text, 19) == r["reference"], f
        k = same_as_reference(text, 19, r["reference"])
        assert k > 20, f
        # every record is a legal 19x19 game for the board restatement as well
        rec = sgf.Sgf.loads(text)
        assert rec.header.size == 19
        o = oracles.Oracle(19, oracle_lib)
        for m in rec:
            if m.action < 0:
                break
            assert int(o.info()[1]) == m.player and o.forward(m.action), (f, m)
