"""Reconstructs tests/golden/sample_san.json, the SAN move text of the 60 games of the reference's
py/validation/sample.csv, for when that CSV is not at hand.

    python oracle/make_golden_san.py

make_golden_chess.py, run where the reference tree is present, stores the CSV's own `id` and `moves`
columns verbatim in that file.  Without the CSV, this script writes the SAN from the UCI move lists in
tests/golden/sample_games.json (which make_golden_chess.py resolved from the CSV), and marks the file as a
reconstruction.  When the file already holds the verbatim CSV text, the script only checks that its
reconstruction equals it.

The writer shares no code with the C oracle whose SAN parser the test checks: legal moves come from the
product's native rules (scb200.rules_probe), the board is tracked here from the moves, and check is an attack
test written here.  Conventions: piece letter; file, else rank, else square disambiguation only where another
legal move of the same piece type reaches the same square; `x` on captures (en passant included); `=Q`
promotions; `O-O` / `O-O-O`; `+` / `#`.  The counts of plies, checks, mates, castles, promotions and en-passant
captures must equal the totals make_golden_chess.py recorded from the CSV.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "smart-chess-rust_b200"))
import scb200  # noqa: E402

GOLDEN = os.path.join(HERE, "..", "tests", "golden")
FILES = "abcdefgh"
VERBATIM = "py/validation/sample.csv"


def sq_name(sq):
    return FILES[sq & 7] + str((sq >> 3) + 1)


def start_board():
    b = {}
    for f, p in enumerate("RNBQKBNR"):
        b[f], b[56 + f] = ("w", p), ("b", p)
        b[8 + f], b[48 + f] = ("w", "P"), ("b", "P")
    return b


def attacked(b, sq, by):
    r, f = sq >> 3, sq & 7

    def at(rr, ff):
        return b.get(rr * 8 + ff) if 0 <= rr < 8 and 0 <= ff < 8 else None

    pr = r - 1 if by == "w" else r + 1
    if any(at(pr, f + d) == (by, "P") for d in (-1, 1)):
        return True
    for dr, df in ((1, 2), (2, 1), (-1, 2), (-2, 1), (1, -2), (2, -1), (-1, -2), (-2, -1)):
        if at(r + dr, f + df) == (by, "N"):
            return True
    for dr in (-1, 0, 1):
        for df in (-1, 0, 1):
            if (dr or df) and at(r + dr, f + df) == (by, "K"):
                return True
    for rays, sliders in ((((1, 0), (-1, 0), (0, 1), (0, -1)), "RQ"), (((1, 1), (1, -1), (-1, 1), (-1, -1)), "BQ")):
        for dr, df in rays:
            rr, ff = r + dr, f + df
            while 0 <= rr < 8 and 0 <= ff < 8:
                p = b.get(rr * 8 + ff)
                if p:
                    if p[0] == by and p[1] in sliders:
                        return True
                    break
                rr, ff = rr + dr, ff + df
    return False


def game_san(ucis, stats):
    b, hist, out = start_board(), [], []
    legal, _, _ = scb200.rules_probe(hist)
    for u in ucis:
        f, t = (int(u[1]) - 1) * 8 + FILES.index(u[0]), (int(u[3]) - 1) * 8 + FILES.index(u[2])
        promo = u[4:].upper()
        assert any(int(m[0]) == f and int(m[1]) == t for m in legal), u
        side, pt = b[f]
        if pt == "K" and abs((t & 7) - (f & 7)) == 2:
            s = "O-O" if (t & 7) > (f & 7) else "O-O-O"
            rook_f, rook_t = (f | 7, f + 1) if (t & 7) > (f & 7) else (f & ~7, f - 1)
            b[rook_t] = b.pop(rook_f)
            stats["castle"] += 1
        elif pt == "P":
            capture = (f & 7) != (t & 7)
            if capture and t not in b:                      # en passant: the captured pawn stands beside the mover
                del b[(f & ~7) | (t & 7)]
                stats["ep"] += 1
            s = (FILES[f & 7] + "x" if capture else "") + sq_name(t) + ("=" + promo if promo else "")
            stats["promo"] += bool(promo)
        else:
            rivals = [int(m[0]) for m in legal if int(m[1]) == t and int(m[0]) != f and b[int(m[0])] == (side, pt)]
            dis = ""
            if rivals:
                if all((r & 7) != (f & 7) for r in rivals):
                    dis = FILES[f & 7]
                elif all((r >> 3) != (f >> 3) for r in rivals):
                    dis = str((f >> 3) + 1)
                else:
                    dis = sq_name(f)
            s = pt + dis + ("x" if t in b else "") + sq_name(t)
        b[t] = (side, promo or pt)
        del b[f]
        hist.append((f, t, "  NBRQK".index(promo) if promo else 0))
        legal, _, _ = scb200.rules_probe(hist)
        king = next(sq for sq, p in b.items() if p == ("b" if side == "w" else "w", "K"))
        if attacked(b, king, side):
            s += "+" if len(legal) else "#"
            stats["check"] += 1
            stats["mate"] += not len(legal)
        out.append(s)
    return " ".join(out)


def main():
    with open(os.path.join(GOLDEN, "sample_games.json")) as f:
        sample = json.load(f)
    stats = dict.fromkeys(("check", "mate", "castle", "promo", "ep"), 0)
    games = [{"id": g["id"], "moves": game_san(g["uci"].split(), stats)} for g in sample["games"]]
    stats["plies"] = sum(len(g["moves"].split()) for g in games)
    assert stats == sample["totals"], (stats, sample["totals"])
    path = os.path.join(GOLDEN, "sample_san.json")
    if os.path.exists(path):
        with open(path) as f:
            old = json.load(f)
        if old["source"] == VERBATIM:
            assert old["games"] == games, "the reconstruction differs from the verbatim CSV text"
            print("reconstruction equals the verbatim CSV text", stats)
            return
    with open(path, "w") as f:
        json.dump({"source": "reconstructed: SAN written by oracle/make_golden_san.py from the UCI lists of "
                             "sample_games.json, not the text of " + VERBATIM, "games": games}, f, indent=0)
        f.write("\n")
    print(stats, len(games))


if __name__ == "__main__":
    main()
