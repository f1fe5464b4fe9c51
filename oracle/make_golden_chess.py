"""Generates tests/golden/sample_games.json and tests/golden/sample_san.json from the reference's only
shipped fixture, py/validation/sample.csv of the reference tree (60 real games in SAN), using the CPU oracle.

Run in the build container (the reference tree is not present on the GPU box):
    python oracle/make_golden_chess.py

Per game it stores the UCI move list (so the games can be replayed where the reference is
absent) and a sha256 over (planes, meta, legal-move indices) of every position, which pins
the oracle against silent regressions; sample_san.json gets the CSV's `id` and `moves` columns
verbatim (make_golden_san.py reconstructs that text where the CSV is not at hand).  What the
replay itself pins about python-chess semantics: every SAN token resolves to exactly one
oracle-legal move, `+`/`#` suffixes agree with the oracle's check / no-legal-move state,
O-O/O-O-O/promotions/en-passant all occur.
"""
import csv
import hashlib
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import chess_oracle as co  # noqa: E402

SRC = "/root/reference/py/validation/sample.csv"
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden", "sample_games.json")


def replay(sans):
    g = co.Game()
    h = hashlib.sha256()
    ucis = []
    stats = {"check": 0, "mate": 0, "castle": 0, "promo": 0, "ep": 0}
    for san in sans:
        planes, meta = g.encode()
        idx = g.move_indices()
        h.update(planes.tobytes()); h.update(meta.tobytes()); h.update(idx.tobytes())
        m = g.parse_san(san)
        f, t, p = int(m[0]), int(m[1]), int(m[2])
        if abs(g.piece_at(f)) == 1 and (f & 7) != (t & 7) and g.piece_at(t) == 0:
            stats["ep"] += 1
        if san.startswith("O-O"):
            stats["castle"] += 1
        if p:
            stats["promo"] += 1
        g.push(m)
        ucis.append(co.uci(m))
        chk = g.is_check()
        nolegal = len(g.legal_moves()) == 0
        assert chk == (san.endswith("+") or san.endswith("#")), (san, chk)
        assert (chk and nolegal) == san.endswith("#"), (san, chk, nolegal)
        stats["check"] += chk
        stats["mate"] += chk and nolegal
    return ucis, h.hexdigest(), stats


def main():
    games, san_rows = [], []
    tot = {"check": 0, "mate": 0, "castle": 0, "promo": 0, "ep": 0, "plies": 0}
    with open(SRC) as f:
        for row in csv.DictReader(f):
            sans = row["moves"].split()
            ucis, digest, st = replay(sans)
            games.append({"id": row["id"], "uci": " ".join(ucis), "sha256": digest})
            san_rows.append({"id": row["id"], "moves": row["moves"]})
            for k, v in st.items():
                tot[k] += int(v)
            tot["plies"] += len(sans)
    with open(DST, "w") as f:
        json.dump({"source": "py/validation/sample.csv", "totals": tot, "games": games}, f, indent=0)
    with open(os.path.join(os.path.dirname(DST), "sample_san.json"), "w") as f:
        json.dump({"source": "py/validation/sample.csv", "games": san_rows}, f, indent=0)
        f.write("\n")
    print(tot, len(games))


if __name__ == "__main__":
    main()
