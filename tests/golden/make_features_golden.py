"""Pins the SQL window-function features (SURVEY.md 8(f) N4) to the REFERENCE'S OWN SQL.

The reference builds its feature views as SQL strings inside create_database.py (:76-190) and executes
them on a MariaDB server at import time.  No MariaDB here - but the statements are plain window-function SQL, so this
script imports the UNMODIFIED module with
  * a stub `mysql.connector` whose cursor forwards every statement to an in-memory sqlite3 database (a dialect shim only:
    CREATE OR REPLACE VIEW -> DROP + CREATE VIEW, `KEY AUTO_INCREMENT` -> sqlite's spelling, identifiers that start with
    a digit get quoted, DESCRIBE -> PRAGMA table_info, a bare `Timestamp` in the window order of the two-table `target` view
    is qualified, and MariaDB's STD() = population standard deviation is registered as a sqlite window aggregate),
  * a stub `pytz` (config.py imports it; nothing on this path uses it),
fills `stock_data_joined` with a seed-fixed synthetic market table (values exactly representable in the FLOAT(6,2) / INT
columns the reference declares) and selects every view plus the `target` view.  Output: tests/golden/features.npz.

  python tests/golden/make_features_golden.py REFERENCE_DIR      (a checkout of the original project)
"""
import math
import os
import re
import sqlite3
import sys
import types

import numpy as np

if len(sys.argv) != 2:
    sys.exit(__doc__)
REF = os.path.abspath(sys.argv[1])
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "features.npz")


class _Std:
    """MariaDB STD(x) OVER (ROWS ...): population standard deviation of the frame, in double."""

    def __init__(self):
        self.vals = []

    def step(self, v):
        if v is not None:
            self.vals.append(float(v))

    def inverse(self, v):
        if v is not None:
            self.vals.remove(float(v))

    def value(self):
        if not self.vals:
            return None
        m = math.fsum(self.vals) / len(self.vals)
        return math.sqrt(math.fsum((x - m) ** 2 for x in self.vals) / len(self.vals))

    def finalize(self):
        return self.value()


def _translate(sql: str) -> list:
    s = sql.strip().rstrip(";")
    up = s.upper()
    if up.startswith("CREATE DATABASE") or up.startswith("USE "):
        return []
    s = s.replace("MEDIUMINT KEY AUTO_INCREMENT", "INTEGER PRIMARY KEY AUTOINCREMENT")
    s = re.sub(r"(?<![\w\"])(\d_[A-Za-z]\w*)", r'"\1"', s)             # 4_close -> "4_close"
    if " sd JOIN ATR " in s:        # `target`: both joined tables have a Timestamp (equal by the join condition); MariaDB
        s = s.replace("(ORDER BY Timestamp)", "(ORDER BY sd.Timestamp)")   # resolves the bare name, sqlite calls it ambiguous
    m = re.match(r"CREATE OR REPLACE VIEW\s+(\w+)", s, re.I)
    if m:
        return [f"DROP VIEW IF EXISTS {m.group(1)}", re.sub(r"CREATE OR REPLACE VIEW", "CREATE VIEW", s, flags=re.I)]
    return [s]


class _Cursor:
    def __init__(self, db):
        self.db, self.rows, self.log = db, [], []

    def execute(self, sql, *a):
        self.log.append(sql)
        m = re.match(r"\s*DESCRIBE\s+(\w+)", sql, re.I)
        if m:
            self.rows = [(r[1],) for r in self.db.execute(f"PRAGMA table_info({m.group(1)})")]
            return
        for stmt in _translate(sql):
            cur = self.db.execute(stmt)
            self.rows = cur.fetchall() if cur.description else []

    def fetchall(self):
        return self.rows


def _install_stubs(db):
    cur = _Cursor(db)
    conn = types.SimpleNamespace(cursor=lambda: cur, close=lambda: None, commit=lambda: None)
    mysql = types.ModuleType("mysql")
    connector = types.ModuleType("mysql.connector")
    connector.connect = lambda **kw: conn
    connector.Error = Exception
    connector.errorcode = types.SimpleNamespace(ER_ACCESS_DENIED_ERROR=1045)
    errorcode = types.ModuleType("mysql.connector.errorcode")
    errorcode.ER_ACCESS_DENIED_ERROR = 1045
    mysql.connector = connector
    sys.modules.update({"mysql": mysql, "mysql.connector": connector, "mysql.connector.errorcode": errorcode})
    pytz = types.ModuleType("pytz")
    pytz.timezone = lambda name: name
    sys.modules["pytz"] = pytz
    return cur


def synthetic_table(n, seed=7):
    rng = np.random.default_rng(seed)
    close = np.round(300 + np.cumsum(rng.normal(0, 0.35, n)), 2)
    close[60:78] = close[60]                                       # a flat stretch: stochastic max == min -> NULL
    high = np.round(close + np.abs(rng.normal(0.3, 0.2, n)), 2)
    low = np.round(close - np.abs(rng.normal(0.3, 0.2, n)), 2)
    volume = rng.integers(1000, 900000, n)
    delta = rng.integers(-5000, 5000, n)
    f32 = lambda a: np.asarray(a, np.float32)                      # MariaDB FLOAT columns hold single precision
    return f32(close), f32(high), f32(low), f32(volume), f32(delta)


def main():
    db = sqlite3.connect(":memory:")
    db.create_window_function("STD", 1, _Std)
    cur = _install_stubs(db)
    sys.path.insert(0, REF)
    import create_database as ref                                   # the UNMODIFIED reference module: creates table + views
    import config
    table = config.mysql_table_name
    n = 400
    close, high, low, volume, delta = synthetic_table(n)
    names = [r[1] for r in db.execute(f"PRAGMA table_info({table})")]
    special = {"4_close": close, "2_high": high, "3_low": low, "5_volume": volume, "delta": delta}
    rows = []
    for i in range(n):
        ts = "2020-01-{:02d} {:02d}:{:02d}:00".format(2 + i // 200, 9 + (i % 200) * 2 // 60, (i % 200) * 2 % 60)
        row = []
        for c in names:
            if c == "ID":
                row.append(i + 1)
            elif c == "Timestamp":
                row.append(ts)
            elif c in special:
                row.append(float(special[c][i]))
            else:
                row.append(0)
        rows.append(tuple(row))
    q = "INSERT INTO {} ({}) VALUES ({})".format(table, ", ".join('"%s"' % c for c in names), ", ".join("?" * len(names)))
    db.executemany(q, rows)

    def col(view, field):
        return np.array([np.nan if r[0] is None else float(r[0]) for r in db.execute(f'SELECT "{field}" FROM {view} ORDER BY Timestamp')])

    feats = [col("bollinger_bands", "upper_BB_dist"), col("bollinger_bands", "lower_BB_dist")]
    feats += [col("vol_MA", f"vol_MA{p}") for p in config.volume_MA_periods]
    feats += [col("price_MA", f"price_MA{p}") for p in config.price_MA_periods]
    feats += [col("delta_MA", f"delta_MA{p}") for p in config.delta_MA_periods]
    feats += [col("stochastic_oscillator", "stoch"), col("ATR", "ATR"), col("price_change", "price_change")]
    tgt = np.stack([col("target", f) for f in ("up1", "up2", "down1", "down2")], axis=1)
    views = [s for s in cur.log if "CREATE OR REPLACE VIEW" in s]
    np.savez_compressed(OUT, close=close, high=high, low=low, volume=volume, delta=delta, features=np.stack(feats, axis=1),
                        targets=tgt, volume_MA_periods=np.array(config.volume_MA_periods), price_MA_periods=np.array(config.price_MA_periods),
                        delta_MA_periods=np.array(config.delta_MA_periods), bollinger_bands_period=config.bollinger_bands_period,
                        bollinger_bands_std=config.bollinger_bands_std, n_views=len(views), join_statement=str(ref.join_statement))
    print(f"{OUT}: {n} rows, {len(feats)} feature columns, {len(views)} reference views executed; "
          f"NULLs: stoch {int(np.isnan(feats[-3]).sum())}, price_change {int(np.isnan(feats[-1]).sum())}")


if __name__ == "__main__":
    main()
