"""Host-side integration pieces (no GPU): the batched metadata join against the per-hit loop it replaces
(/root/reference/search.py:137-153), and the integration patch applying cleanly to the reference tree."""
import os
import shutil
import sqlite3
import subprocess

import numpy as np
import pytest

from wise_b200.metadata_join import join_hits_batched

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _db(n_media=40, n_vec=3000):
    conn = sqlite3.connect(":memory:")
    conn.execute("CREATE TABLE media (id INTEGER PRIMARY KEY AUTOINCREMENT, path TEXT NOT NULL)")
    conn.execute("CREATE TABLE vectors (id INTEGER PRIMARY KEY AUTOINCREMENT, modality TEXT, media_id INTEGER NOT NULL, "
                 "timestamp FLOAT, end_timestamp FLOAT)")
    conn.executemany("INSERT INTO media (path) VALUES (?)", [(f"videos/clip_{i:03d}.mp4",) for i in range(n_media)])
    rng = np.random.default_rng(0)
    rows = [("video" if i % 3 else "audio", int(rng.integers(1, n_media + 1)), float(i) * 0.5,
             None if i % 3 else float(i) * 0.5 + 4.0) for i in range(n_vec)]
    conn.executemany("INSERT INTO vectors (modality, media_id, timestamp, end_timestamp) VALUES (?,?,?,?)", rows)
    return conn


def _per_hit_loop(conn, ids, dist):
    """The reference's loop: 2 SELECTs per hit, stop at id -1."""
    files, pts, scores = [], [], []
    for rank in range(len(ids)):
        vid = int(ids[rank])
        if vid == -1:
            break
        media_id, ts, end_ts = conn.execute("SELECT media_id, timestamp, end_timestamp FROM vectors WHERE id=?", (vid,)).fetchone()
        (path,) = conn.execute("SELECT path FROM media WHERE id=?", (media_id,)).fetchone()
        files.append(path)
        pts.append(ts if end_ts is None else [ts, end_ts])
        scores.append(float(dist[rank]))
    return {"match_filename_list": files, "match_pts_list": pts, "match_score_list": scores}


@pytest.mark.parametrize("topk,valid", [(10, 10), (1000, 1000), (2048, 1500), (20, 0)])
def test_batched_join_equals_per_hit_loop(topk, valid):
    conn = _db()
    rng = np.random.default_rng(topk)
    ids = np.full(topk, -1, np.int64)
    ids[:valid] = rng.permutation(3000)[:valid] + 1
    dist = np.sort(rng.random(topk).astype(np.float32))[::-1]
    assert join_hits_batched(conn, ids, dist) == _per_hit_loop(conn, ids, dist)


def test_batched_join_reports_unknown_ids():
    conn = _db()
    with pytest.raises(RuntimeError):
        join_hits_batched(conn, np.array([5, 999999, -1]), np.array([0.9, 0.8, 0.0], np.float32))


# A checkout of the WISE 2 sources (https://github.com/ox-vgg/wise) that integration/wise_b200.patch targets.
WISE_SRC = os.environ.get("WISE_SRC", "")


@pytest.mark.skipif(not WISE_SRC or not os.path.isdir(os.path.join(WISE_SRC, "src", "index"))
                    or shutil.which("patch") is None,
                    reason="needs WISE_SRC set to a WISE 2 checkout, and patch(1)")
def test_integration_patch_applies_to_the_reference(tmp_path):
    """integration/wise_b200.patch: backend switch (src/index/feature_search_index.py:1), request batcher
    (api/routes.py:1407) and batched metadata join (search.py:137-153) - applies cleanly and leaves valid python."""
    import ast
    for f in ("src/index/feature_search_index.py", "search.py", "api/routes.py"):
        os.makedirs(tmp_path / os.path.dirname(f), exist_ok=True)
        shutil.copy(os.path.join(WISE_SRC, f), tmp_path / f)
    r = subprocess.run(["patch", "-p1", "--dry-run", "-i", os.path.join(ROOT, "integration", "wise_b200.patch")], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run(["patch", "-p1", "-i", os.path.join(ROOT, "integration", "wise_b200.patch")], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    for f in ("src/index/feature_search_index.py", "search.py", "api/routes.py"):
        src = (tmp_path / f).read_text()
        ast.parse(src)
        assert "wise_b200" in src
