"""Host-side mirror of the reference's `Engine` for the similarity-search path only.

Same method names, argument meaning and error behaviour as src/engine.rs for the calls the UI makes
on this path (`open`, `new`, `query_by_image_hash_from_image`, `get_query_results`,
`clear_query_results`, `insert_image_from_memory`, `max_distance_from_query`), plus `load_more_results`, over Python's sqlite3 and
the C-ABI library.  The reference's toolchain (Rust) is absent from this image, so this is the
executable form of the patch INTEGRATION.md describes.  Everything outside the path (text search,
tags, crawling, image decoding, thumbnails) is not built.
"""
from __future__ import annotations

import sqlite3
import sys
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

from .corpus import Corpus

# src/engine.rs:22-25
DEFAULT_MAX_QUERY_DISTANCE = 1e3
DEFAULT_MAX_SEARCH_RESULTS = 100

# src/engine.rs:31-48
IMAGE_SCHEMA_V1 = """CREATE TABLE images (
	id               INTEGER PRIMARY KEY,
	filename         TEXT NOT NULL,
	path             TEXT NOT NULL,
	image_width      INTEGER,
	image_height     INTEGER,
	thumbnail        BLOB,
	created          DATETIME,
	indexed          DATETIME,
	UNIQUE(path)
)"""
TAG_SCHEMA_V1 = "CREATE TABLE tags (image_id INTEGER, name TEXT NOT NULL, value TEXT)"
WATCHED_DIRECTORIES_SCHEMA_V1 = "CREATE TABLE watched_directories (glob TEXT PRIMARY KEY)"
HASH_TABLE_SCHEMA_V1 = "CREATE TABLE $tablename$ (image_id INTEGER PRIMARY KEY, hash BLOB)"
# src/engine.rs:51-58
SELECT_FIELDS = "images.id, images.filename, images.path, images.image_width, images.image_height, images.thumbnail"


@dataclass
class IndexedImage:
    """The fields of src/indexed_image.rs:16-32 that exist without decoding an image."""
    id: int = 0
    filename: str = ""
    path: str = ""
    resolution: Tuple[int, int] = (0, 0)
    thumbnail: bytes = b""
    tags: Dict[str, str] = field(default_factory=dict)
    phash: Optional[bytes] = None
    visual_hash: Optional[bytes] = None            # :28, the query / the stored embedding
    distance_from_query: Optional[float] = None    # :31, f64


class Engine:
    def __init__(self, db_path: str, device: int = 0, _create: bool = False):
        """Engine::open (src/engine.rs:117-145): opens the DB and -- the GPU hook after :129 -- loads
        `SELECT image_id, hash FROM semantic_hashes ORDER BY image_id` into the device corpus."""
        self.db_path = db_path
        self.device = device
        self.write_connection = sqlite3.connect(db_path, check_same_thread=False)
        if _create:                     # Engine::new, on the connection that is kept (a ':memory:' DB lives and dies with it)
            self._create_tables(self.write_connection)
        self.read_connection = sqlite3.connect(f"file:{db_path}?mode=ro", uri=True, check_same_thread=False) \
            if db_path != ":memory:" else self.write_connection
        if db_path != ":memory:":
            self.write_connection.execute("PRAGMA journal_mode=WAL")     # :122
        self.max_search_results = DEFAULT_MAX_SEARCH_RESULTS            # :91 (unused by queries upstream too)
        self.max_distance_from_query = DEFAULT_MAX_QUERY_DISTANCE       # :92
        self.cached_search_results: Optional[List[IndexedImage]] = None
        self._last_query: Optional[dict] = None                          # load_more_results continues it
        self.corpus: Optional[Corpus] = None
        self.skipped_rows = 0
        self._load_corpus()

    # -- construction -------------------------------------------------------------------------------
    @classmethod
    def new(cls, db_path: str, device: int = 0) -> "Engine":
        """Engine::new (src/engine.rs:98-115): creates the tables, then opens."""
        return cls(db_path, device, _create=True)

    @staticmethod
    def _create_tables(conn: sqlite3.Connection) -> None:
        conn.execute(IMAGE_SCHEMA_V1)                                                    # :105-109
        conn.execute(WATCHED_DIRECTORIES_SCHEMA_V1)
        conn.execute(TAG_SCHEMA_V1)
        conn.execute(HASH_TABLE_SCHEMA_V1.replace("$tablename$", "phashes"))
        conn.execute(HASH_TABLE_SCHEMA_V1.replace("$tablename$", "semantic_hashes"))
        conn.commit()

    @classmethod
    def open(cls, db_path: str, device: int = 0) -> "Engine":
        return cls(db_path, device)

    def _load_corpus(self) -> None:
        rows = self.read_connection.execute("SELECT image_id, hash FROM semantic_hashes ORDER BY image_id").fetchall()
        if not rows:
            return
        # The BLOB column is length-agnostic (:48); the device corpus has one dim.  Rows of another
        # length cannot be represented (the reference would zip-truncate them, :585): they are skipped
        # and counted, never silently mis-scored.
        # dim = the modal blob length among the non-NULL rows.
        lengths: Dict[int, int] = {}
        for _, h in rows:
            if h is not None and len(h) > 0:
                lengths[len(h)] = lengths.get(len(h), 0) + 1
        if not lengths:
            self.skipped_rows = len(rows)
            return
        dim = max(lengths.items(), key=lambda kv: (kv[1], -kv[0]))[0]
        keep = [(i, h) for i, h in rows if h is not None and len(h) == dim]
        self.skipped_rows = len(rows) - len(keep)
        self.corpus = Corpus(dim, capacity_hint=len(keep), device=self.device)
        ids = np.fromiter((i for i, _ in keep), dtype=np.int64, count=len(keep))
        hashes = np.frombuffer(b"".join(h for _, h in keep), dtype=np.uint8).reshape(len(keep), dim)
        self.corpus.load(ids, hashes)

    def close(self) -> None:
        if self.corpus is not None:
            self.corpus.close()
            self.corpus = None
        if self.read_connection is not self.write_connection:
            self.read_connection.close()
        self.write_connection.close()

    # -- search -------------------------------------------------------------------------------------
    _JOIN_SQL = (f"SELECT {SELECT_FIELDS}, semantic_hashes.hash FROM images "
                 "JOIN semantic_hashes ON images.id = semantic_hashes.image_id WHERE images.id = ?")

    def query_by_image_hash_from_image(self, indexed_image: IndexedImage) -> None:
        """src/engine.rs:363-396.  Returns silently when the hash is missing (:364-368); otherwise fills
        cached_search_results with at most 100 images (:381) with dist < max_distance_from_query (:379),
        ordered by dist ascending (:380), each carrying visual_hash and distance_from_query (:385-386).
        Upstream applies LIMIT 100 after the INNER JOIN with `images`, so a hash without an image row does not use up
        one of the 100: the GPU rows are taken in pages of 100 after the last one consumed until 100 joined rows are
        found or the table is exhausted, however many such hashes come first."""
        self._similarity_query(indexed_image, None)

    def query_by_image_hash_within_folder(self, indexed_image: IndexedImage, folder: str) -> None:
        """query_by_image_hash_from_image restricted to the images under `folder`: the similarity SQL with
        `AND substr(images.path, 1, length(?)) = ?` added (folder with a trailing separator, so that /a/b does not match
        /a/bc; no LIKE, whose % and _ occur in real paths).  The folder's ids come from `images`; a row deleted between
        the id query and the search is dropped by the join like any other hash without an image row."""
        self._similarity_query(indexed_image, folder)

    def load_more_results(self, count: int = DEFAULT_MAX_SEARCH_RESULTS) -> None:
        """"Show more": extends cached_search_results with the next `count` joined rows of the last similarity query
        (query_by_image_hash_from_image or ..._within_folder), in the same order -- the verbatim SQL with
        LIMIT count OFFSET (rows shown so far).  Each call is one keyset page after the last GPU row consumed, over the
        table as it is now; nothing happens without a previous query."""
        if self._last_query is None or self.cached_search_results is None:
            return
        t0 = time.perf_counter()
        more = self._joined_rows(int(count))
        self.cached_search_results = self.cached_search_results + more
        sys.stderr.write(f"Time to search DB: {time.perf_counter() - t0:.6f}s  Results: {len(more)} more\n")

    def _similarity_query(self, indexed_image: IndexedImage, folder: Optional[str]) -> None:
        if indexed_image.visual_hash is None:
            sys.stderr.write("TODO: IndexedImage is somehow missing a hash!\n")
            return
        self.cached_search_results = None
        self._last_query = None
        t0 = time.perf_counter()
        results: List[IndexedImage] = []
        if self.corpus is not None:
            within = None
            if folder is not None:
                prefix = folder if folder.endswith(("/", "\\")) else folder + "/"
                within = np.fromiter((r[0] for r in self.read_connection.execute(
                    "SELECT id FROM images WHERE substr(path, 1, length(?)) = ? ORDER BY id", (prefix, prefix))), dtype=np.int64)
            # what load_more_results continues from: the query, its max_dist and folder, the last GPU row consumed
            self._last_query = dict(query=np.frombuffer(indexed_image.visual_hash, np.uint8), max_dist=self.max_distance_from_query,
                                    within=within, cursor=None, exhausted=False)
            results = self._joined_rows(DEFAULT_MAX_SEARCH_RESULTS)                  # LIMIT 100, :381
        self.cached_search_results = results
        sys.stderr.write(f"Time to search DB: {time.perf_counter() - t0:.6f}s  Results: {len(results)}\n")

    def _joined_rows(self, count: int) -> List[IndexedImage]:
        """The next `count` rows of the last similarity query that have an `images` row (INNER JOIN semantics), hydrated
        by indexed lookups in the GPU's order (SURVEY.md 8f N1).  GPU rows come in pages of 100 after the last row
        consumed; a page shorter than 100 is the end of the table."""
        st = self._last_query
        out: List[IndexedImage] = []
        while len(out) < count and not st["exhausted"]:
            after = None if st["cursor"] is None else [st["cursor"]]
            res = self.corpus.search(st["query"], DEFAULT_MAX_SEARCH_RESULTS, st["max_dist"], within=st["within"], after=after)[0]
            for image_id, dist in zip(res.ids, res.dist):
                st["cursor"] = (dist, int(image_id))
                row = self.read_connection.execute(self._JOIN_SQL, (int(image_id),)).fetchone()
                if row is not None:
                    out.append(IndexedImage(id=row[0], filename=row[1], path=row[2], resolution=(row[3], row[4]),
                                            thumbnail=row[5], visual_hash=row[6], distance_from_query=float(dist)))
                    if len(out) == count:
                        break
            else:
                st["exhausted"] = len(res.ids) < DEFAULT_MAX_SEARCH_RESULTS
        return out

    def get_query_results(self) -> Optional[List[IndexedImage]]:
        return None if self.cached_search_results is None else list(self.cached_search_results)   # :398-400

    def clear_query_results(self) -> None:
        self.cached_search_results = None                                                         # :402

    # -- ingest -------------------------------------------------------------------------------------
    def insert_image_from_memory(self, img: IndexedImage) -> None:
        """insert_image_from_connection (src/engine.rs:228-259) for the columns this path owns, plus the GPU
        append hook: the hash is appended only when the INSERT changed a row -- a duplicate path makes
        `INSERT OR IGNORE INTO images` a no-op, last_insert_rowid() stale (:234) and the hash INSERT ignored."""
        conn = self.write_connection
        appended = None
        try:
            conn.execute("INSERT OR IGNORE INTO images (filename, path, image_width, image_height, thumbnail) VALUES (?, ?, ?, ?, ?)",
                         (img.filename, img.path, img.resolution[0], img.resolution[1], img.thumbnail))
            img.id = conn.execute("SELECT last_insert_rowid()").fetchone()[0]
            if img.visual_hash is not None:
                cur = conn.execute("INSERT OR IGNORE INTO semantic_hashes (image_id, hash) VALUES (?, ?)", (img.id, img.visual_hash))
                if cur.rowcount == 1:
                    appended = (img.id, img.visual_hash)
            conn.commit()
        except Exception:
            conn.rollback()
            raise
        # the device corpus is a cache of the committed table: append only what the DB now holds
        if appended is not None:
            if self.corpus is None:
                self.corpus = Corpus(len(appended[1]), device=self.device)
            if len(appended[1]) == self.corpus.dim:
                self.corpus.append(np.array([appended[0]], np.int64), np.frombuffer(appended[1], np.uint8).reshape(1, -1))
            else:
                self.skipped_rows += 1

    def remove_images(self, ids) -> None:
        """Deletes images from the two tables the similarity query joins (`images`, `semantic_hashes`) in one
        transaction, then removes their hashes from the device corpus: the hook the TODO in remove_tracked_folder
        (src/engine.rs:414) would call with the folder's image ids."""
        ids = [int(i) for i in np.asarray(ids, dtype=np.int64).reshape(-1)]
        if not ids:
            return
        conn = self.write_connection
        try:
            for first in range(0, len(ids), 500):                        # SQLite's bound-parameter limit
                part = ids[first:first + 500]
                marks = ",".join("?" * len(part))
                conn.execute(f"DELETE FROM semantic_hashes WHERE image_id IN ({marks})", part)
                conn.execute(f"DELETE FROM images WHERE id IN ({marks})", part)
            conn.commit()
        except Exception:
            conn.rollback()
            raise
        # as for inserts, the device corpus follows only what has been committed
        if self.corpus is not None:
            self.corpus.remove(np.asarray(ids, np.int64))

    def update_image_hashes(self, pairs) -> None:
        """`UPDATE semantic_hashes SET hash = ? WHERE image_id = ?` for every (image_id, hash) pair, in order, in one
        transaction; then the device corpus follows the rows the UPDATE changed, as a re-open would load them: a row
        that keeps a hash of the corpus' dim is replaced in place, a row whose new hash has another length (or is NULL)
        leaves the device and counts in skipped_rows, and a row skipped before that now has the corpus' dim is
        appended.  Ids without a semantic_hashes row change nothing.  The hook for a re-index of a modified file."""
        pairs = [(int(i), None if h is None else bytes(h)) for i, h in pairs]
        if not pairs:
            return
        conn = self.write_connection
        changed: Dict[int, Tuple[Optional[bytes], Optional[bytes]]] = {}      # image_id -> (hash before, last hash set)
        try:
            for image_id, h in pairs:
                old = conn.execute("SELECT hash FROM semantic_hashes WHERE image_id = ?", (image_id,)).fetchone()
                if conn.execute("UPDATE semantic_hashes SET hash = ? WHERE image_id = ?", (h, image_id)).rowcount:
                    changed[image_id] = (changed[image_id][0] if image_id in changed else old[0], h)
            conn.commit()
        except Exception:
            conn.rollback()
            raise
        if self.corpus is None or not changed:
            return
        dim = self.corpus.dim
        fits = lambda h: h is not None and len(h) == dim                            # noqa: E731
        replace = [(i, new) for i, (old, new) in changed.items() if fits(old) and fits(new)]
        leave = [i for i, (old, new) in changed.items() if fits(old) and not fits(new)]
        enter = [(i, new) for i, (old, new) in changed.items() if not fits(old) and fits(new)]
        if leave:
            self.skipped_rows += self.corpus.remove(np.array(leave, np.int64))
        for part, op in ((replace, self.corpus.replace), (enter, self.corpus.append)):
            if part:
                op(np.array([i for i, _ in part], np.int64), np.frombuffer(b"".join(h for _, h in part), np.uint8).reshape(len(part), dim))
        self.skipped_rows -= len(enter)
