"""Collections whose chunks carry allowed_users, for the ACL tests (tests/test_host_acl.py, tests/test_gpu_acl.py):
random ACL sets of every kind (None, [], one user, overlapping groups) over several folders, and the brute-force
predicate the search results are held to."""
from __future__ import annotations

import numpy as np

USERS = [f"u{i}@x.org" for i in range(24)]
GROUPS = [f"group-{i}" for i in range(8)]


def acl_choices(n_sets: int, seed: int) -> list:
    """n_sets allowed_users values: None, [], single users and overlapping user + group lists."""
    rng = np.random.RandomState(seed)
    out = [None, [], [USERS[0]], [GROUPS[0]]]
    pool = USERS + GROUPS
    while len(out) < n_sets:
        k = int(rng.randint(1, 6))
        out.append(sorted(rng.choice(pool, size=k, replace=False).tolist()))
    return out


def principal_lists(n: int, seed: int) -> list:
    """Callers: empty lists, unknown names, one user, a user with groups."""
    rng = np.random.RandomState(seed)
    out = [[], ["nobody@x.org"], [USERS[0]], [USERS[1], GROUPS[0], GROUPS[1]]]
    while len(out) < n:
        k = int(rng.randint(0, 4))
        p = rng.choice(USERS, size=1).tolist() + rng.choice(GROUPS, size=k, replace=False).tolist()
        if rng.rand() < 0.3:
            p.append("stranger@y.org")
        out.append(p)
    return out


def visible(allowed_users, principals) -> bool:
    """The ACL semantics, stated once more independently of the library and the oracle."""
    if allowed_users is None:
        return True
    return len(set(allowed_users) & set(principals)) > 0


def make_chunks(metadata_cls, n_files: int, chunks_per_file: int, dim: int, n_folders: int, acls: list, seed: int,
                vocab: int = 4000):
    """(chunks, sparse_vectors) for store_chunks: files spread over n_folders folders under three index folders, each
    file with one ACL of ``acls`` and timestamps that are sometimes missing."""
    rng = np.random.RandomState(seed)
    chunks, sparse = [], []
    for f in range(n_files):
        k = f % n_folders
        index_folder = f"root{k % 3}"
        folder = f"{index_folder}/folder{k:03d}"
        acl = acls[int(rng.randint(len(acls)))]
        created = None if rng.rand() < 0.1 else int(1420070400 + rng.randint(0, 300_000_000))
        modified = None if rng.rand() < 0.1 else int(1420070400 + rng.randint(0, 300_000_000))
        for c in range(chunks_per_file):
            m = metadata_cls(f"{folder}/file{f:05d}.txt", folder, index_folder, f"file{f:05d}.txt", c, chunks_per_file,
                             100 * c, 100 * c + 99, "2025-01-01T00:00:00", source_created_at=created,
                             source_modified_at=modified, allowed_users=None if acl is None else list(acl))
            chunks.append((f"text {f} {c}", rng.standard_normal(dim).astype(np.float32).tolist(), m))
            nnz = int(rng.randint(1, 12))
            idx = rng.choice(vocab, size=nnz, replace=False)
            sparse.append((idx.tolist(), rng.uniform(0.1, 3.0, nnz).tolist()))
    return chunks, sparse


def filter_specs(folders: list, n: int, seed: int) -> list:
    """n _build_filter keyword sets: none, each folder clause kind and date ranges on both fields."""
    rng = np.random.RandomState(seed)
    specs = [{}]
    while len(specs) < n:
        kw = {}
        kind = rng.randint(5)
        if kind == 0:
            kw["folder_filter"] = folders[rng.randint(len(folders))]
        elif kind == 1:
            kw["include_folders"] = sorted(rng.choice(folders, size=rng.randint(1, len(folders)), replace=False).tolist())
        elif kind == 2:
            kw["exclude_folders"] = sorted(rng.choice(folders, size=rng.randint(1, 4), replace=False).tolist())
            if rng.rand() < 0.5:
                kw["exclude_index_folders"] = ["root%d" % rng.randint(3)]
        if kind == 3 or rng.rand() < 0.4:
            lo = 1420070400 + int(rng.randint(0, 200_000_000))
            kw["date_start"], kw["date_end"] = lo, lo + int(rng.randint(20_000_000, 200_000_000))
            kw["date_field"] = ["created", "modified", None][rng.randint(3)]
        specs.append(kw)
    return specs
