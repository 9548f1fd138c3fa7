"""Host-side readers of the reference's on-disk formats -> the integer tables the B200 path consumes (SURVEY 8 f2, a13).

The reference keeps pandas frames and dicts of per-news tensors and assembles every minibatch from strings
(`src/dataset.py:17-85`, `src/evaluate.py:51-157`).  Here each file is read ONCE into flat integer arrays:

  news_parsed.tsv        (data_preprocess.py: header `id category subcategory title abstract title_entities
                          abstract_entities`; list columns are Python-list literals)
      -> NewsTable: ids, `title` int64 [N, num_words_title] (+ `abstract` [N, num_words_abstract], `category` /
         `subcategory` [N] on request); the text widths are those the file was written with
  behaviors_parsed.tsv   (data_preprocess.py:77-81: header `user clicked_news candidate_news clicked`)
      -> TrainRows: `cand_rows` int64 [B, 1+K], `hist_rows` int64 [B, num_clicked] -- news-row indices for
         `TrainStep.step_rows` (first 50 clicks, LEFT-padded, dataset.py:69-83; the pad index is row N of
         `NewsTable.token_table_with_pad()`, an all-zero title = the reference's `padding` entry, dataset.py:45-60)
  behaviors.tsv          (raw MIND, no header: impression_id user time clicked_news impressions)
      -> the arguments of `evaluate.EvalHost`: `hist_rows` [I, num_clicked] (-1 = PADDED_NEWS), CSR candidates and labels
         (`"N123-1"` split on '-', evaluate.py:252,261-263; first 50 clicks, left-padded, :117-124)

Duplicate news ids: the first row wins (evaluate.py:197-201) -- `NewsTable.row_of`.
"""
from __future__ import annotations

import csv
import json
from dataclasses import dataclass, field

import numpy as np

TEXT_COLUMNS = ("title", "abstract")
ELEMENT_COLUMNS = ("category", "subcategory")


@dataclass
class NewsTable:
    ids: list
    columns: dict                      # name -> int64 array ([N, L] for text columns, [N] for element columns)
    row_of: dict = field(default_factory=dict)

    def __post_init__(self):
        for i, nid in enumerate(self.ids):
            self.row_of.setdefault(nid, i)          # first occurrence wins

    def __len__(self):
        return len(self.ids)

    @property
    def title(self):
        return self.columns["title"]

    def token_table_with_pad(self, column="title"):
        """[N + 1, L]: the column plus an all-zero row (index N) that padded history slots point to."""
        c = self.columns[column]
        return np.concatenate([c, np.zeros((1,) + c.shape[1:], dtype=c.dtype)])


def load_news_parsed(path, attributes=("title",)) -> NewsTable:
    """`news_parsed.tsv` -> NewsTable with the requested attribute columns (`config.dataset_attributes['news']`)."""
    for a in attributes:
        if a not in TEXT_COLUMNS + ELEMENT_COLUMNS:
            raise ValueError(f"unsupported news attribute {a!r} (supported: {TEXT_COLUMNS + ELEMENT_COLUMNS})")
    ids, cols = [], {a: [] for a in attributes}
    with open(path, newline="") as f:
        reader = csv.DictReader(f, delimiter="\t", quoting=csv.QUOTE_NONE)
        missing = [a for a in ("id",) + tuple(attributes) if a not in (reader.fieldnames or [])]
        if missing:
            raise KeyError(f"{path}: missing columns {missing}")
        for row in reader:
            ids.append(row["id"])
            for a in attributes:
                cols[a].append(json.loads(row[a]) if a in TEXT_COLUMNS else int(row[a]))
    out = {}
    for a, v in cols.items():
        arr = np.asarray(v, dtype=np.int64)
        if a in TEXT_COLUMNS and arr.ndim != 2:
            raise ValueError(f"{path}: column {a!r} must hold equally long token lists")
        out[a] = arr.reshape(len(ids), -1) if a in TEXT_COLUMNS else arr.reshape(len(ids))
    return NewsTable(ids, out)


@dataclass
class TrainRows:
    cand_rows: np.ndarray              # int64 [B, 1+K]
    hist_rows: np.ndarray              # int64 [B, num_clicked]
    clicked: np.ndarray                # int8  [B, 1+K]  (the 0/1 labels of the candidates; NRMS trains with label 0)
    users: list


def load_behaviors_parsed(path, news: NewsTable, num_clicked=50) -> TrainRows:
    """`behaviors_parsed.tsv` -> index-only training samples (what `BaseDataset.__getitem__` builds per sample,
    dataset.py:62-85): candidate rows, the FIRST `num_clicked` clicked rows left-padded with the pad row (index N)."""
    pad = len(news)
    cand, hist, clicked, users = [], [], [], []
    with open(path, newline="") as f:
        reader = csv.DictReader(f, delimiter="\t", quoting=csv.QUOTE_NONE)
        for row in reader:
            c = [news.row_of[x] for x in row["candidate_news"].split()]
            h = [news.row_of[x] for x in (row["clicked_news"] or "").split()[:num_clicked]]
            cand.append(c)
            hist.append([pad] * (num_clicked - len(h)) + h)
            clicked.append([int(x) for x in row["clicked"].split()])
            users.append(row["user"])
    width = {len(c) for c in cand}
    if len(width) > 1:
        raise ValueError(f"{path}: samples with different numbers of candidates {sorted(width)}")
    return TrainRows(np.asarray(cand, dtype=np.int64).reshape(len(cand), -1),
                     np.asarray(hist, dtype=np.int64).reshape(len(hist), num_clicked),
                     np.asarray(clicked, dtype=np.int8).reshape(len(clicked), -1), users)


@dataclass
class EvalRows:
    hist_rows: np.ndarray              # int64 [I, num_clicked], -1 = PADDED_NEWS
    cand_offsets: np.ndarray           # int64 [I + 1]
    cand_rows: np.ndarray              # int64 [sum C]
    labels: np.ndarray                 # int8  [sum C]
    impression_ids: list
    clicked_news_strings: list         # the reference's user key (evaluate.py:218,256)


def load_behaviors(path, news: NewsTable, num_clicked=50, max_count=None) -> EvalRows:
    """Raw `behaviors.tsv` -> the impression tables of `evaluate.EvalHost` (evaluate.py:111-124, 127-157, 245-265).
    `max_count`: the reference stops BEFORE the max_count-th impression (`count == max_count: break`, :247-249)."""
    hist, offs, rows, labels, imp_ids, keys = [], [0], [], [], [], []
    with open(path, newline="") as f:
        for n, rec in enumerate(csv.reader(f, delimiter="\t", quoting=csv.QUOTE_NONE), 1):
            if max_count is not None and n == max_count:
                break
            impression_id, _user, _time, clicked_news, impressions = rec[:5]
            clicked_news = clicked_news if clicked_news else " "          # fillna(' ') of the reference
            h = [news.row_of[x] for x in clicked_news.split()[:num_clicked]]
            hist.append([-1] * (num_clicked - len(h)) + h)
            for item in impressions.split():
                nid, lab = item.split("-")
                rows.append(news.row_of[nid])
                labels.append(int(lab))
            offs.append(len(rows))
            imp_ids.append(impression_id)
            keys.append(clicked_news)
    return EvalRows(np.asarray(hist, dtype=np.int64).reshape(len(hist), num_clicked), np.asarray(offs, dtype=np.int64),
                    np.asarray(rows, dtype=np.int64), np.asarray(labels, dtype=np.int8), imp_ids, keys)
