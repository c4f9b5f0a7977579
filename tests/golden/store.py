"""On-disk format of the golden fixtures: one fixture (a dict whose list-valued sections hold case dicts) is stored as
`<stem>.<part>.pt` files of at most 1,000,000 bytes each, so that no file in the repository exceeds 1 MB. A part holds
(section, case index, field, value) entries; `load` puts them back together into the dict `save` was given, bit for bit."""
import glob
import io
import os

import torch

PART_LIMIT = 1_000_000


def _size(obj) -> int:
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.tell()


def save(fixture: dict, directory: str, stem: str) -> list:
    """Writes `fixture` as parts and returns their paths (parts of an earlier save under the same stem are removed)."""
    entries = []
    for key, value in fixture.items():
        if isinstance(value, list):
            entries.append((key, -1, None, len(value)))             # the section's length (it may be empty)
            entries += [(key, i, field, v) for i, case in enumerate(value) for field, v in case.items()]
        else:
            entries.append((key, None, None, value))
    parts, sizes = [[]], [_size([])]
    for e in entries:
        s = _size(e)
        assert s + _size([]) <= PART_LIMIT, f'one field of {e[0]} alone is {s} bytes'
        if sizes[-1] + s > PART_LIMIT:
            parts.append([])
            sizes.append(_size([]))
        parts[-1].append(e)
        sizes[-1] += s
    for old in glob.glob(os.path.join(directory, f'{stem}.*.pt')):
        os.remove(old)
    paths = []
    for i, part in enumerate(parts):
        path = os.path.join(directory, f'{stem}.{i:02d}.pt')
        torch.save(part, path)
        assert os.path.getsize(path) <= PART_LIMIT, path
        paths.append(path)
    return paths


def load(directory: str, stem: str) -> dict:
    paths = sorted(glob.glob(os.path.join(directory, f'{stem}.*.pt')))
    if not paths:
        raise FileNotFoundError(f'no {stem}.*.pt under {directory}')
    fixture = {}
    for path in paths:
        for key, index, field, value in torch.load(path, weights_only=False):
            if index is None:
                fixture[key] = value
            elif index < 0:
                fixture[key] = [{} for _ in range(value)]
            else:
                fixture[key][index][field] = value
    return fixture
