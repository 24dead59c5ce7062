"""A tiny VQA-like dataset and left-padding collate for the teacher-cache tests: sample i has its own text length, ids
and image features, all fixed by (seed, i), so that a memory sample is the same whenever it is drawn."""
import torch

PAD_ID = 1


class VLSamples(torch.utils.data.Dataset):
    def __init__(self, n, n_vis=8, patch=12, vocab=97, min_txt=2, max_txt=6, seed=0):
        self.n, self.n_vis, self.patch, self.vocab = n, n_vis, patch, vocab
        self.min_txt, self.max_txt, self.seed = min_txt, max_txt, seed

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        g = torch.Generator().manual_seed(self.seed * 100003 + int(i))
        txt = int(torch.randint(self.min_txt, self.max_txt + 1, (1,), generator=g))
        ids = torch.randint(2, self.vocab, (txt,), generator=g)
        return {"input_ids": ids, "pixel_values": torch.randn(self.n_vis, self.patch, generator=g), "id": int(i)}


def collate(items):
    """Left-pads the text to the batch's longest (mask 0, PAD_ID, labels -100), as the reference's collate does."""
    txt = max(len(it["input_ids"]) for it in items)
    ids = torch.full((len(items), txt), PAD_ID, dtype=torch.int64)
    am = torch.zeros((len(items), txt), dtype=torch.int64)
    for b, it in enumerate(items):
        n = len(it["input_ids"])
        ids[b, txt - n:] = it["input_ids"]
        am[b, txt - n:] = 1
    return {"input_ids": ids, "pixel_values": torch.stack([it["pixel_values"] for it in items]), "attention_mask": am,
            "labels": torch.where(am.bool(), ids, torch.full_like(ids, -100)), "ids": [it["id"] for it in items]}
