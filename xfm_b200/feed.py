"""Batch feeder: the loader half of SURVEY.md §8 f4 — everything between a decoded crop / a caption string and the tensors
`XFM.forward` takes on the device.

Host half (bit-exact restatements of the reference's sample and batch assembly, same `random` call order so that a seeded
run produces the reference's batches):
  * `TextMasker`              dataset/pretrain_dataset.py:60-150  (TextMaskingGenerator: n-gram / whole-word MLM masking)
  * `pre_caption`             dataset/utils.py:38-66
  * `TextPreprocessor`        dataset/pretrain_dataset.py:264-300 (image-text) and :690-726 (text-only corpus)
  * `LineShards`, `split_shard`  dataset/dist_dataset.py:44-94 (files sharded over ranks, then DataLoader workers; shuffles)
  * `ImageTextStream`         dataset/pretrain_dataset.py:225-262, :368-394 (JSON line -> decoded image + text sample)
  * `region_image_atts`       dataset/pretrain_dataset.py:577-592 (box -> patch mask with token 0 always on)
  * `RegionSampler`           dataset/pretrain_dataset.py:445-575 (random crop around a region, careful hflip, per-region texts,
                              patch masks and cxcywh targets; the pixel work stays with the caller between the two phases)
  * `collate`, `region_collate`  dataset/pretrain_dataset.py:302-312, :594-643 (`idx_to_group_img`, fixed-size region batches)
  * `vqa_collate`             dataset/__init__.py:200-208
  * `pre_question`, `retrieval_image_index`, `retrieval_eval_index`, `nlvr_label`, `vqa_train_sample`
                              the sample logic of the fine-tuning loaders (dataset/utils.py:22-35, retrieval_dataset.py:18-57,
                              nlvr_dataset.py:38-43, vqa_dataset.py:44-125): `idx`, txt2img / img2txt, answer weights

  * `ImageTextJsonDataset`, `ImageJsonDataset`, `RegionTextJsonDataset`, `TextJsonDataset`
                              the four IterableDatasets of dataset/pretrain_dataset.py assembled from the pieces above: same
                              constructor arguments, configuration keys, samples and `collate_fn`
  * `RandAugmentSampler`, `channel_table`  dataset/randaugment.py:13-70,129-135,215-340 (which operations fire with which
                              arguments; the four look-up-table operations.  The cv2 warps / filter stay with the caller)

Device half:
  * `to_uint8_hwc`            replaces the `ToTensor(), normalize` tail of every Compose in dataset/__init__.py:26-68: the
                              worker hands over the crop as uint8 [H, W, 3]
  * `DeviceFeeder`            pinned double-buffered staging, host->device copies on a side stream `depth` batches ahead, and
                              `xfm_image_u8_to_f32` (csrc/feed.cu) doing ToTensor + Normalize (+ hflip) on the GPU: a 224-px
                              batch of 96 crosses PCIe as 14.5 MB instead of 57.8 MB and the result is bit-identical to the CPU
                              transform.

  * `crop_resize`             `RandomResizedCrop(BICUBIC)` / `Resize(BICUBIC)` (dataset/__init__.py:28-30,63-67) and the region
                              loader's crop + resize (pretrain_dataset.py:470-483) on the GPU for ragged uint8 images:
                              Pillow's fixed-point separable resampler, tap tables from the host (`pillow_bicubic_taps`),
                              integer passes in `xfm_resize_bicubic_u8`; bit-identical to PIL.  Complete for the evaluation
                              transform (decode -> resize -> normalize); the training Compose keeps RandAugment (cv2, on the
                              host) between crop and ToTensor, so there it is an option for loaders that augment after it.

  * `decode_jpeg`, `decode_crop_resize`  baseline JPEG decode on the GPU (`xfm_jpeg_plan` on the host, `xfm_jpeg_decode`:
                              Huffman, ISLOW IDCT, fancy upsampling, YCbCr -> RGB), bit-identical to
                              `Image.open(f).convert("RGB")`; other files (progressive, CMYK, PNG, ...) are decoded by Pillow
                              into the same buffer.  With `crop_resize`'s device half, the evaluation transform runs from file
                              bytes to the normalized tensor on the GPU.  `jpeg_size` reads a file's size from its header.

RandAugment stays CPU work in the DataLoader workers (DESIGN §7).  There is no CPU path for the device half:
`DeviceFeeder`, `crop_resize` and `decode_jpeg` raise without a CUDA device.
"""
import math
import random as _random
import re

import torch

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)   # dataset/__init__.py:26
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)
PAD_MASK = -100                                   # pretrain_dataset.py:195: the MLM loss ignores it


# ------------------------------------------------------------------------------------------------------------ text side
class TextMasker:
    """MLM position sampling and token corruption (pretrain_dataset.py:60-150).

    `vocab`: a tokenizer (anything with get_vocab / cls_token / mask_token) or a (id2token, cls_token, mask_token) triple.
    `rng`: an object with shuffle / random / randint — the `random` module by default, because the reference draws from
    the process-global generator (`from random import randint, shuffle`), so `random.seed(s)` reproduces its stream.
    The draws happen in the reference's order: one shuffle of the candidate positions; per visited position one
    random() for the n-gram decision (only when skipgram_prb > 0 and skipgram_size >= 2) followed by randint(2, size)
    when it fires; one shuffle if whole-word / n-gram expansion overshot; per kept position random() < 0.8 -> mask token,
    else random() < 0.5 -> randint over the vocabulary, else unchanged."""

    def __init__(self, vocab, mask_prob, mask_max, skipgram_prb=0.2, skipgram_size=3, mask_whole_word=True, use_roberta=False,
                 rng=None):
        if hasattr(vocab, "get_vocab"):
            table = vocab.get_vocab()
            self.id2token = {i: w for w, i in table.items()}
            self.cls_token, self.mask_token = vocab.cls_token, vocab.mask_token
        else:
            id2token, self.cls_token, self.mask_token = vocab
            self.id2token = dict(enumerate(id2token)) if not isinstance(id2token, dict) else id2token
        n = len(self.id2token)
        if any(i not in self.id2token for i in range(n)):
            raise ValueError("TextMasker: vocabulary ids must be dense 0..V-1 (pretrain_dataset.py:67-68)")
        self.vocab_size = n
        self.mask_prob, self.mask_max = mask_prob, mask_max
        self.skipgram_prb, self.skipgram_size = skipgram_prb, skipgram_size
        self.mask_whole_word, self.use_roberta = mask_whole_word, use_roberta
        self.rng = rng if rng is not None else _random

    def _word_span(self, tokens, st, end):
        """Grow [st, end) to word boundaries: byte-level BPE marks a word START with 'Ġ', WordPiece a CONTINUATION with
        '##' (pretrain_dataset.py:102-118, including its asymmetric lower bounds 1 and 0)."""
        n = len(tokens)
        if self.use_roberta:
            while st > 1 and tokens[st][0] != "Ġ":
                st -= 1
            while end < n and tokens[end][0] != "Ġ":
                end += 1
        else:
            while st >= 0 and tokens[st].startswith("##"):
                st -= 1
            while end < n and tokens[end].startswith("##"):
                end += 1
        return st, end

    def __call__(self, tokens):
        """tokens: list of token strings starting with the cls token; corrupted IN PLACE.  Returns (tokens, masked_pos)."""
        rng = self.rng
        if tokens[0] != self.cls_token:
            raise AssertionError("TextMasker: tokens must start with the cls token")
        budget = min(self.mask_max, max(1, int(round(len(tokens) * self.mask_prob))))
        order = list(range(1, len(tokens)))
        rng.shuffle(order)
        last = max(order)
        ngrams = self.skipgram_prb > 0 and self.skipgram_size >= 2
        chosen = set()                    # a set, like the reference: list(chosen) below inherits CPython's set order
        for pos in order:
            if len(chosen) >= budget:
                break
            if pos in chosen:
                continue
            width = rng.randint(2, self.skipgram_size) if (ngrams and rng.random() < self.skipgram_prb) else 1
            st, end = (self._word_span(tokens, pos, pos + width) if self.mask_whole_word else (pos, pos + width))
            for mp in range(st, end):
                if not 0 < mp <= last:
                    break
                chosen.add(mp)
        masked_pos = list(chosen)
        if len(masked_pos) > budget:
            rng.shuffle(masked_pos)
            masked_pos = masked_pos[:budget]
        for pos in masked_pos:
            if rng.random() < 0.8:
                tokens[pos] = self.mask_token
            elif rng.random() < 0.5:
                tokens[pos] = self.id2token[rng.randint(0, self.vocab_size - 1)]
        return tokens, masked_pos


_PUNCT = re.compile(r"([,.'!?\"()*#:;~])")
_SPACES = re.compile(r"\s{2,}")


def pre_caption(caption, max_words):
    """dataset/utils.py:38-66: lower-case, punctuation -> space, '-' and '/' -> space, '<person>' -> 'person', runs of
    white space collapsed, stripped, truncated to max_words; an empty result is an error."""
    raw = caption
    c = _PUNCT.sub(" ", caption.lower()).replace("-", " ").replace("/", " ").replace("<person>", "person")
    c = _SPACES.sub(" ", c).rstrip("\n").strip(" ")
    words = c.split(" ")
    if len(words) > max_words:
        c = " ".join(words[:max_words])
    if not c:
        raise ValueError(f"pre_caption yields invalid text (raw: {raw})")
    return c


class TextPreprocessor:
    """caption -> (text_ids, text_atts, text_ids_masked, masked_pos, masked_ids), python int lists padded to max_tokens /
    max_masks (pretrain_dataset.py:264-300; `corpus=True`: the text-only stream of :690-726, which skips pre_caption and
    splits pre-tokenized text on spaces)."""

    def __init__(self, tokenizer, masker, max_tokens, max_masks, max_words=None, tokenized=False, language_chosen=None,
                 corpus=False, add_eos=True):
        self.tokenizer, self.masker = tokenizer, masker
        self.max_tokens, self.max_masks, self.max_words = max_tokens, max_masks, max_words
        self.tokenized, self.language_chosen, self.corpus, self.add_eos = tokenized, language_chosen, corpus, add_eos
        self.cls_token, self.eos_token = tokenizer.cls_token, tokenizer.sep_token
        self.pad_token_id = tokenizer.pad_token_id

    def tokens_of(self, text):
        if self.corpus:
            if self.tokenized:
                return text.strip().split(" ")
            if self.language_chosen == "zh":
                text = text.replace(" ", "")
            return self.tokenizer.tokenize(text)
        if self.tokenized:      # regions tokenized by BERT earlier: glue the word pieces back before re-tokenizing
            text = text.strip().replace(" ##", "")
        if self.language_chosen == "zh":
            text = text.replace(" ", "")
        return self.tokenizer.tokenize(pre_caption(text, self.max_words))

    def preprocess(self, text):
        L = self.max_tokens
        tokens = [self.cls_token] + self.tokens_of(text)[:L - 1]
        if self.add_eos:
            tokens = tokens[:L - 1] + [self.eos_token]
        n = len(tokens)
        if n < 2:
            raise AssertionError("len(word tokens) < 2")
        ids = self.tokenizer.convert_tokens_to_ids(tokens)
        corrupted, masked_pos = self.masker(list(tokens))
        ids_masked = self.tokenizer.convert_tokens_to_ids(corrupted)
        masked_ids = [ids[p] for p in masked_pos]
        pad, mpad = [self.pad_token_id] * (L - n), self.max_masks - len(masked_ids)
        return (ids + pad, [1] * n + [0] * (L - n), ids_masked + pad, masked_pos + [0] * mpad, masked_ids + [PAD_MASK] * mpad)


def pick_caption(c, language_chosen=None, rng=None):
    """One caption out of a str / list of them / {language: str} (pretrain_dataset.py:206-223): a list costs one
    rng.choice, a multilingual dict another one unless a language is fixed."""
    rng = rng if rng is not None else _random
    if isinstance(c, list):
        c = rng.choice(c)
    if isinstance(c, str):
        return c
    if isinstance(c, dict):
        v = rng.choice(list(c.values())) if language_chosen is None else c[language_chosen]
        if not isinstance(v, str):
            raise AssertionError("caption entry is not a string")
        return v
    raise ValueError(c)


# ---------------------------------------------------------------------------------------------------------- sample streams
def split_shard(data, shard_idx, shard_size):
    """Contiguous shard shard_idx of shard_size (dataset/dist_dataset.py:88-94); fewer items than shards is an error."""
    n = len(data)
    if n < shard_size:
        raise RuntimeError("num:{} < shard size:{}".format(n, shard_size))
    return data[n * shard_idx // shard_size: n * (shard_idx + 1) // shard_size]


class LineShards:
    """Lines of this rank's (and this DataLoader worker's) share of `files` (dataset/dist_dataset.py:44-83, local files): files
    are sharded over ranks unless there is one rank or one file, then over workers; with `shuffle` the rank's list is
    shuffled IN PLACE once per epoch and the worker's list once more (the same list twice without workers), as the reference
    does — the in-place permutation carries over to the next epoch of `repeat`."""

    def __init__(self, files, rank=0, world_size=1, shuffle=False, repeat=False, rng=None, worker_info=None):
        self.files = [f for f in files if f.find("_SUCCESS") < 0]
        self.rank, self.world_size, self.shuffle, self.repeat = rank, world_size, shuffle, repeat
        self.rng = rng if rng is not None else _random
        self.worker_info = worker_info if worker_info is not None else torch.utils.data.get_worker_info

    def __iter__(self):
        mine = self.files if (self.world_size == 1 or len(self.files) == 1) else split_shard(self.files, self.rank, self.world_size)
        while True:
            if self.shuffle:
                self.rng.shuffle(mine)
            info = self.worker_info()
            part = mine if info is None else split_shard(mine, info.id, info.num_workers)
            if self.shuffle:
                self.rng.shuffle(part)
            for path in part:
                with open(path, "r") as reader:
                    yield from reader
            if not self.repeat:
                return


def _open_rgb(ref, is_path):
    import io
    from base64 import b64decode
    from PIL import Image
    return Image.open(ref if is_path else io.BytesIO(b64decode(ref))).convert("RGB")


class ImageTextStream:
    """JSON lines -> (image, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids) samples
    (ImageTextJsonDataset.__iter__, pretrain_dataset.py:225-262; `text=None`: the image-only stream of ImageJsonDataset.__iter__,
    :368-394, which yields (image, None x 5)).  A list of images costs one rng.choice for the prompt prefix and one for the
    image; broken lines are reported through `on_error` and skipped, like the reference's try / except."""

    PREFIX = ("A image of ", "The image contains ", "We can see ", "A picture of ")

    def __init__(self, lines, transform, text, image_key, caption_key=None, is_image_rpath=False, rng=None, on_error=None):
        self.lines, self.transform, self.text = lines, transform, text
        self.image_key, self.caption_key, self.is_image_rpath = image_key, caption_key, is_image_rpath
        self.rng = rng if rng is not None else _random
        self.on_error = on_error

    def _sample(self, ann):
        rng, ref = self.rng, ann[self.image_key]
        several = type(ref) == list
        caption = None
        if self.text is not None:
            prefix = rng.choice(self.PREFIX) if several else ""          # drawn before the caption, as in the reference
            caption = prefix + pick_caption(ann[self.caption_key], self.text.language_chosen, rng)
        if several and not self.is_image_rpath:
            ref = rng.choice(ref)
        image = self.transform(_open_rgb(ref, self.is_image_rpath))
        if self.text is None:
            return (image, None, None, None, None, None)
        if not len(caption):
            raise ValueError({k: v for k, v in ann.items() if k != self.image_key})
        return (image, *self.text.preprocess(caption))

    def __iter__(self):
        import json
        for line in self.lines:
            try:
                ann = json.loads(line)
                if not isinstance(ann, dict):
                    raise AssertionError("ann is not dict")
                if type(ann[self.image_key]) == list and len(ann[self.image_key]) == 0:
                    continue
                yield self._sample(ann)
            except Exception as e:  # noqa: BLE001 — the reference skips any broken sample
                if self.on_error is not None:
                    self.on_error(e)


# ----------------------------------------------------------------------- fine-tuning loaders (BASELINE configs #3 - #5)
def pre_question(question, max_ques_words):
    """dataset/utils.py:22-35: lower-case, punctuation -> space, '-' and '/' -> space, trailing blanks stripped, truncated."""
    q = _PUNCT.sub(" ", question.lower()).replace("-", " ").replace("/", " ").rstrip(" ")
    words = q.split(" ")
    return " ".join(words[:max_ques_words]) if len(words) > max_ques_words else q


def retrieval_image_index(anns):
    """image_id -> dense index in first-appearance order (re_train_dataset, dataset/retrieval_dataset.py:18-25): the `idx`
    of ITC / ITM at fine-tuning time (captions of one image share it)."""
    index = {}
    for ann in anns:
        index.setdefault(ann["image_id"], len(index))
    return index


def retrieval_eval_index(anns, max_words=30):
    """Evaluation split -> (texts, images, txt2img, img2txt) (re_eval_dataset, dataset/retrieval_dataset.py:44-57): captions
    cleaned with pre_caption and numbered in file order; what `retrieval_eval.itm_eval` scores against."""
    texts, images, txt2img, img2txt = [], [], {}, {}
    for img_id, ann in enumerate(anns):
        images.append(ann["image"])
        img2txt[img_id] = []
        for caption in ann["caption"]:
            txt2img[len(texts)] = img_id
            img2txt[img_id].append(len(texts))
            texts.append(pre_caption(caption, max_words))
    return texts, images, txt2img, img2txt


def nlvr_label(ann):
    """'True' / 'False' -> 1 / 0 (dataset/nlvr_dataset.py:38-43)."""
    if ann["label"] == "True":
        return 1
    if ann["label"] == "False":
        return 0
    raise ValueError(f"unsupported label: {ann['label']}")


def vqa_mentions_side(question, answer):
    """dataset/vqa_dataset.py:44-62: 'left' / 'right' in the question or any answer — such samples are never mirrored."""
    answers = answer if isinstance(answer, list) else [answer]
    return any(("left" in s) or ("right" in s) for s in [question] + answers)


def vqa_train_sample(ann, max_ques_words=30, rng=None):
    """One VQA training annotation -> (hflip, question, answers, weights) (dataset/vqa_dataset.py:64-125, minus the pixels):
    one rng.random() decides the mirror (suppressed for left / right samples), Visual-Genome answers weigh 0.5, VQA answers
    their share among the annotators, in first-appearance order."""
    rng = rng if rng is not None else _random
    hflip = rng.random() < 0.5 and not vqa_mentions_side(ann["question"], ann["answer"])
    question = pre_question(ann["question"], max_ques_words)
    if ann.get("dataset") == "vg":
        return hflip, question, [ann["answer"]], [0.5]
    share = {}
    for a in ann["answer"]:
        share[a] = share[a] + 1 / len(ann["answer"]) if a in share else 1 / len(ann["answer"])
    return hflip, question, list(share.keys()), list(share.values())


# ---------------------------------------------------------------------------------------------------------- region side
def region_image_atts(x, y, w, h, patch_size, num_patch):
    """Pixel box (after crop / flip / resize) -> 0/1 list of length 1 + num_patch^2: token 0 always on, then every patch the
    box touches, at least one per axis (pretrain_dataset.py:577-592)."""
    x0 = min(math.floor(x / patch_size), num_patch - 1)
    x1 = max(x0 + 1, min(math.ceil((x + w) / patch_size), num_patch))
    y0 = min(math.floor(y / patch_size), num_patch - 1)
    y1 = max(y0 + 1, min(math.ceil((y + h) / patch_size), num_patch))
    atts = [0] * (1 + num_patch * num_patch)
    atts[0] = 1
    for i in range(y0, y1):
        row = num_patch * i + 1
        for j in range(x0, x1):
            if not 0 < row + j <= num_patch * num_patch:
                raise AssertionError(f"patch index out of range, index: {row + j}")
            atts[row + j] = 1
    return atts


class RegionSampler:
    """One region-annotated image -> the per-region samples of pretrain_dataset.py:445-575, in two phases because the pixel
    work (crop, flip, resize, box_transform — whose RandAugment draws from the same global generator) sits between them:

        plan = sampler.plan(ann, W, H)            # random crop containing one region + the flip decision
        image = box_transform(resize(maybe_hflip(pil.crop(plan.crop_box))))
        sample = sampler.finish(ann, plan, image)  # texts, patch masks, cxcywh targets, is_image flags
    """

    class Plan:
        __slots__ = ("x0", "y0", "w0", "h0", "hflip")

        @property
        def crop_box(self):
            return (self.x0, self.y0, self.x0 + self.w0, self.y0 + self.h0)

    def __init__(self, text, image_res, patch_size, max_regions, min_perc_in_image, careful_hflip=False, rng=None):
        self.text, self.image_res, self.patch_size = text, image_res, patch_size
        if image_res % patch_size:
            raise AssertionError("image_res must be a multiple of patch_size")
        self.num_patch = image_res // patch_size
        self.max_regions, self.min_perc, self.careful_hflip = max_regions, min_perc_in_image, careful_hflip
        self.rng = rng if rng is not None else _random

    @staticmethod
    def _bb(elem):
        x, y, w, h = elem["bb"]
        return int(x), int(y), int(w), int(h)

    @staticmethod
    def mentions_side(ann):
        """'left' / 'right' in any caption of the image or its regions (pretrain_dataset.py:425-443): such images are not
        flipped when careful_hflip is set."""
        def has(e):
            c = e["caption"]
            return any(("left" in s) or ("right" in s) for s in (c if isinstance(c, list) else [c]))
        return ("caption" in ann and has(ann)) or any(has(e) for e in ann["elems"])

    def _caption(self, c):
        return pick_caption(c, self.text.language_chosen, self.rng)

    def plan(self, ann, W, H):
        rng = self.rng
        x, y, w, h = self._bb(rng.choice(ann["elems"]))
        if not (x >= 0 and y >= 0 and x + w <= W and y + h <= H and w > 0 and h > 0):
            raise AssertionError("elem invalid")
        p = self.Plan()
        p.x0, p.y0 = rng.randint(0, math.floor(x)), rng.randint(0, math.floor(y))
        x1, y1 = rng.randint(min(math.ceil(x + w), W), W), rng.randint(min(math.ceil(y + h), H), H)
        p.w0, p.h0 = x1 - p.x0, y1 - p.y0
        if not (p.x0 >= 0 and p.y0 >= 0 and p.x0 + p.w0 <= W and p.y0 + p.h0 <= H and p.w0 > 0 and p.h0 > 0):
            raise AssertionError("elem randomcrop, invalid")
        p.hflip = rng.random() < 0.5 and not (self.careful_hflip and self.mentions_side(ann))
        return p

    def finish(self, ann, plan, image):
        res, left = self.image_res, self.max_regions
        cols = [[] for _ in range(8)]   # ids, atts, ids_masked, masked_pos, masked_ids, image_atts, target_bbox, is_image

        def push(text5, atts, box, flag):
            for c, v in zip(cols, (*text5, atts, box, flag)):
                c.append(v)

        if "caption" in ann:
            push(self.text.preprocess(self._caption(ann["caption"])), [1] * (self.num_patch ** 2 + 1),
                 torch.tensor([0.5, 0.5, 1, 1], dtype=torch.float), 1)
            left -= 1
        x0, y0, W, H = plan.x0, plan.y0, plan.w0, plan.h0
        for elem in self.rng.sample(ann["elems"], len(ann["elems"])):
            if left <= 0:
                break
            x, y, w, h = self._bb(elem)
            xx, yy, xm, ym = max(x0, x), max(y0, y), min(x0 + W, x + w), min(y0 + H, y + h)
            if not (xm > xx and ym > yy and (xm - xx) * (ym - yy) / (w * h) > self.min_perc):
                continue
            x, y, w, h = xx - x0, yy - y0, xm - xx, ym - yy        # the visible part, in crop coordinates
            if plan.hflip:
                x = (W - x) - w
            x, w, y, h = res / W * x, res / W * w, res / H * y, res / H * h
            caption = self._caption(elem["caption"])
            if "attributes" in elem:
                caption = self._caption(elem["attributes"]) + " " + caption
            text5 = self.text.preprocess(caption)
            push(text5, region_image_atts(x, y, w, h, self.patch_size, self.num_patch),
                 torch.tensor([(x + 1 / 2 * w) / res, (y + 1 / 2 * h) / res, w / res, h / res], dtype=torch.float), 0)
            left -= 1
        return ([image] if cols[0] else [], *cols)


def _stack_column(x):
    if x[0] is None:
        return None
    if isinstance(x[0], torch.Tensor):
        return torch.stack(x)
    return torch.tensor(x, dtype=torch.long)


def collate(batch):
    """List of per-sample tuples -> list of batch tensors: tensors stacked, int lists as int64, None kept
    (pretrain_dataset.py:302-312)."""
    return [_stack_column(x) for x in zip(*batch)]


def vqa_collate(batch):
    """[(image, question str, answers [str], weights [float])] -> (images [B, ...], questions, flattened answers, weights as a
    float32 tensor, answers per question) — `vqa_collate_fn`, dataset/__init__.py:200-208 (BASELINE config #5 loader)."""
    images, questions, answers, weights, counts = [], [], [], [], []
    for image, question, ans, w in batch:
        images.append(image)
        questions.append(question)
        answers += ans
        weights += w
        counts.append(len(ans))
    return torch.stack(images, dim=0), questions, answers, torch.Tensor(weights), counts


def region_collate(batch_sample, batch_size, rng=None, warn=print):
    """RegionSampler samples -> [images, idx_to_group_img, text_ids, text_atts, text_ids_masked, masked_pos, masked_ids,
    image_atts, target_bbox, is_image] with exactly batch_size region samples (pretrain_dataset.py:594-643): all images that
    produced at least one sample are stacked, the flattened samples are sub-sampled (or padded by re-sampling, or by
    repetition when fewer than half are there) to the fixed size every rank must have."""
    rng = rng if rng is not None else _random
    images, *cols = (list(c) for c in zip(*batch_sample))
    group, img = [], -1
    for s in cols[0]:
        if len(s):
            img += 1
            group += [img] * len(s)
    n = len(group)
    keep = list(range(n))
    if n >= batch_size:
        keep = rng.sample(keep, batch_size)
    else:
        try:
            extra = rng.sample(keep, batch_size - n)
            keep += extra
            warn("### warning: pad region_batch by sampling, ", len(extra), flush=True)
        except ValueError:
            warn("### warning: pad region_batch by expanding, ", batch_size - n, flush=True)
            keep = (keep * math.ceil(batch_size / n))[:batch_size]
    out = [torch.stack([im for per in images for im in per]), torch.tensor([group[i] for i in keep], dtype=torch.long)]
    for c in cols:
        flat = [v for per in c for v in per]
        out.append(_stack_column([flat[i] for i in keep]))
    return out


# -------------------------------------------------------------------------- the reference's dataset classes, assembled
def list_files(data_path):
    """'dir_or_file[,dir_or_file...]' -> file list (utils/hdfs_io.py:55-79, local paths: a directory contributes
    os.listdir order, a file itself).  hdfs:// paths need the reference's hadoop client and are refused."""
    import os
    files = []
    for folder in data_path.split(","):
        if folder.startswith("hdfs"):
            raise NotImplementedError("xfm_b200.feed reads local files; mount or copy hdfs:// data first")
        if os.path.isdir(folder):
            files.extend(os.path.join(folder, d) for d in os.listdir(folder))
        elif os.path.isfile(folder):
            files.append(folder)
        else:
            print("Path {} is invalid".format(folder), flush=True)
    return files


def _report_broken(enabled):
    import traceback

    def report(e):
        if enabled:
            print("".join(traceback.format_exception(type(e), e, e.__traceback__)))
            print("encounter broken data: %s" % e)
            print("-" * 20, flush=True)
    return report


class _JsonLineDataset(torch.utils.data.IterableDataset):
    """Shared constructor work of the four pre-training datasets (pretrain_dataset.py:154-204,315-365,408-419,645-671):
    file list, rank / worker sharding, tokenizer, masker with the configuration's MLM settings.  `tokenizer=None` builds
    the HuggingFace tokenizer of config['text_encoder'] like `build_tokenizer` (:35-57)."""

    def __init__(self, config, data_path, rank, world_size, shuffle, repeat, tokenizer, section, whole_word):
        super().__init__()
        self.lines = LineShards(list_files(data_path), rank, world_size, shuffle, repeat)
        self.batch_size = config[section]["batch_size"]
        self.tokenized = config[section]["tokenized"]
        self.report = _report_broken(config["print_broken_data"] if "print_broken_data" in config else True)
        self.tokenizer = tokenizer if tokenizer is not None else build_tokenizer(config["text_encoder"])
        self.masker = TextMasker(self.tokenizer, whole_word["mask_prob"], whole_word["max_masks"], config["skipgram_prb"],
                                 config["skipgram_size"], whole_word["mask_whole_word"])


def build_tokenizer(text_encoder):
    """pretrain_dataset.py:35-57: BERT / RoBERTa / XLM-R tokenizer by directory name, with bos / eos aliases filled in."""
    from transformers import BertTokenizer, RobertaTokenizer, XLMRobertaTokenizer
    if any(k in text_encoder for k in ("bert-base-uncased", "bert-large-uncased", "chinese-roberta-wwm-ext")):
        tok = BertTokenizer.from_pretrained(text_encoder)
    elif "xlm-roberta-base" in text_encoder or "xlm-roberta-large" in text_encoder:
        tok = XLMRobertaTokenizer.from_pretrained(text_encoder)
    elif "roberta-base" in text_encoder or "roberta-large" in text_encoder:
        tok = RobertaTokenizer.from_pretrained(text_encoder)
    else:
        raise NotImplementedError(f"tokenizer for {text_encoder}")
    if tok.bos_token is None:
        tok.add_special_tokens({"bos_token": tok.cls_token})
    if tok.eos_token is None:
        tok.add_special_tokens({"eos_token": tok.sep_token})
    return tok


def _mlm_settings(config):
    """Image-text streams take the top-level MLM keys; whole-word masking is forced off unless the encoder is
    bert-{base,large}-uncased, and the change is written back into config like the reference does (:186-189)."""
    if "bert-base-uncased" not in config["text_encoder"] and "bert-large-uncased" not in config["text_encoder"]:
        config["mask_whole_word"] = False
    return dict(mask_prob=config["mask_prob"], max_masks=config["max_masks"], mask_whole_word=config["mask_whole_word"])


class ImageTextJsonDataset(_JsonLineDataset):
    """pretrain_dataset.py:154-312: same constructor arguments and configuration keys (config[config_key]: image_key,
    is_image_rpath, caption_key / aux_caption_key, batch_size, tokenized, optional language_chosen; config: text_encoder,
    mask_prob, max_masks, skipgram_prb, skipgram_size, mask_whole_word, max_words, max_tokens, image_res, patch_size),
    same samples, same `collate_fn`.  Use with `DataLoader(ds, batch_size=ds.batch_size, collate_fn=ds.collate_fn, ...)`."""

    text_stream = True

    def __init__(self, config, data_path, rank=0, world_size=1, shuffle=True, repeat=True, transform=None, add_eos=True,
                 is_aux=False, config_key="images", tokenizer=None):
        super().__init__(config, data_path, rank, world_size, shuffle, repeat, tokenizer, config_key, _mlm_settings(config))
        sec = config[config_key]
        self.image_key, self.is_image_rpath = sec["image_key"], sec["is_image_rpath"]
        self.caption_key = sec["aux_caption_key"] if is_aux else sec["caption_key"]
        self.language_chosen = sec.get("language_chosen")
        if self.language_chosen is not None and not isinstance(self.language_chosen, str):
            raise AssertionError("language_chosen must be a string")
        self.transform, self.image_res, self.patch_size = transform, config["image_res"], config["patch_size"]
        if self.image_res % self.patch_size:
            raise AssertionError("image_res must be a multiple of patch_size")
        self.num_patch = self.image_res // self.patch_size
        self.text = TextPreprocessor(self.tokenizer, self.masker, config["max_tokens"], config["max_masks"], config["max_words"],
                                     tokenized=self.tokenized, language_chosen=self.language_chosen)

    def __iter__(self):
        return iter(ImageTextStream(self.lines, self.transform, self.text if self.text_stream else None, self.image_key,
                                    self.caption_key, self.is_image_rpath, on_error=self.report))

    def collate_fn(self, batch):
        return collate(batch)


class ImageJsonDataset(ImageTextJsonDataset):
    """pretrain_dataset.py:314-407: the image-only stream (ImageNet-style data for MIM): samples are (image, None x 5)."""
    text_stream = False


class RegionTextJsonDataset(ImageTextJsonDataset):
    """pretrain_dataset.py:409-643: one annotated image -> a random crop around one of its regions, mirrored with probability
    1/2 (never when careful_hflip is set and a caption says left / right), resized to image_res (BICUBIC), `box_transform`,
    and up to max_regions (text, patch mask, box) samples; `collate_fn` = the fixed-size region batch."""

    def __init__(self, config, data_path, rank=0, world_size=1, shuffle=True, repeat=True, transform=None, box_transform=None,
                 config_key="regions", tokenizer=None):
        super().__init__(config, data_path, rank=rank, world_size=world_size, shuffle=shuffle, repeat=repeat, transform=transform,
                         config_key=config_key, tokenizer=tokenizer)
        if self.caption_key != "caption":
            raise AssertionError("please follow my data format")
        sec = config[config_key]
        self.box_transform = box_transform
        self.sampler = RegionSampler(self.text, self.image_res, self.patch_size, sec["max_regions"], sec["min_perc_in_image"],
                                     careful_hflip=sec.get("careful_hflip", False))

    def __iter__(self):
        import json
        from PIL import Image
        for line in self.lines:
            try:
                ann = json.loads(line)
                if not isinstance(ann, dict):
                    raise AssertionError("ann is not dict")
                image = _open_rgb(ann[self.image_key], self.is_image_rpath)
                plan = self.sampler.plan(ann, *image.size)
                image = image.crop(plan.crop_box)
                if plan.hflip:
                    image = image.transpose(Image.FLIP_LEFT_RIGHT)
                image = self.box_transform(image.resize((self.image_res, self.image_res), Image.BICUBIC))
                yield self.sampler.finish(ann, plan, image)
            except Exception as e:  # noqa: BLE001 — the reference skips any broken sample
                self.report(e)

    def collate_fn(self, batch_sample):
        return region_collate(batch_sample, self.batch_size)


class TextJsonDataset(_JsonLineDataset):
    """pretrain_dataset.py:645-737: the text-only corpus stream (config['texts']: text_key, batch_size, tokenized, mask_prob,
    max_masks, mask_whole_word, max_words, max_tokens); samples are the five text lists."""

    def __init__(self, config, data_path, rank=0, world_size=1, shuffle=True, repeat=True, tokenizer=None):
        sec = config["texts"]
        super().__init__(config, data_path, rank, world_size, shuffle, repeat, tokenizer, "texts", sec)
        self.text_key = sec["text_key"]
        self.text = TextPreprocessor(self.tokenizer, self.masker, sec["max_tokens"], sec["max_masks"], sec["max_words"],
                                     tokenized=self.tokenized, corpus=True)

    def __iter__(self):
        import json
        for line in self.lines:
            try:
                ann = json.loads(line)
                if not isinstance(ann, dict):
                    raise AssertionError("ann is not dict")
                yield self.text.preprocess(ann[self.text_key].strip())
            except Exception as e:  # noqa: BLE001
                self.report(e)

    def collate_fn(self, batch):
        return collate(batch)


# ------------------------------------------------------------------------------------------- RandAugment (host logic)
class RandAugmentSampler:
    """Which operations `RandomAugment(N, M, augs=...)` applies to one image, and with which arguments
    (dataset/randaugment.py:215-340): N names drawn with replacement by ONE rng.choice, then per name one rng.random() — the
    operation is skipped when it exceeds 0.5 — and, for the geometric operations, one more rng.random() for the sign of the
    magnitude (Rotate negates below 0.5, the shears / translations above).  `rng` defaults to `numpy.random`, the generator
    the reference draws from.  Magnitudes at level M of 10: enhancement factor 0.1 + 1.8 M/10, shear 0.3 M/10, translation
    10 M/10 pixels, rotation 30 M/10 degrees, solarize threshold int(256 M/10), posterize bits int(4 M/10); fill (128, 128, 128)."""

    MAX_LEVEL, TRANSLATE, FILL = 10, 10, (128, 128, 128)
    ALL = ("Identity", "AutoContrast", "Equalize", "Rotate", "Solarize", "Color", "Contrast", "Brightness", "Sharpness", "ShearX",
           "TranslateX", "TranslateY", "Posterize", "ShearY")

    def __init__(self, N=2, M=10, augs=None, rng=None):
        import numpy as np
        self.N, self.M, self.augs = N, M, list(augs) if augs else list(self.ALL)
        self.rng = rng if rng is not None else np.random

    def _args(self, name):
        rng, frac = self.rng, self.M / self.MAX_LEVEL
        if name in ("Identity", "AutoContrast", "Equalize"):
            return ()
        if name in ("Color", "Contrast", "Brightness", "Sharpness"):
            return (frac * 1.8 + 0.1,)
        if name == "Solarize":
            return (int(frac * 256),)
        if name == "Posterize":
            return (int(frac * 4),)
        if name == "Rotate":
            level = frac * 30
            return (-level if rng.random() < 0.5 else level, self.FILL)
        level = frac * 0.3 if name in ("ShearX", "ShearY") else frac * float(self.TRANSLATE)
        return (-level if rng.random() > 0.5 else level, self.FILL)

    def sample(self):
        """[(name, args)] of the operations that fire, in application order."""
        fired = []
        for name in self.rng.choice(self.augs, self.N):
            if self.rng.random() > 0.5:
                continue
            fired.append((str(name), self._args(str(name))))
        return fired


def channel_table(ch, name, args=()):
    """The 256-entry uint8 look-up table that Identity / AutoContrast / Equalize / Brightness apply to one channel `ch`
    (uint8 [H, W]) of an image (dataset/randaugment.py:13-70,129-135; cutoff 0): these four of the box_transform's five
    operations (dataset/__init__.py:57-61) are per-channel tables of the channel's own histogram, so they compose with each
    other — and with ToTensor + Normalize — into ONE table per image and channel."""
    import numpy as np
    ident = np.arange(256)
    if name == "Identity":
        table = ident
    elif name == "Brightness":
        return (np.arange(256, dtype=np.float32) * args[0]).clip(0, 255).astype(np.uint8)
    elif name == "AutoContrast":
        high, low = ch.max(), ch.min()
        if high <= low:
            table = ident
        else:
            # the reference negates `low` as a numpy uint8 scalar (randaugment.py:36 `offset = -low * scale`), which wraps to
            # 256 - low: for low > 0 the table saturates early instead of stretching [low, high] to [0, 255].  Kept as is —
            # this restates what the reference's loaders feed the model, not PIL's autocontrast.
            scale = 255 / (int(high) - int(low))
            table = (ident * scale + ((256 - int(low)) % 256) * scale).clip(0, 255)
    elif name == "Equalize":
        hist = np.bincount(ch.reshape(-1), minlength=256).astype(np.float32)
        step = np.sum(hist[hist != 0][:-1]) // 255
        if step == 0:
            table = ident
        else:
            shifted = np.empty_like(hist)
            shifted[0], shifted[1:] = step // 2, hist[:-1]
            table = np.cumsum(shifted) // step
    else:
        raise ValueError(f"{name} is not a per-channel table operation")
    return np.asarray(table).clip(0, 255).astype(np.uint8)


def apply_channel_tables(img, name, args=()):
    """img uint8 [H, W, 3] -> the operation applied channel by channel (table[ch] per channel)."""
    import numpy as np
    return np.stack([channel_table(img[:, :, c], name, args)[img[:, :, c]] for c in range(img.shape[2])], axis=2)


# ---------------------------------------------------------------------------------------------------------- device side
def to_uint8_hwc(pic):
    """The transform that replaces `transforms.ToTensor(), normalize` at the end of a Compose: PIL RGB image or uint8
    ndarray [H, W, 3] -> torch.uint8 [H, W, 3] (no arithmetic; DeviceFeeder finishes the transform on the GPU)."""
    import numpy as np

    a = np.asarray(pic)
    if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
        raise ValueError(f"to_uint8_hwc: expected an RGB uint8 image, got {a.dtype} {a.shape}")
    return torch.from_numpy(np.ascontiguousarray(a) if a.flags.writeable else np.array(a))


# ------------------------------------------------------------------------------------- crop + bicubic resize (Pillow-exact)
_PRECISION_BITS = 32 - 8 - 2      # Pillow, src/libImaging/Resample.c: 8-bit pixels, 22 fractional bits, int32 accumulator


def pillow_bicubic_taps(in_size, out_size):
    """The tap tables Pillow builds for `resize(..., BICUBIC)` of an axis of in_size pixels to out_size
    (precompute_coeffs with box (0, in_size) + normalize_coeffs_8bpc; bicubic with a = -0.5, support 2 * max(scale, 1)):
    (first int32 [out], count int32 [out], taps int32 [out, ksize]) with output = clip8((2^21 + sum taps * pixels) >> 22).
    float64 arithmetic in Pillow's operation order, so the integers are Pillow's."""
    import numpy as np

    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    center = 0.0 + (np.arange(out_size, dtype=np.float64) + 0.5) * scale
    first = np.maximum((center - support + 0.5).astype(np.int64), 0)          # C's (int) cast: truncation
    count = np.minimum((center + support + 0.5).astype(np.int64), in_size) - first
    k = np.arange(ksize)[None, :]
    x = np.abs((k + first[:, None] - center[:, None] + 0.5) * (1.0 / fs))
    a = -0.5
    w = np.where(x < 1.0, ((a + 2.0) * x - (a + 3.0)) * x * x + 1, np.where(x < 2.0, (((x - 5) * x + 8) * x - 4) * a, 0.0))
    live = k < count[:, None]
    w = np.where(live, w, 0.0)
    total = np.zeros(out_size)
    for j in range(ksize):            # Pillow sums the taps left to right
        total = total + w[:, j]
    w = np.where(live & (total[:, None] != 0.0), w / np.where(total == 0.0, 1.0, total)[:, None], w)
    q = w * (1 << _PRECISION_BITS)
    taps = np.where(w < 0, (-0.5 + q).astype(np.int64), (0.5 + q).astype(np.int64)).astype(np.int32)
    return first.astype(np.int32), count.astype(np.int32), taps


def bicubic_ksize(in_size, out_size):
    """Width of Pillow's tap table for this axis: ceil(2 * max(in / out, 1)) * 2 + 1."""
    return int(math.ceil(2.0 * max(float(in_size) / out_size, 1.0))) * 2 + 1


def crop_resize_plan(sizes, boxes, out_h, out_w, taps=True):
    """Host tables for `xfm_resize_bicubic_u8`: sizes [(h, w)] of the packed images, boxes [(x0, y0, x1, y1)] integer crop
    boxes (PIL convention, inside the image).  Returns dict(desc, KH, KV, tmp_bytes, max_rows, src_bytes) and, with
    taps=True, the tap tables hb / hk / vb / vk computed on the host (`xfm_resize_taps` computes the same on the device)."""
    import numpy as np

    B = len(sizes)
    desc = np.zeros((B, 8), dtype=np.int64)
    src_off = tmp_off = 0
    KH = KV = 1
    for b, ((h, w), (x0, y0, x1, y1)) in enumerate(zip(sizes, boxes)):
        if not (0 <= x0 < x1 <= w and 0 <= y0 < y1 <= h):
            raise ValueError(f"crop box {(x0, y0, x1, y1)} is not inside image {b} of size {(h, w)}")
        cw, ch = x1 - x0, y1 - y0
        desc[b] = (src_off, w, x0, y0, cw, ch, tmp_off, 0)
        KH, KV = max(KH, bicubic_ksize(cw, out_w)), max(KV, bicubic_ksize(ch, out_h))
        src_off += h * w * 3
        tmp_off += ch * out_w * 3
    plan = dict(desc=torch.from_numpy(desc), KH=KH, KV=KV, tmp_bytes=max(tmp_off, 1), src_bytes=src_off,
                max_rows=int(desc[:, 5].max()) if B else 1)
    if taps:
        hb, hk = np.zeros((B, out_w, 2), np.int32), np.zeros((B, out_w, KH), np.int32)
        vb, vk = np.zeros((B, out_h, 2), np.int32), np.zeros((B, out_h, KV), np.int32)
        for b in range(B):
            hf, hc, ht = pillow_bicubic_taps(int(desc[b, 4]), out_w)
            vf, vc, vt = pillow_bicubic_taps(int(desc[b, 5]), out_h)
            hb[b, :, 0], hb[b, :, 1], hk[b, :, :ht.shape[1]] = hf, hc, ht
            vb[b, :, 0], vb[b, :, 1], vk[b, :, :vt.shape[1]] = vf, vc, vt
        plan.update(hb=torch.from_numpy(hb), hk=torch.from_numpy(hk), vb=torch.from_numpy(vb), vk=torch.from_numpy(vk))
    return plan


def random_resized_crop_box(width, height, scale=(0.2, 1.0), ratio=(3.0 / 4.0, 4.0 / 3.0), generator=None):
    """The crop box `transforms.RandomResizedCrop(res, scale=scale)` (dataset/__init__.py:28-29,37-38) draws for an image of
    this size, as a PIL box (x0, y0, x1, y1) for `crop_resize`.  torchvision's rule (third party): up to ten attempts of
    area ~ U(scale) * image area and log-aspect ~ U(log ratio), accepted when the box fits, then its corner uniformly; else the
    largest centred box whose aspect is clamped into `ratio`.  The draws are the same torch calls in the same order, so with
    the global generator (generator=None) a seeded run crops exactly what torchvision would."""
    area = height * width
    log_ratio = torch.log(torch.tensor(ratio))
    for _ in range(10):
        target = area * torch.empty(1).uniform_(scale[0], scale[1], generator=generator).item()
        aspect = torch.exp(torch.empty(1).uniform_(log_ratio[0], log_ratio[1], generator=generator)).item()
        w, h = int(round(math.sqrt(target * aspect))), int(round(math.sqrt(target / aspect)))
        if 0 < w <= width and 0 < h <= height:
            y0 = torch.randint(0, height - h + 1, size=(1,), generator=generator).item()
            x0 = torch.randint(0, width - w + 1, size=(1,), generator=generator).item()
            return (x0, y0, x0 + w, y0 + h)
    image_ratio = float(width) / float(height)
    if image_ratio < min(ratio):
        w, h = width, int(round(width / min(ratio)))
    elif image_ratio > max(ratio):
        w, h = int(round(height * max(ratio))), height
    else:
        w, h = width, height
    x0, y0 = (width - w) // 2, (height - h) // 2
    return (x0, y0, x0 + w, y0 + h)


def flipped_crops(images, boxes, flips):
    """Images whose flag is set are replaced by their mirrored crop (and the box by None = whole image): crop -> hflip ->
    resize, the order of the region loader (pretrain_dataset.py:470-483), then is a plain resize of the mirrored crop.  Host
    work: one crop-sized copy per mirrored image."""
    if flips is None:
        return list(images), list(boxes)
    out_images, out_boxes = [], []
    for im, bx, fl in zip(images, boxes, flips):
        if fl:
            x0, y0, x1, y1 = (0, 0, im.shape[1], im.shape[0]) if bx is None else bx
            im, bx = im[y0:y1, x0:x1].flip(1).contiguous(), None
        out_images.append(im)
        out_boxes.append(bx)
    return out_images, out_boxes


def crop_resize(images, boxes, out_h, out_w, device=None, taps="device", flips=None):
    """images: list of uint8 [h, w, 3] host tensors (decoded RGB, any sizes); boxes: integer crop boxes (x0, y0, x1, y1) or
    None = the whole image.  Returns uint8 [B, out_h, out_w, 3] on the device, bit-identical to
    PIL `image.crop(box).resize((out_w, out_h), BICUBIC)` — i.e. to `RandomResizedCrop` / `Resize` with
    InterpolationMode.BICUBIC once the crop box is drawn.  `lib.image_u8_to_f32` finishes the transform.  taps="device"
    (default) builds Pillow's tap tables on the GPU (`xfm_resize_taps`); taps="host" computes them in numpy (same integers).
    flips: optional per-image flags — the crop is mirrored before it is resized (`flipped_crops`)."""
    from . import lib
    if not torch.cuda.is_available():
        raise RuntimeError("xfm_b200.feed.crop_resize needs a CUDA device (sm_100a); there is no CPU path")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    images, boxes = flipped_crops(images, boxes, flips)      # flips: optional per-image flags, mirror the crop before resizing
    sizes = [(int(im.shape[0]), int(im.shape[1])) for im in images]
    for im in images:
        if im.dtype != torch.uint8 or im.dim() != 3 or im.shape[2] != 3:
            raise ValueError("crop_resize: images must be uint8 [h, w, 3]")
    boxes = [(0, 0, w, h) if bx is None else tuple(int(v) for v in bx) for bx, (h, w) in zip(boxes, sizes)]
    plan = crop_resize_plan(sizes, boxes, out_h, out_w, taps=(taps == "host"))
    B = len(images)
    out = torch.empty((B, out_h, out_w, 3), dtype=torch.uint8, device=device)
    if B == 0:
        return out
    packed = torch.empty(plan["src_bytes"], dtype=torch.uint8, pin_memory=True)
    lib.host_pack([im.contiguous() for im in images], packed)      # multi-threaded gather into the staging buffer
    return _resize_on_device(packed.to(device, non_blocking=True), plan, out, taps)


def _resize_on_device(src, plan, out, taps="device"):
    """Device half of `crop_resize` / `decode_crop_resize`: src = the packed images on the device, in the layout of
    `crop_resize_plan` (image b at byte desc[b, 0]); taps as in `crop_resize`."""
    from . import lib
    B, out_h, out_w, _ = out.shape
    desc = plan["desc"].pin_memory().to(out.device, non_blocking=True)
    if taps == "host":
        hb, hk, vb, vk = (plan[k].pin_memory().to(out.device, non_blocking=True) for k in ("hb", "hk", "vb", "vk"))
    else:
        hb, hk, vb, vk = lib.resize_taps(desc, out_h, out_w, plan["KH"], plan["KV"])
    tmp = torch.empty(plan["tmp_bytes"], dtype=torch.uint8, device=out.device)
    return lib.resize_bicubic_u8(src, desc, hb, hk, vb, vk, tmp, out, plan["max_rows"])


# --------------------------------------------------------------------------------------------------- baseline JPEG decode
def _pil_rgb(blob):
    """What the evaluation loaders do to a file: `Image.open(f).convert("RGB")`, as uint8 [h, w, 3]."""
    import io
    import numpy as np
    from PIL import Image
    with Image.open(io.BytesIO(blob)) as im:
        return torch.from_numpy(np.array(im.convert("RGB")))


def jpeg_size(blob):
    """(width, height) of an image file's bytes, read from its header (for `random_resized_crop_box` before decoding):
    the marker walk of `xfm_jpeg_plan` for the device subset, Pillow's header parser for anything else."""
    import io
    from PIL import Image
    from . import lib
    st, w, h = (int(v) for v in lib.jpeg_plan([bytes(blob)], threads=1)[0, :3])
    if st == 0:
        return w, h
    with Image.open(io.BytesIO(blob)) as im:
        return im.size


def decode_jpeg(blobs, device=None, threads=8):
    """Decode a batch of image files (a list of `bytes`) on the GPU: returns (out, meta, n_fallback) with out = uint8 on the
    device, image b = out[meta[b, 0] : + meta[b, 1] * meta[b, 2] * 3] viewed as [meta[b, 2] (height), meta[b, 1] (width), 3],
    packed back to back in order (the source layout of `crop_resize_plan`), and meta int64 [B, 3] (offset, width, height) on
    the host.  Every image equals `Image.open(BytesIO(b)).convert("RGB")` byte for byte (or the call raises what Pillow
    raises): baseline Huffman JPEGs (grayscale or YCbCr, 4:4:4 / 4:2:2 / 4:2:0, with or without restart markers) are decoded
    by `xfm_jpeg_decode` (csrc/jpeg.cu); every other file, and every file the device decoder flags (invalid code, data
    ending early, unexpected marker), is decoded by Pillow into the same place.  n_fallback counts those.
    One synchronisation per call: the device->host read of the per-image status words that decides the second group."""
    import numpy as np
    from PIL import Image
    from . import lib
    if not torch.cuda.is_available():
        raise RuntimeError("xfm_b200.feed.decode_jpeg needs a CUDA device (sm_100a); there is no CPU path")
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    blobs = [b if isinstance(b, bytes) else bytes(b) for b in blobs]
    B = len(blobs)
    info = lib.jpeg_plan(blobs, threads)
    limit = Image.MAX_IMAGE_PIXELS
    host = {}
    for i in range(B):
        if info[i, 0] == 0 and limit is not None and info[i, 1] * info[i, 2] > limit:
            info[i, 0] = -1                                  # Pillow's decompression-bomb check decides (warning or error)
        if info[i, 0] != 0:
            host[i] = _pil_rgb(blobs[i])
            info[i, 1], info[i, 2] = host[i].shape[1], host[i].shape[0]
    dev = info[:, 0] == 0
    nbytes = info[:, 1] * info[:, 2] * 3
    offs = np.zeros((B, 4), np.int64)
    for col, size in ((0, np.array([len(b) for b in blobs], np.int64)), (1, info[:, 4]), (2, info[:, 5]), (3, nbytes)):
        size = size if col == 3 else np.where(dev, size, 0)
        offs[:, col] = np.cumsum(size) - size
    meta = torch.from_numpy(np.stack([offs[:, 3], info[:, 1], info[:, 2]], 1) if B else np.zeros((0, 3), np.int64))
    out = torch.empty(max(int(nbytes.sum()), 1), dtype=torch.uint8, device=device)
    if dev.any():
        desc, intervals = lib.jpeg_tables(blobs, info, offs, threads)
        data = torch.empty(int(sum(len(blobs[i]) for i in np.nonzero(dev)[0])), dtype=torch.uint8, pin_memory=True)
        lib.host_pack([blobs[i] for i in np.nonzero(dev)[0]], data, threads)
        status_h = torch.from_numpy(np.where(dev, 0, 1).astype(np.int32)).pin_memory()
        nb = lambda n: torch.empty(max(int(n), 1), dtype=torch.uint8, device=device)  # noqa: E731
        coef = torch.empty((max(int(info[dev, 4].sum()), 1), 64), dtype=torch.int16, device=device)
        planes, status = nb(info[dev, 5].sum()), status_h.to(device, non_blocking=True)
        lib.jpeg_decode(data.to(device, non_blocking=True), desc.to(device, non_blocking=True),
                        intervals.to(device, non_blocking=True), B, coef, planes, out, status,
                        int(info[dev, 4].max()), int(info[dev, 1].max()), int(info[dev, 2].max()))
    for i, img in host.items():
        out[offs[i, 3]:offs[i, 3] + nbytes[i]].copy_(img.reshape(-1))
    n_fallback = len(host)
    if dev.any():
        flagged = torch.nonzero(status.cpu() != 0).flatten().tolist()     # the one synchronisation of the call
        for i in flagged:
            if i in host:
                continue
            img = _pil_rgb(blobs[i])
            if tuple(img.shape) != (int(info[i, 2]), int(info[i, 1]), 3):
                raise RuntimeError(f"decode_jpeg: image {i}: Pillow returned {tuple(img.shape)}, the header says "
                                   f"{int(info[i, 1])} x {int(info[i, 2])}")
            out[offs[i, 3]:offs[i, 3] + nbytes[i]].copy_(img.reshape(-1))
            n_fallback += 1
    return out, meta, n_fallback


def decode_crop_resize(blobs, boxes, out_h, out_w, device=None):
    """Decode + crop + bicubic resize of image files on the GPU: uint8 [B, out_h, out_w, 3] on the device equal to
    `Image.open(BytesIO(b)).convert("RGB").crop(box).resize((out_w, out_h), BICUBIC)`; boxes entries (x0, y0, x1, y1) or
    None = the whole image.  `decode_jpeg` -> `xfm_resize_taps` -> `xfm_resize_bicubic_u8` reading the decoded batch in
    place (no copy in between); `lib.image_u8_to_f32` finishes the evaluation transform."""
    src, meta, _ = decode_jpeg(blobs, device)
    sizes = [(int(h), int(w)) for _, w, h in meta.tolist()]
    boxes = [(0, 0, w, h) if bx is None else tuple(int(v) for v in bx) for bx, (h, w) in zip(boxes, sizes)]
    if len(boxes) != len(sizes):
        raise ValueError("decode_crop_resize: one box (or None) per image")
    plan = crop_resize_plan(sizes, boxes, out_h, out_w, taps=False)
    out = torch.empty((len(sizes), out_h, out_w, 3), dtype=torch.uint8, device=src.device)
    if not sizes:
        return out
    return _resize_on_device(src, plan, out)


def _is_u8_image(t):
    return t.dtype == torch.uint8 and t.dim() == 4 and t.shape[3] == 3


class DeviceFeeder:
    """Iterate `loader` (batches = list / tuple / dict of tensors, None or plain python values) and yield the same
    structure on the device, `depth` batches ahead of the consumer.

    Per batch: every host tensor is staged in a pinned buffer of its slot (skipped when the loader already pins), copied on a
    private copy stream, and uint8 [B, H, W, 3] image tensors are finished there by `xfm_image_u8_to_f32` (ToTensor +
    Normalize with `mean` / `std`, optional random hflip with probability `flip_prob` per sample drawn from `generator`).
    `__next__` makes the consumer's current stream wait for that batch's event — no host synchronisation — and hands the
    tensors over with `record_stream`, so the caching allocator does not recycle them under the consumer.
    `h2d_bytes` counts what crossed PCIe."""

    def __init__(self, loader, device=None, depth=2, mean=CLIP_MEAN, std=CLIP_STD, flip_prob=0.0, generator=None):
        from . import lib
        if not torch.cuda.is_available():
            raise RuntimeError("xfm_b200.feed.DeviceFeeder needs a CUDA device (sm_100a); there is no CPU path")
        lib.lib()
        self._L = lib
        self.loader, self.depth = loader, max(1, int(depth))
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.mean, self.std, self.flip_prob, self.generator = tuple(mean), tuple(std), float(flip_prob), generator
        self.stream = torch.cuda.Stream(self.device)
        self._slots = [dict(pinned={}, event=None) for _ in range(self.depth + 1)]
        self._n = 0
        self.h2d_bytes = 0

    def __len__(self):
        return len(self.loader)

    def _stage(self, slot, key, t):
        if t.is_pinned():
            return t
        t = t.contiguous()
        buf = slot["pinned"].get(key)
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = slot["pinned"][key] = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        buf.copy_(t)
        return buf

    def _upload(self, batch):
        slot = self._slots[self._n % len(self._slots)]
        self._n += 1
        if slot["event"] is not None:
            slot["event"].synchronize()      # the copies that last read this slot's pinned buffers (depth + 1 batches ago)
        items = batch.items() if isinstance(batch, dict) else enumerate(batch)
        out = {}
        with torch.cuda.stream(self.stream):
            for k, v in items:
                if not isinstance(v, torch.Tensor):
                    out[k] = v
                    continue
                if v.device.type != "cpu":
                    out[k] = v
                    continue
                d = self._stage(slot, k, v).to(self.device, non_blocking=True)
                self.h2d_bytes += d.numel() * d.element_size()
                if _is_u8_image(d):
                    flip = None
                    if self.flip_prob > 0:
                        draw = torch.rand(d.shape[0], generator=self.generator) < self.flip_prob
                        flip = self._stage(slot, (k, "flip"), draw.to(torch.uint8)).to(self.device, non_blocking=True)
                        self.h2d_bytes += flip.numel()
                    d = self._L.image_u8_to_f32(d, self.mean, self.std, flip=flip)
                out[k] = d
            ev = torch.cuda.Event()
            ev.record(self.stream)
        slot["event"] = ev
        if isinstance(batch, dict):
            return out, ev
        seq = [out[i] for i in range(len(out))]
        return (tuple(seq) if isinstance(batch, tuple) else seq), ev

    def __iter__(self):
        it = iter(self.loader)
        queue = []
        done = False
        while True:
            while not done and len(queue) < self.depth:
                try:
                    queue.append(self._upload(next(it)))
                except StopIteration:
                    done = True
            if not queue:
                return
            batch, ev = queue.pop(0)
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(ev)
            for v in (batch.values() if isinstance(batch, dict) else batch):
                if isinstance(v, torch.Tensor) and v.is_cuda:
                    v.record_stream(cur)
            yield batch
