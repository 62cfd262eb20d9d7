"""Host-side input handling that sits on the hot path: caption token indexing (bit-exact mirror of
txt2vid/data/__init__.py:260-355 Vocab / collate_fn), a pinned-memory prefetcher with the reference's
`data_prefetcher.next()` contract (:131-156), and synthetic batches of the shapes SURVEY.md 8(d) names.
The reference's file/LMDB datasets, DALI hooks and caches are out of scope (SURVEY.md 2.1 rows 15-17).
"""
import torch


class Vocab(object):
    START, END, UNKNOWN, PAD = '<start>', '<end>', '<unk>', '<pad>'   # PAD is always index 0

    def __init__(self):
        self.word2idx, self.idx2word, self.idx = {}, {}, 0
        for w in (self.PAD, self.START, self.END, self.UNKNOWN):
            self.add_word(w)

    def add_word(self, word):
        word = word.lower()
        if word not in self.word2idx:
            self.word2idx[word] = self.idx
            self.idx2word[self.idx] = word
            self.idx += 1

    def get_word(self, idx):
        return self.idx2word.get(idx, self.UNKNOWN)

    def __call__(self, word):
        return self.word2idx.get(word.lower(), self.word2idx[self.UNKNOWN])

    def __len__(self):
        return len(self.word2idx)

    def tokenize(self, sentence):
        """START, then the words; a word ending in '.' yields the word without it followed by END."""
        yield self.START
        for word in sentence.split():
            if word[-1] == '.':
                yield word[0:-1]
                yield self.END
            else:
                yield word

    def encode(self, sentence):
        """Caption part of Dataset.__getitem__ (data/__init__.py:250-254): END appended when missing."""
        toks = [self(t) for t in self.tokenize(sentence)]
        if toks[-1] != self(self.END):
            toks.append(self(self.END))
        return torch.tensor(toks, dtype=torch.long)

    def to_words(self, tokens):
        out = u''
        for i, tok in enumerate(tokens):
            word = self.get_word(int(tok))
            if word != self.END and i != 0:
                out += ' '
            out += word
        return out


def build_vocab(sentences):
    vocab = Vocab()
    for s in sentences:
        for w in vocab.tokenize(s):
            vocab.add_word(w)
    return vocab


def collate_fn(data):
    """[(video, caption)] -> (videos (B,...), tokens (B,Lmax) zero padded, lengths), sorted by caption
    length, longest first (stable), as pack_padded_sequence requires (data/__init__.py:326-355)."""
    data.sort(key=lambda item: len(item[1]), reverse=True)
    vids, caps = zip(*data)
    lengths = [len(c) for c in caps]
    tokens = torch.zeros(len(caps), max(lengths)).long()
    for i, c in enumerate(caps):
        tokens[i, :lengths[i]] = c[:lengths[i]]
    return torch.stack(vids, 0), tokens, lengths


class data_prefetcher(object):
    """`x, y = prefetcher.next()` with y = [tokens, lengths] (or []); None, None at the end.  The next
    batch is staged through pinned memory and copied on a side stream while the current one trains.

    Four persistent device staging slots per batch field (a fresh 0.8 GB allocation per step would make the caching
    allocator fall back to cudaMalloc, a device-wide sync).  Slot reuse is guarded on the HOST: before batch i+1 is
    copied into the slot batch i-3 lived in, the host waits for an event recorded when batch i-2 was handed out (it
    fires once everything enqueued for batch i-3 has run).  [measured on B200, scripts/h2d_probe.py; step 86.5 ms
    with resident inputs] a device-side `copy_stream.wait_stream(compute_stream)` in front of the copies serialises
    them with the graph replay that follows (100-115 ms); a host-side wait on the PREVIOUS step's event stalls the
    host, which must stay more than one step ahead of the device for back-to-back graph launches (100 ms); with the
    guard two steps back the event has always fired and the copies overlap (91 ms)."""
    CHUNK_BYTES = 48 << 20
    SLOTS = 4
    GUARD = "host"

    def __init__(self, loader, device=None, normalize=True):
        # normalize=False: uint8 frames are handed out as stored; the consumer normalises them where it needs them
        # (trainer.GraphedTrainStep fuses ToTensor + Normalize into the fill of its static input: one pass reading
        # 1 byte and writing 4 per pixel instead of a side-stream pass plus a 4-byte copy)
        self.normalize = normalize
        self.loader = iter(loader)
        self.device = torch.device(device if device is not None else
                                   ('cuda' if torch.cuda.is_available() else 'cpu'))
        self.stream = torch.cuda.Stream() if self.device.type == 'cuda' else None
        self._slots, self._slot = tuple({} for _ in range(self.SLOTS)), 0
        self._handed = [None] * self.SLOTS      # event recorded when the slot's batch was handed to the consumer
        self._prev_event = None
        self._norm = [None] * self.SLOTS        # fp32 images of uint8 clips (see _normalize)
        self._deferred = False
        self._preload()

    def _to_dev(self, t, key):
        if not isinstance(t, torch.Tensor) or self.device.type != 'cuda':
            return t
        if t.is_cuda:                            # an on-device generator (MovingDigits) hands out resident batches
            return t
        if not t.is_pinned():
            t = t.pin_memory()
        bufs = self._slots[self._slot]
        buf = bufs.get(key)
        if buf is None or buf.shape != t.shape or buf.dtype != t.dtype:
            buf = bufs[key] = torch.empty(t.shape, dtype=t.dtype, device=self.device)
        # [measured on B200] ONE 805 MB cudaMemcpyAsync on the side stream stalls the kernels of a concurrently
        # replayed graph for its whole duration (step 100.6 -> 117.5 ms); the same bytes in <= 64 MB pieces overlap
        # (102.4 ms): scripts/h2d_probe.py
        nbytes = t.numel() * t.element_size()
        pieces = min(t.size(0), -(-nbytes // self.CHUNK_BYTES)) if t.dim() > 0 and t.is_contiguous() else 1
        if pieces <= 1:
            buf.copy_(t, non_blocking=True)
        else:
            for d, h in zip(buf.chunk(pieces), t.chunk(pieces)):
                d.copy_(h, non_blocking=True)
        return buf

    def _normalize(self, frames_u8):
        """uint8 frames -> the reference's transforms.ToTensor() + Normalize(0.5, 0.5) (data/__init__.py:362-364) in
        fp32 on the device (side stream): x / 255, then (x - 0.5) / 0.5 -- the same IEEE operations, so the same values.
        A loader that hands out the frames as stored moves a quarter of the bytes over PCIe."""
        out = self._norm[self._slot]
        if out is None or out.shape != frames_u8.shape:
            out = self._norm[self._slot] = torch.empty(frames_u8.shape, dtype=torch.float32, device=self.device)
        from . import kernels as K
        return K.u8_normalize(frames_u8, out)             # t2v_u8_normalize: IEEE division, bit-exact (tested)

    def _preload(self):
        try:
            batch = next(self.loader)
        except StopIteration:
            self.next_x = self.next_y = None
            return
        if self.stream is not None:
            self._slot = (self._slot + 1) % self.SLOTS
            free = self._handed[self._slot]
            if free is not None:                 # host-side guard (see class docstring); normally already fired
                if self.GUARD == "host":
                    free.synchronize()
                elif self.GUARD == "device":
                    self.stream.wait_event(free)
            if any(isinstance(a, torch.Tensor) and a.is_cuda for a in batch):
                # a device-resident batch (MovingDigits) was produced on the consumer's stream: order the side stream
                # (uint8 normalisation) behind it
                self.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.stream):
                self.next_x = self._to_dev(batch[0], 0)
                if self.normalize and isinstance(self.next_x, torch.Tensor) and self.next_x.dtype == torch.uint8:
                    self.next_x = self._normalize(self.next_x)
                self.next_y = [self._to_dev(a, 1 + i) for i, a in enumerate(batch[1:])]
        else:
            self.next_x, self.next_y = batch[0], list(batch[1:])

    def preload(self):
        """Stage the following batch now (after next(preload=False)): callers that launch their step first keep the
        step's own small transfers ahead of the bulk copy in the copy-engine queue."""
        if self._deferred:
            self._deferred = False
            self._preload()

    def next(self, preload=True):
        if self._deferred:
            self.preload()
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)
        x, y = self.next_x, self.next_y
        if x is not None and not preload:
            if self.stream is not None:
                ev = torch.cuda.Event()
                ev.record()
                self._handed[(self._slot - 1) % self.SLOTS] = ev
            self._deferred = True
            return x, y
        if x is not None:
            if self.stream is not None:
                # fires when everything enqueued so far (the step of the PREVIOUS batch) has run; it guards the slot
                # of the previous batch: by then its consumer has finished with it
                ev = torch.cuda.Event()
                ev.record()
                prev = (self._slot - 1) % self.SLOTS
                self._handed[prev] = ev
            self._preload()
        return x, y


class SyntheticVideoCaptions(object):
    """Iterable of `num_batches` synthetic (video (B,T,C,H,W) in [-1,1], tokens, lengths) batches:
    U(-1,1) clips and MSRVDC-shaped captions (lengths U{4..20}, tokens U{4..V-1}, START/END framed),
    SURVEY.md 8(d).  Stands in for get_loader(...) in benchmarks and tests."""

    def __init__(self, batch_size, num_batches, vocab_size=1000, frames=16, size=64, channels=3, captions=True,
                 seed=1234, as_uint8=False):
        self.B, self.n, self.V = batch_size, num_batches, vocab_size
        self.T, self.S, self.C = frames, size, channels
        self.captions = captions
        self.seed = seed
        self.as_uint8 = as_uint8        # frames as stored (uint8); data_prefetcher applies ToTensor + Normalize on the device

    def __len__(self):
        return self.n

    def batch(self, i):
        g = torch.Generator().manual_seed(self.seed + i)
        if self.as_uint8:
            x = torch.randint(0, 256, (self.B, self.C, self.T, self.S, self.S), generator=g, dtype=torch.uint8)
        else:
            x = torch.rand(self.B, self.C, self.T, self.S, self.S, generator=g) * 2 - 1
        x = x.permute(0, 2, 1, 3, 4)                         # loader order (B,T,C,H,W); train() permutes back
        if not self.captions:
            return (x,)
        lengths = sorted([int(v) for v in torch.randint(4, 21, (self.B,), generator=g)], reverse=True)
        tokens = torch.zeros(self.B, lengths[0], dtype=torch.long)
        for b, L in enumerate(lengths):
            tokens[b, 0] = 1
            tokens[b, 1:L - 1] = torch.randint(4, self.V, (L - 2,), generator=g)
            tokens[b, L - 1] = 2
        return x, tokens, lengths

    def __iter__(self):
        for i in range(self.n):
            yield self.batch(i)


class MovingDigits(object):
    """On-device synthetic moving-MNIST batches with their captions (SURVEY 8(f1)): the generator of
    txt2vid/data/synthetic/generate.py:59-182 re-designed so that only a few integers per clip cross PCIe.

    Host: the per-clip random decisions in the REFERENCE'S RNG ORDER (numpy for class / digit / coordinates, `random`
    for animation length / axis / direction, generate.py:82-166) and the per-frame patch positions of generate_frames
    (:18-47, float64 arithmetic truncated to int32).  Device: t2v_moving_digits pastes the patches from a resident digit
    bank into the clips (bit-exact frames, stored uint8 or already ToTensor + Normalize'd fp32) and t2v_grammar_tokens
    writes the token rows Vocab.tokenize + collate_fn would produce for the sentences.  A batch is B * (T + 1) * 2 + 2 B
    int32 over PCIe instead of B * T * 3 * H * W floats.  Iterating yields (clips (B,T,3,H,W), tokens (B,8), lengths):
    the loader contract of data/__init__.py:326-355, usable as `dataset` of trainer.train() (data_prefetcher passes
    resident tensors through).

    bank: {class: uint8 array (n_c, oh, ow)} (MNIST resized to 28 x 28 in the reference, generate.py:184-207)."""

    MOVES = (("bottom", "top"), ("top", "bottom"), ("right", "left"), ("left", "right"))   # horizontal * 2 + forward

    def __init__(self, batch_size, num_batches, bank, vocab=None, frames=16, size=64, device="cuda", as_uint8=False,
                 seed=None):
        import numpy as np
        self.B, self.n, self.T, self.W, self.H = batch_size, num_batches, frames, size, size
        self.device, self.as_uint8 = torch.device(device), as_uint8
        self.classes = sorted(bank.keys())
        self.counts = [len(bank[c]) for c in self.classes]
        self.offsets = [0]
        for n in self.counts:
            self.offsets.append(self.offsets[-1] + n)
        flat = np.concatenate([np.asarray(bank[c], dtype=np.uint8) for c in self.classes], axis=0)
        self.oh, self.ow = int(flat.shape[1]), int(flat.shape[2])
        self.bank = torch.from_numpy(flat).contiguous().to(self.device)
        self.vocab = vocab if vocab is not None else build_vocab(self.all_sentences())
        v = self.vocab
        table = [v(v.START), v("digit")] + [v(str(c)) for c in range(10)] + [v("is"), v("and"), v(v.END)]
        for a, b in self.MOVES:
            table += [v(a), v(b)]
        self.table = torch.tensor(table, dtype=torch.int64, device=self.device)
        if seed is not None:
            import random
            random.seed(seed)
            np.random.seed(seed)

    @classmethod
    def all_sentences(cls):
        return ["digit %d is %s and %s." % (c, a, b) for c in range(10) for a, b in cls.MOVES]

    def __len__(self):
        return self.n

    def draw(self):
        """One clip's decisions, consuming numpy / random exactly as generate_examples does per example."""
        import random
        import numpy as np
        W, H, T = self.W, self.H, self.T
        ci = int(np.random.randint(0, len(self.classes)))
        di = int(np.random.randint(0, self.counts[ci]))
        anim = random.randint(int(0.1 * T), T)
        horizontal = random.randint(0, 1)
        forward = random.randint(0, 1)
        if horizontal:
            y = int(np.random.randint(0, H))
            x1 = int(np.random.randint(0, int(0.1 * W)))
            x2 = int(np.random.randint(int(0.9 * W), W))
            a, b = [x1, y], [x2, y]
        else:
            x = int(np.random.randint(0, W))
            y1 = int(np.random.randint(0, int(0.1 * H)))
            y2 = int(np.random.randint(int(0.9 * H), H))
            a, b = [x, y1], [x, y2]
        if not forward:
            a, b = b, a
        lim = (W - self.ow, H - self.oh)
        a = [min(max(a[k], 0), lim[k]) for k in (0, 1)]
        b = [min(max(b[k], 0), lim[k]) for k in (0, 1)]
        return {"cls": self.classes[ci], "digit": self.offsets[ci] + di, "anim": anim, "move": horizontal * 2 + forward,
                "a": a, "b": b}

    @staticmethod
    def frame_positions(a, b, frames, anim, bounce=True):
        """Top-left corner of the patch in every frame: the walk of generate_frames (generate.py:24-43): the fraction
        (i - start + 1) / (anim + 1) clipped to [0, 1] moves the patch from `a` to `b`; on frame i == end the window
        advances by `anim` and the end points swap (the bounce); coordinates truncate toward zero like
        np.array(..., dtype=np.int32)."""
        import numpy as np
        src, dst = np.array(a), np.array(b)
        start, end = 0, anim
        out = []
        for i in range(frames):
            frac = float(np.clip((i - start + 1) / (end - start + 1), 0, 1))
            p = np.array(src + (dst - src) * frac, dtype=np.int32)
            if bounce and i == end:
                start, end = start + anim, end + anim
                src, dst = dst, src
            out.append([int(p[0]), int(p[1])])
        return out

    def sentence(self, d):
        a, b = self.MOVES[d["move"]]
        return "digit %d is %s and %s." % (d["cls"], a, b)

    def batch(self, draws=None):
        draws = draws if draws is not None else [self.draw() for _ in range(self.B)]
        B = len(draws)
        pos = torch.tensor([self.frame_positions(d["a"], d["b"], self.T, d["anim"]) for d in draws], dtype=torch.int32)
        small = torch.tensor([[d[k] for d in draws] for k in ("digit", "cls", "move")], dtype=torch.int32)   # (3, B)
        if self.device.type == "cuda":
            pos, small = pos.pin_memory().to(self.device, non_blocking=True), small.pin_memory().to(self.device, non_blocking=True)
        from . import kernels as K
        clips = K.moving_digits(self.bank, small[0], pos, self.T, self.H, self.W, out_f32=not self.as_uint8, layout=0)
        tokens = K.grammar_tokens(small[1], small[2], self.table)
        return clips, tokens, [8] * B

    def __iter__(self):
        for _ in range(self.n):
            yield self.batch()


class MovingDigitsDataset(MovingDigits):
    """`--data` target of txt2vid.train.gan (created by reflection with `vocab=` and `anno=`, train/gan.py:132): the
    on-device moving-MNIST generator over a seeded random digit bank (MNIST itself is a download; pass `bank_path`, a
    torch.save'd {class: uint8 (n, 28, 28)} dict, for real digits).  Example config:
        {"class": "txt2vid.data.MovingDigitsDataset", "args": {"batch_size": 64, "num_batches": 100}}"""

    def __init__(self, vocab=None, anno=None, batch_size=64, num_batches=100, frames=16, size=64, seed=None,
                 bank_path=None, bank_seed=7, per_class=3, as_uint8=False, device="cuda"):
        import numpy as np
        if bank_path is not None:
            bank = {int(c): np.asarray(v, dtype=np.uint8) for c, v in torch.load(bank_path, weights_only=False).items()}
        else:
            rng = np.random.RandomState(bank_seed)
            bank = {c: np.stack([rng.randint(0, 256, (28, 28)).astype(np.uint8) for _ in range(per_class)])
                    for c in range(10)}
        super().__init__(batch_size, num_batches, bank, vocab=vocab, frames=frames, size=size, device=device,
                         as_uint8=as_uint8, seed=seed)
