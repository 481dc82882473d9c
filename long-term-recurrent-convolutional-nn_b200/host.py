"""Host-side mirror of the reference's interface for the hot path (lrcn.jl), above the C ABI.

Julia is not installed in the build image, so the host side is written in Python with the
reference's own function names, argument meaning and error behaviour; the Julia `ccall` shim a
maintainer would add is julia/lrcn_b200.jl (INTEGRATION.md).  Everything numeric happens inside
liblrcn_b200.so -- this module only marshals the reference's data formats:

  model      : list of 9 column-major Float32 matrices            (initweights, lrcn.jl:489-510)
  seq        : (sequence, input_ids, lengths) as built by minibatch (lrcn.jl:257-297):
               sequence[k][j] = token at global time row k, batch slot j (1-based ids),
               input_ids[b][j] = image id of slot j in batch b, lengths[n] = caption length
  feats      : dict image id -> 4096 Float32                        (lrcn.jl:121-123)
"""
from __future__ import annotations

import struct
import sys

import numpy as np

from . import abi, synth

EOS, BOS, UNK = synth.EOS, synth.BOS, synth.UNK


class LRCN:
    """The decoder on one B200.  Replaces the (param, optim, state) triple the reference threads
    through train1 / average_loss / generate."""

    def __init__(self, hidden, vocab_size, embed, batchsize, max_len=28, precision=abi.PREC_BF16X3, device=0,
                 max_gen_rows=1024, use_graphs=True):
        if len(hidden) != 2:
            raise ValueError("lrcn() hard-wires two LSTM layers (lrcn.jl:540-551): --hidden needs exactly 2 sizes")
        self.hidden = [int(hidden[0]), int(hidden[1])]
        self.vocab_size, self.embed, self.batchsize = int(vocab_size), int(embed), int(batchsize)
        cfg = abi.default_config(embed=self.embed, hidden1=self.hidden[0], hidden2=self.hidden[1], vocab=self.vocab_size,
                                 max_batch=self.batchsize, max_len=max_len, max_gen_rows=max_gen_rows, device=device,
                                 precision=precision, use_graphs=1 if use_graphs else 0)
        self.h = abi.Handle(cfg)
        self._step = 0

    def close(self):
        self.h.close()

    # ---- weights (lrcn.jl:86-93, 183-186)
    def initweights(self, seed=1):
        """initweights(atype,hidden,vocab,embed) + upload; returns the host copy (list of 9)."""
        model = synth.initweights(self.hidden, self.vocab_size, self.embed, seed=seed)
        self.load_model(model)
        return model

    def load_model(self, model):
        if len(model) != 9:
            raise ValueError("model must hold 9 matrices (2*length(hidden)+5, lrcn.jl:492)")
        self.h.set_model(model)

    def model(self):
        """Host copy of the 9 matrices, e.g. for save(file,"model",model,...) (lrcn.jl:185,230)."""
        return self.h.get_model()

    # ---- checkpoint (lrcn.jl:88-93 load, :183-186 / :228-231 save; sidecar format of include/lrcn_b200.h)
    def save(self, path, vocab=None, with_adam=True):
        """save(file,"model",model,"vocab",vocab): weights (+ Adam m, v, t) and the vocab Dict in one sidecar file."""
        self.h.checkpoint_save(path, with_adam, vocab_to_bytes(vocab) if vocab else b"")

    def load(self, path):
        """load(file): restores the weights (and the optimizer state when the file has it); returns the vocab dict or None."""
        _, aux = self.h.checkpoint_load(path)
        return vocab_from_bytes(aux) if aux else None

    # ---- features (lrcn.jl:121-123)
    def load_features(self, feats: dict, split=0):
        ids = np.fromiter(feats.keys(), dtype=np.int64, count=len(feats))
        mat = np.stack([np.asarray(feats[int(i)], dtype=np.float32).reshape(4096) for i in ids])
        self.h.load_features(split, ids, mat)

    def load_feature_matrix(self, ids, mat, split=0):
        self.h.load_features(split, ids, mat)

    # ---- fc7 producer (lrcn.jl:190-221, 697-773; SURVEY 8 row f-4)
    def load_cnn(self, params):
        """get_params_cnn + get_convnet: params = 15 (filter, bias) pairs conv1_1..conv5_3, fc6, fc7 in MatConvNet's layout
        (filter kh x kw x Cin x Cout, bias of Cout values), uploaded once."""
        if len(params) != abi.CNN_LAYERS:
            raise ValueError(f"VGG-16 up to fc7 has {abi.CNN_LAYERS} layers, got {len(params)}")
        for layer, (w, b) in enumerate(params, start=1):
            self.h.set_cnn_param(layer, 0, w)
            self.h.set_cnn_param(layer, 1, b)

    def extract_features(self, images, ids, normalize=True):
        """extract_features (lrcn.jl:190-221) for preprocessed images (224 x 224 x 3 x n, resized and mean-subtracted on the
        host like read_image_data): the id -> relu7 Dict it saves, each row divided by its sum when normalize is set."""
        ids = list(ids)
        if np.ndim(images) != 4 or np.shape(images)[3] != len(ids):
            raise ValueError("images must be 224 x 224 x 3 x n with one id per image")
        feats = self.h.extract_features(images, abi.FEAT_L1 if normalize else 0)
        return {int(i): feats[k] for k, i in enumerate(ids)}

    # ---- one batch (lrcn.jl:553-583)
    @staticmethod
    def _tokens(sequence, rng):
        rows = [np.asarray(sequence[t], dtype=np.int64) for t in rng]
        return np.stack(rows) if rows else np.zeros((0, 0), dtype=np.int64)

    def loss(self, input_ids, sequence, rng, split=0):
        """loss(param,state,input,sequence,range): mean NLL over B*(l+1) tokens."""
        tok = self._tokens(sequence, rng)
        if tok.size == 0:
            tok = np.zeros((0, len(input_ids)), dtype=np.int64)
        s, n = self.h.loss(split, input_ids, tok)
        return -s / n

    def lossgradient(self, input_ids, sequence, rng, pdrop=0.0, seed=0, split=0):
        """lossgradient(param,copy(state),input,sequence,range;pdrop) -> list of 9 gradients."""
        tok = self._tokens(sequence, rng)
        self.last_loss = self.h.grad(split, input_ids, tok, pdrop, seed)
        return [self.h.get_grad(k) for k in range(1, 10)]

    def update(self):
        """update!(param,gloss,optim) on the gradients held by the library (lrcn.jl:394)."""
        self.h.adam_update()

    # ---- epoch drivers
    @staticmethod
    def _start_indices(lengths, batch_size):
        starts, index = [], 0
        for t in range(0, len(lengths), batch_size):  # lrcn.jl:336-342
            starts.append(index)
            index += int(lengths[t])
        return starts

    def train1(self, seq, batch_size=None, pdrop=0.0, shuffle_seed=0, split=0, progress=None, per_step=False):
        """One epoch of the hot loop lrcn.jl:351-396: shuffled batch order, skip l>28,
        gradient + Adam per batch.  `lr`/`gclip` are ignored by the reference and so not taken.
        Default: ONE library call for the epoch (batches staged on the device, no per-step host work; SURVEY 8 row f-1);
        per_step=True or a progress callback drives one lrcn_train_step per batch instead.  Both give the same losses."""
        sequence, input_ids, lengths = seq
        batch_size = batch_size or self.batchsize
        starts = self._start_indices(lengths, batch_size)
        order = np.arange(0, len(lengths), batch_size)
        np.random.RandomState(shuffle_seed).shuffle(order)
        if not per_step and progress is None and len(order):
            blens = np.asarray(lengths, dtype=np.int64)[::batch_size]
            seq_m = np.stack([np.asarray(r, dtype=np.int64) for r in sequence]) if len(sequence) else np.zeros((0, batch_size), np.int64)
            ids_m = np.stack([np.asarray(r, dtype=np.int64) for r in input_ids])
            losses = self.h.train_epoch(split, seq_m, ids_m, blens, order // batch_size, pdrop, self._step + 1)
            self._step += len(losses)
            return losses
        losses = []
        for t in order:
            l = int(lengths[t])
            if l > 28:  # lrcn.jl:353
                continue
            b = t // batch_size
            index = starts[b]
            tok = self._tokens(sequence, range(index, index + l))
            self._step += 1
            losses.append(self.h.train_step(split, input_ids[b], tok, pdrop, self._step))
            if progress:
                progress(len(losses), losses[-1])
        return losses

    def average_loss(self, seq, split=0, per_step=False):
        """average_loss(param,seq,feats): token-weighted mean NLL, pdrop=0 (lrcn.jl:407-486).  Default: one library call for
        the split (lrcn_loss_epoch, batches staged on the device); per_step=True: one lrcn_loss call per batch."""
        sequence, input_ids, lengths = seq
        batch_size = len(sequence[0])
        if not per_step:
            blens = np.asarray(lengths, dtype=np.int64)[::batch_size]
            s, n = self.h.loss_epoch(split, np.stack([np.asarray(r, dtype=np.int64) for r in sequence]),
                                     np.stack([np.asarray(r, dtype=np.int64) for r in input_ids]), blens)
            return -s / n
        starts = self._start_indices(lengths, batch_size)
        total, count = 0.0, 0
        for b, t in enumerate(range(0, len(lengths), batch_size)):
            l = int(lengths[t])
            if l > 28:
                continue
            tok = self._tokens(sequence, range(starts[b], starts[b] + l))
            s, n = self.h.loss(split, input_ids[b], tok)
            total += s
            count += n
        return -total / count

    def train(self, sequence, vocab=None, epochs=1, batch_size=None, savefile=None, pdrop=0.4, out=sys.stdout, datasheet=None, shuffle_seed=0):
        """train!(model, optim, sequence, vocab, o), lrcn.jl:222-239 (SURVEY 8 row f-3): per epoch one train1 pass at pdrop 0.4 over
        sequence[0], the checkpoint (`save(o[:savefile], "model", model, "vocab", vocab)`), then average_loss at pdrop 0 on the
        training split (feats, split 0) and the validation split (featsvl, split 1), printed -- and appended to the data sheet
        the reference hard-codes -- as `(:epoch,e,:loss,l_trn,l_val)`.  Three library calls per epoch (lrcn_train_epoch, 2x
        lrcn_loss_epoch): no per-batch host work.  Returns the list of (l_trn, l_val)."""
        history = []
        for epoch in range(1, epochs + 1):
            self.train1(sequence[0], batch_size=batch_size, pdrop=pdrop, shuffle_seed=shuffle_seed + epoch)
            if savefile is not None:
                print(f"INFO: Saving last model to {savefile}", file=sys.stderr)   # info(...) lrcn.jl:227
                self.save(savefile, vocab)
            losses = (np.float32(self.average_loss(sequence[0], split=0)), np.float32(self.average_loss(sequence[1], split=1)))
            line = f"(:epoch,{epoch},:loss,{losses[0]}f0,{losses[1]}f0)"
            print(line, file=out)
            if datasheet is not None:
                with open(datasheet, "a+") as f:
                    print(line, file=f)
            history.append((float(losses[0]), float(losses[1])))
        self.h.sync()  # gpu()>=0 && Knet.cudaDeviceSynchronize()  lrcn.jl:240
        return history

    # ---- generation (lrcn.jl:585-642)
    def beam_search(self, image_ids, nword, beam_width, split=1):
        """Numeric part of generate()+beam_search() for many images; returns
        (list of token lists incl. bos, fp32 probabilities, per-token log-probs)."""
        toks, lens, prob, lps = self.h.beam_search(split, image_ids, beam_width, nword)
        out = [toks[i, :lens[i]].tolist() for i in range(len(lens))]
        return out, prob, [lps[i, :lens[i] - 1] for i in range(len(lens))]

    def generate(self, input, vocab, nword, beam_width, split=1, out=sys.stdout, in_out=sys.stdout):
        """generate(param,state,input::Int,vocab,nword,beam_width,val_feats;out,in_out):
        writes the id line and the caption line exactly like lrcn.jl:600,633-640."""
        index_to_char = [None] * len(vocab)
        for k, v in vocab.items():
            index_to_char[v - 1] = k
        print(input, file=in_out)
        try:
            hyps, _, _ = self.beam_search([input], nword, beam_width, split)
        except abi.LrcnError as e:
            if e.code == abi.ERR_MISSING:
                raise RuntimeError("misssing features!!!!!!") from e  # lrcn.jl:603
            raise
        print(caption_text(hyps[0], index_to_char), file=out)
        return hyps[0]


# ---- checkpoint sidecar: pure-host reader / writer of the library's format (no GPU needed; the Julia shim has the same pair)
CKPT_MAGIC = b"LRCNB2CK"


def vocab_to_bytes(vocab: dict) -> bytes:
    """vocab Dict{String,Int} (lrcn.jl:98-118) as "word\tindex\n" lines, UTF-8, in index order."""
    return "".join(f"{w}\t{i}\n" for w, i in sorted(vocab.items(), key=lambda kv: kv[1])).encode("utf-8")


def vocab_from_bytes(b: bytes) -> dict:
    out = {}
    for line in b.decode("utf-8").split("\n"):
        if line:
            w, i = line.rsplit("\t", 1)
            out[w] = int(i)
    return out


def write_checkpoint(path, model, dims, vocab=None, adam=None):
    """model: 9 column-major float32 matrices; dims = (E, H1, H2, V); adam = (m[9], v[9], t) or None."""
    aux = vocab_to_bytes(vocab) if vocab else b""
    with open(path, "wb") as f:
        f.write(CKPT_MAGIC)
        f.write(struct.pack("<II4iqq", 1, 1 if adam else 0, *[int(d) for d in dims], int(adam[2]) if adam else 0, len(aux)))
        sections = [model] + ([adam[0], adam[1]] if adam else [])
        for mats in sections:
            for w in mats:
                w = np.asfortranarray(w, dtype=np.float32)
                f.write(struct.pack("<qq", *w.shape))
                f.write(w.tobytes(order="F"))
        f.write(aux)


def read_checkpoint(path):
    """-> dict(dims, adam_t, model[9], m[9] | None, v[9] | None, vocab | None).  Validates magic, version and sizes."""
    with open(path, "rb") as f:
        if f.read(8) != CKPT_MAGIC:
            raise ValueError(f"{path}: not an LRCNB2CK checkpoint")
        version, flags, E, H1, H2, V, adam_t, aux_bytes = struct.unpack("<II4iqq", f.read(40))
        if version != 1:
            raise ValueError(f"{path}: unsupported checkpoint version {version}")
        shapes = synth.param_shapes(E, [H1, H2], V)

        def mats():
            out = []
            for k in range(9):
                r, c = struct.unpack("<qq", f.read(16))
                if (r, c) != shapes[k]:
                    raise ValueError(f"{path}: matrix {k + 1} is {r}x{c}, expected {shapes[k]} (lrcn.jl:489-510)")
                raw = f.read(4 * r * c)
                if len(raw) != 4 * r * c:
                    raise ValueError(f"{path}: truncated")
                out.append(np.frombuffer(raw, dtype="<f4").reshape((r, c), order="F").copy(order="F"))
            return out

        model = mats()
        m = v = None
        if flags & 1:
            m, v = mats(), mats()
        aux = f.read(aux_bytes)
        if len(aux) != aux_bytes:
            raise ValueError(f"{path}: truncated")
    return dict(dims=(E, H1, H2, V), adam_t=adam_t, model=model, m=m, v=v, vocab=vocab_from_bytes(aux) if aux else None)


def caption_text(word_indices, index_to_char):
    """lrcn.jl:633-640: tokens[2:] up to the first eos, each followed by ' ', then '.'."""
    parts = []
    for tok in word_indices[1:]:
        if tok == EOS:
            break
        parts.append(index_to_char[tok - 1] + " ")
    return "".join(parts) + "."


# ---- batching (SURVEY §8 row f-1: lrcn.jl:257-327) -- integer-only host data prep -----------------
def delete_unbatchable_captions(caption_dict, batch_size):
    """delete_unbatchable_captions!(caption_dict,batch_size), lrcn.jl:299-327.  caption_dict is a
    length-sorted list of ((id, words), length).  Returns the surviving list (new list)."""
    lengths = [t[1] for t in caption_dict]
    n = len(lengths)
    if n == 0:
        return []
    limit = n - batch_size + 1
    max_length = max(lengths)
    current_length = lengths[0]
    current_index = 1  # 1-based, as in the reference
    drop = set()
    while current_index < limit:
        if lengths[current_index + batch_size - 2] == current_length:
            current_index += batch_size
        else:
            old_index = current_index
            current_index = 0
            while current_index == 0:
                current_length += 1
                if current_length > max_length:
                    break
                try:
                    current_index = lengths.index(current_length) + 1  # findfirst
                except ValueError:
                    current_index = 0
            if current_index == 0:  # ran past max_length: everything from old_index on is unbatchable
                drop.update(range(old_index, n + 1))
                break
            drop.update(range(old_index, current_index))
        if current_index >= limit:
            drop.update(range(current_index, n + 1))
            break
    return [caption_dict[k - 1] for k in range(1, n + 1) if k not in drop]


def minibatch(caption_dict, word_to_index, batch_size):
    """minibatch(caption_dict,word_to_index,batch_size), lrcn.jl:257-297 -> (sequence,input_ids,lengths).
    Splits with <= 30000 captions are forced to batch_size 10 (lrcn.jl:260-269)."""
    if len(caption_dict) <= 30000:
        batch_size = 10
    caption_dict = delete_unbatchable_captions(caption_dict, batch_size)
    lengths = [t[1] for t in caption_dict]
    nbatch = sum(lengths) // batch_size
    sequence = [np.zeros(batch_size, dtype=np.int64) for _ in range(nbatch)]
    input_ids = [np.zeros(batch_size, dtype=np.int64) for _ in range(0, len(lengths), batch_size)]
    index = 0
    for b, i in enumerate(range(0, len(lengths), batch_size)):
        l = lengths[i]
        for j in range(i, i + batch_size):
            (img_id, words), _ = caption_dict[j]
            input_ids[b][j - i] = img_id
            for k in range(l):
                sequence[index + k][j - i] = word_to_index.get(words[k], UNK)  # lrcn.jl:288
        index += l
    return sequence, input_ids, lengths


# ---- data-parallel sharding (SURVEY §8e): a global batch of equal-length captions splits by rows -------------
def shard_batch(image_ids, tokens, rank, world):
    """Rows [rank*b, (rank+1)*b) of a global batch (image_ids: Bg, tokens: l x Bg, time-major).
    Every rank keeps the same caption length l, so control flow is identical across ranks; the library
    scales each rank's gradient by 1/(world*b*(l+1)) and the allreduce(sum) yields the global-batch gradient."""
    image_ids = np.asarray(image_ids)
    tokens = np.asarray(tokens)
    bg = len(image_ids)
    if bg % world:
        raise ValueError(f"global batch {bg} not divisible by {world} ranks")
    b = bg // world
    sl = slice(rank * b, (rank + 1) * b)
    return np.ascontiguousarray(image_ids[sl]), np.ascontiguousarray(tokens[:, sl])


def shard_images(image_ids, rank, world):
    """Generation shards images across ranks with no collective: contiguous, near-equal slices in input order."""
    n = len(image_ids)
    lo = (n * rank) // world
    hi = (n * (rank + 1)) // world
    return image_ids[lo:hi], (lo, hi)
