"""Device pipeline: the B200 replacement for ``ErrorModel.detect`` (errors.py:545-582) and the
inference half of ``RepairModel._run`` (model.py:1288-1408).

Everything that touches table-sized data is a call into ``libb200repair.so``; PyTorch tensors are
only the buffers those calls read and write (plus ``torch.distributed`` for the one exchange step
of the row-sharded multi-GPU path).  Host code here handles dictionaries, the tiny count tensors
and model bookkeeping.
"""
import logging
import re

import time

import numpy as np

from . import constraints as DC
from . import stats_host as SH
from ._native import DR_OP, Context
from .table import DeviceTable

_logger = logging.getLogger("repair")

MAX_FD_KEY_SPACE = 1 << 27      # int32 lo + hi tables: 1 GiB
MAX_PROJECTION_BITS = 1 << 31   # projection-presence bitmap of a general denial constraint: 256 MiB
PRESENCE_SAMPLE_ROWS = 1 << 20  # rows used for distinct-pair lower bounds


_RED = {"sum": 0, "min": 1, "max": 2, "or": 3}
_GATHER_LIMIT = 1 << 24   # elements per part above which a part gets its own all-reduce


class Dist:
    """The exchange step of the row-sharded path.  ``exchange`` reduces a list of count tensors across
    the ranks with ONE collective: every rank packs its parts into an int64 buffer, one all-gather
    (NCCL over NVLink) moves the G copies, and ``dr_combine_counts`` folds them segment by segment --
    SUM for histograms / pair tables / cell counts, MIN / MAX for per-key bounds, OR for presence
    bits -- so a pass needs one collective whatever mix of reductions it has (SURVEY.md 8e)."""

    def __init__(self, group=None):
        import torch.distributed as td
        self.td = td
        self.group = group
        self.rank = td.get_rank(group)
        self.world = td.get_world_size(group)
        self.n_exchanges = 0
        self.bytes_exchanged = 0

    def sum_(self, t):
        self.td.all_reduce(t, op=self.td.ReduceOp.SUM, group=self.group)

    def min_(self, t):
        self.td.all_reduce(t, op=self.td.ReduceOp.MIN, group=self.group)

    def max_(self, t):
        self.td.all_reduce(t, op=self.td.ReduceOp.MAX, group=self.group)

    def all_gather_rows(self, t):
        """Concatenation, in rank order, of every rank's [n_r, ...] tensor (n_r may differ)."""
        import torch
        cnt = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
        counts = torch.empty(self.world, dtype=torch.int64, device=t.device)
        self.td.all_gather_into_tensor(counts, cnt, group=self.group)
        counts = [int(c) for c in counts.cpu()]
        m = max(counts + [1])
        pad = torch.zeros((m,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        pad[:t.shape[0]] = t
        flat = torch.empty((self.world * m,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        self.td.all_gather_into_tensor(flat, pad, group=self.group)
        return torch.cat([flat[r * m:r * m + counts[r]] for r in range(self.world)]), counts

    def exchange(self, ctx, parts):
        """parts: [(tensor, "sum" | "min" | "max" | "or")], reduced IN PLACE across the ranks."""
        import torch
        parts = [(t, op) for t, op in parts if t is not None and t.numel() > 0]
        small = []
        for t, op in parts:
            if t.numel() > _GATHER_LIMIT and op != "or":   # huge key tables: a plain all-reduce of their own
                {"sum": self.sum_, "min": self.min_, "max": self.max_}[op](t)
                self.n_exchanges += 1
                self.bytes_exchanged += t.numel() * t.element_size()
            else:
                small.append((t, op))
        if not small:
            return
        buf = torch.cat([t.reshape(-1).to(torch.int64) for t, _ in small])
        n = int(buf.numel())
        flat = torch.empty(self.world * n, dtype=torch.int64, device=buf.device)
        self.td.all_gather_into_tensor(flat, buf, group=self.group)
        gathered = flat.view(self.world, n)
        self.n_exchanges += 1
        self.bytes_exchanged += n * 8
        off = [0]
        for t, _ in small:
            off.append(off[-1] + int(t.numel()))
        if buf.is_cuda:
            # merge adjacent segments with the same reduction (dr_combine_counts takes <= 32 segments)
            seg_off, seg_op = [0], []
            for (t, op), o in zip(small, off[1:]):
                if seg_op and seg_op[-1] == _RED[op]:
                    seg_off[-1] = o
                else:
                    seg_op.append(_RED[op])
                    seg_off.append(o)
            if len(seg_op) > 32:
                raise ValueError("too many segments in one exchange")
            ctx.combine_counts(gathered, self.world, n, seg_off, seg_op, buf)
        else:
            # CPU tensors only occur in the gloo tests of the host logic (no device, no library call)
            for (t, op), lo, hi in zip(small, off[:-1], off[1:]):
                g = gathered[:, lo:hi]
                buf[lo:hi] = {"sum": lambda x: x.sum(0), "min": lambda x: x.amin(0), "max": lambda x: x.amax(0),
                              "or": lambda x: torch.from_numpy(
                                  np.bitwise_or.reduce(x.numpy(), axis=0))}[op](g)
        for (t, _), lo, hi in zip(small, off[:-1], off[1:]):
            t.copy_(buf[lo:hi].view(t.shape))


class _PresenceMap:
    """{(x, y): bool [dom_x + 1, dom_y + 1]} over the packed presence bits of a pair_presence launch; a
    pair's matrix is only unpacked when somebody asks for it (the skip tables of the few counted pairs)."""

    def __init__(self, pairs, offs, words, dom):
        self._at = {p: q for q, p in enumerate(pairs)}
        self._offs, self._words, self._dom, self._cache = offs, words, dom, {}

    def __contains__(self, key):
        return key in self._at

    def __getitem__(self, key):
        if key not in self._cache:
            q = self._at[key]
            x, y = key
            n_e = (self._dom[x] + 1) * (self._dom[y] + 1)
            w = self._words[self._offs[q]:self._offs[q + 1]]
            b = np.unpackbits(w.view(np.uint8), bitorder="little")[:n_e].astype(bool)
            self._cache[key] = b.reshape(self._dom[x] + 1, self._dom[y] + 1)
        return self._cache[key]

    def get(self, key, default=None):
        return self[key] if key in self._at else default


class DetectResult:
    def __init__(self):
        self.bitmaps = {}            # attr -> device int32 words (noisy / error cells)
        self.noisy_columns = []
        self.target_columns = []
        self.pairwise_stats = {}
        self.domain_stats = {}
        self.disc_attrs = []
        self.n_cells = {}
        self.n_cells_detected = {}
        self.n_cells_global = {}
        self.weak_removed_dev = None


class Engine:
    def __init__(self, table, device_index=0, dist=None, device_table=None, ctx=None):
        import torch
        self.torch = torch
        self.ctx = ctx if ctx is not None else Context.acquire(device_index)
        self._launches0 = self.ctx.launch_count
        self.device = torch.device("cuda", device_index)
        torch.cuda.set_device(self.device)
        self.table = table
        self.dt = device_table if device_table is not None else DeviceTable(table, self.device, ctx=self.ctx)
        self.dist = dist
        self.n_rows = table.n_rows
        self.n_words = (self.dt.n_pad + 31) // 32
        self._hist_cache = {}
        self._raw_cache = {}     # attr -> global int64 counts of the raw column (slot 0 = NULL)
        self.disc_cols = {}      # attr -> device int32 column of the discretised table
        self.disc_dom = {}       # attr -> domain size of that column
        self.timings = {}
        self.trace = None        # list of (label, seconds since the previous mark) when tracing

    # ------------------------------------------------------------------------------------------
    @property
    def n_rows_global(self):
        return self.table.n_rows_global

    def pinned_i32(self, n):
        """Page-locked int32 staging of at least n elements, kept for the life of the engine
        (cudaHostAlloc of a few hundred MB per run would cost more than the copy it serves)."""
        buf = getattr(self, "_pinned", None)
        if buf is None or buf.numel() < n:
            buf = self.torch.empty(int(n * 1.25) + 1024, dtype=self.torch.int32, pin_memory=True)
            self._pinned = buf
        return buf[:n]

    def mark(self, label):
        """Tracing aid (bench.py --trace): device-synchronised wall-clock split points."""
        if self.trace is None:
            return
        self.torch.cuda.synchronize()
        now = time.perf_counter()
        self.trace.append((label, now - getattr(self, "_t_mark", now)))
        self._t_mark = now

    def new_bitmap(self):
        return self.torch.zeros(self.n_words, dtype=self.torch.int32, device=self.device)

    def _sync(self):
        self.torch.cuda.current_stream().synchronize()

    def bitmap_rows(self, bitmap, n=None, out=None, count=None):
        """Ascending row indices (device int32 tensor) of the set bits (written into `out` if given).
        With `count` (the popcount, e.g. from ctx.bitmap_count_many) there is no host round trip."""
        n = self.n_rows if n is None else n
        if count is not None:
            rows = out if out is not None else \
                self.torch.empty(max(count, 1), dtype=self.torch.int32, device=self.device)
            assert rows.numel() >= count
            if count:
                self.ctx.bitmap_to_rows_async(bitmap, n, rows, count)
            return rows[:count]
        cnt = self.ctx.bitmap_count(bitmap, n)
        rows = out if out is not None else \
            self.torch.empty(max(cnt, 1), dtype=self.torch.int32, device=self.device)
        assert rows.numel() >= cnt
        if cnt:
            self.ctx.bitmap_rows_after_count(bitmap, n, rows, cnt)  # reuses the block offsets of the count
        return rows[:cnt]

    # ---- a7: discretisation ------------------------------------------------------------------
    def discretize(self, discrete_thres):
        """convertToDiscretizedTable (RepairApi.scala:126-169) -> domain_stats; fills disc_cols."""
        assert 2 <= discrete_thres < 65536
        domain_stats = {}
        self.disc_cols, self.disc_dom = {}, {}
        for c in self.table.columns:
            ndv = c.dict_size
            domain_stats[c.name] = ndv
            if c.continuous:
                out = self.torch.full((self.dt.n_pad,), -1, dtype=self.torch.int32, device=self.device)
                if ndv > 0:
                    vmin, den = SH.discretize_params(c.kind, c.dictionary[0], c.dictionary[-1])
                    self.ctx.discretize(self.dt.val(c.name), self.n_rows, vmin, den, discrete_thres, out)
                self.disc_cols[c.name] = out
                self.disc_dom[c.name] = discrete_thres + 1
            elif 1 < ndv <= discrete_thres:
                self.disc_cols[c.name] = self.dt.col(c.name)
                self.disc_dom[c.name] = ndv
            else:
                _logger.warning("'{}' dropped because of its unsuitable domain (size={})".format(c.name, ndv))
        return domain_stats

    # ---- exchange helper -------------------------------------------------------------------------
    def exchange(self, parts):
        """Reduce count tensors across the shards (no-op on one GPU): ONE collective per call."""
        if self.dist is not None and parts:
            self.dist.exchange(self.ctx, parts)

    # ---- histograms ----------------------------------------------------------------------------
    def launch_scan_hist(self, attrs, null_bitmaps):
        """Launches the fused NULL scan + histogram over the discretised columns `attrs` without waiting
        for it.  -> [(attrs, doms, device int64 histogram)] for exchange() / _absorb_hists()."""
        out = []
        for i in range(0, len(attrs), 64):
            part = attrs[i:i + 64]
            dom = [self.disc_dom[a] for a in part]
            hist = self.torch.zeros(sum(d + 1 for d in dom), dtype=self.torch.int64, device=self.device)
            self.ctx.scan_hist([self.disc_cols[a] for a in part], dom, self.n_rows,
                               [null_bitmaps.get(a) for a in part], hist)
            out.append((part, dom, hist))
        return out

    def _absorb_hists(self, launched):
        for part, dom, hist in launched:
            h = hist.cpu().numpy()
            off = 0
            for a, d in zip(part, dom):
                self._hist_cache[a] = h[off:off + d + 1].copy()
                off += d + 1

    def scan_hist(self, attrs, null_bitmaps):
        """Fused NULL scan + histogram over discretised columns `attrs`; caches the (global) hist per attr."""
        if not attrs:
            return
        launched = self.launch_scan_hist(attrs, null_bitmaps)
        self.exchange([(h, "sum") for _, _, h in launched])
        self._absorb_hists(launched)

    def raw_value_counts(self, attr):
        """int64[dict_size + 1] counts of the RAW column (slot 0 = NULL), over all shards."""
        col = self.table.by_name[attr]
        if attr in self._hist_cache and not col.continuous and attr in self.disc_cols:
            return self._hist_cache[attr]
        if attr in self._raw_cache:
            return self._raw_cache[attr]
        hist = self.torch.zeros(col.dict_size + 1, dtype=self.torch.int64, device=self.device)
        self.ctx.scan_hist([self.dt.col(attr)], [col.dict_size], self.n_rows, [None], hist)
        self.exchange([(hist, "sum")])
        self._raw_cache[attr] = hist.cpu().numpy()
        return self._raw_cache[attr]

    # ---- detectors -----------------------------------------------------------------------------
    def _or_rows_into(self, row_bitmap, attrs, bitmaps):
        for a in attrs:
            if a not in bitmaps:
                bitmaps[a] = self.new_bitmap()
            self.ctx.bitmap_or(bitmaps[a], row_bitmap, self.n_rows)

    def detect_null(self, targets, bitmaps, fused):
        """NullErrorDetector: columns of the discretised table get their bits from the fused scan
        (`fused` collects them); the others take a NULL-only LUT scan of the raw codes."""
        for a in self.table.names:
            if a not in targets:
                continue
            if a not in bitmaps:
                bitmaps[a] = self.new_bitmap()
            col = self.table.by_name[a]
            if a in self.disc_cols and not col.continuous:
                fused[a] = bitmaps[a]
            else:
                self.ctx.lut_scan(self.dt.col(a), self.n_rows, None, 0, bitmaps[a])

    def detect_regex(self, attr, regex, targets, bitmaps):
        if attr not in targets or regex is None or regex.strip() == "" or attr not in self.table.by_name:
            return
        col = self.table.by_name[attr]
        pat = re.compile(regex)
        lut = np.fromiter((0 if pat.search(s) is not None else 1 for s in col.strings()), dtype=np.uint8,
                          count=col.dict_size)
        d_lut = self.torch.from_numpy(lut).to(self.device) if col.dict_size else None
        if attr not in bitmaps:
            bitmaps[attr] = self.new_bitmap()
        self.ctx.lut_scan(self.dt.col(attr), self.n_rows, d_lut, col.dict_size, bitmaps[attr])

    def domain_values_regex(self, attr, values, autofill, min_count_thres):
        """DomainValues._detect_impl (errors.py:112-129) -> regex or None (continuous attribute)."""
        if attr not in self.table.by_name:
            return "$^" if not values or autofill else "({})".format("|".join(values))
        col = self.table.by_name[attr]
        if col.continuous:
            return None
        domain_values = [] if autofill else list(values)
        if autofill:
            counts = self.raw_value_counts(attr)
            strs = col.strings()
            filled = [strs[c] for c in range(col.dict_size) if counts[c + 1] > min_count_thres]
            if filled:
                domain_values = filled
        return "({})".format("|".join(domain_values)) if domain_values else "$^"

    def detect_constraints(self, constraint_path, constraints, targets, bitmaps, ex_parts=None, after=None):
        """ConstraintErrorDetector (ErrorDetectorApi.scala:189-244).  Every constraint first builds its
        LOCAL tables (per-key bounds or projection-presence bits); they join the pass's exchange
        (`ex_parts`) and the row flags are set afterwards (`after`: closures run once the tables are
        global).  Called without ex_parts / after (stand-alone detector) it does both at once."""
        stmts = DC.load_statements(constraint_path, constraints)
        if not stmts:
            return
        now = ex_parts is None
        if now:
            ex_parts, after = [], []
        pred_lists = DC.parse_and_verify(stmts, [self.table.row_id] + self.table.names, self.table.name)
        for preds in pred_lists:
            attrs = [r for r in DC.references(preds) if r in targets]
            if not attrs:
                continue
            for a in attrs:
                if a not in bitmaps:
                    bitmaps[a] = self.new_bitmap()
            shape, payload = DC.classify(preds)
            rowmask = self.new_bitmap()
            if shape == "CONST":
                cols, ops, args = [], [], []
                for p in payload:
                    col = self.table.by_name[p.left]
                    lit, quoted = DC.constant_literal(p.right)
                    cols.append(self.dt.col(p.left))
                    ops.append(DR_OP[p.sign])
                    if p.sign in ("EQ", "IQ"):
                        args.append(col.code_of(lit))
                    else:
                        lo, hi = col.rank_bounds(lit)
                        args.append(lo if p.sign == "LT" else hi)
                self.ctx.dc_const(cols, ops, args, self.n_rows, rowmask)
                self._or_rows_into(rowmask, attrs, bitmaps)
            elif shape == "EQ_ONLY":
                rowmask.fill_(-1)
                self._or_rows_into(rowmask, attrs, bitmaps)
            elif shape in ("FD", "INEQ") and (self._key_space(payload[0]) <= MAX_FD_KEY_SPACE or
                                              (self.dist is None and self._key_space(payload[0]) < 2 ** 62)):
                if shape == "FD":
                    keys, b = payload
                    x, mode = self.dt.col(b), 0
                else:
                    keys, sign, b = payload
                    x, mode = self.dt.col(b), 1
                    if sign == "GT":   # "some row has a smaller b" = "some row has a larger reversed code"
                        dom = self.table.by_name[b].dict_size
                        x = self.torch.where(x >= 0, dom - 1 - x, x)
                self._flag_by_key_group(keys, x, mode, rowmask, attrs, bitmaps, ex_parts, after)
            else:
                self._generic_constraint(preds, rowmask, attrs, bitmaps, ex_parts, after)
        if now:
            self.exchange(ex_parts)
            for fn in after:
                fn()

    def _key_space(self, keys):
        space = 1
        for k in keys:
            space *= self.table.by_name[k].dict_size + 1
        return space

    def _flag_by_key_group(self, keys, x, mode, rowmask, attrs, bitmaps, ex_parts, after):
        """Rows whose NULL-safe key group (attributes `keys`) holds two distinct x (mode 0: EQ.. & IQ(x))
        or a larger x than their own (mode 1: EQ.. & LT(x)): per-key min / max of x + 1 in direct tables
        over the mixed-radix key space (idempotent reductions: the shards' tables combine in the exchange)."""
        torch = self.torch
        strides, space = [], 1
        for k in keys:
            strides.append(space)
            space *= self.table.by_name[k].dict_size + 1
        key_cols = [self.dt.col(k) for k in keys] or [x]
        if not keys:
            strides = [0]
        if space > MAX_FD_KEY_SPACE:
            # one GPU, key space beyond the direct tables: open-addressing hash table keyed by the 64-bit
            # mixed-radix key (sharded runs take the projection path of _generic_constraint instead)
            assert self.dist is None
            cap = 1 << max(1, (2 * max(self.n_rows, 1) - 1).bit_length())
            tkeys = torch.full((cap,), -1, dtype=torch.int64, device=self.device)
            lo = torch.full((cap,), 2 ** 31 - 1, dtype=torch.int32, device=self.device)
            hi = torch.full((cap,), -2 ** 31, dtype=torch.int32, device=self.device)
            self.ctx.dc_hash_build(key_cols, strides, x, self.n_rows, cap, tkeys, lo, hi)
            self.ctx.dc_hash_flag(key_cols, strides, x if mode == 1 else None, mode, self.n_rows, cap, tkeys, lo, hi,
                                  rowmask)
            self._or_rows_into(rowmask, attrs, bitmaps)
            return
        lo = torch.full((space,), 2 ** 31 - 1, dtype=torch.int32, device=self.device)
        hi = torch.full((space,), -2 ** 31, dtype=torch.int32, device=self.device)
        self.ctx.dc_fd_build(key_cols, strides, x, self.n_rows, space, lo, hi)
        ex_parts += [(lo, "min"), (hi, "max")]

        def flag():
            if mode == 0:
                self.ctx.dc_fd_flag(key_cols, strides, self.n_rows, space, lo, hi, rowmask)
            else:
                self.ctx.dc_lt_flag(key_cols, strides, x, self.n_rows, space, hi, rowmask)
            self._or_rows_into(rowmask, attrs, bitmaps)
        after.append(flag)

    def _value_ranks(self, a, b):
        """Rank LUTs (device int32, index code + 1, NULL -> -1) that put the values of attributes a and b
        into ONE order, so that t1.a can be compared with t2.b in rank space."""
        torch = self.torch
        ca, cb = self.table.by_name[a], self.table.by_name[b]
        if a == b:
            r = np.r_[-1, np.arange(ca.dict_size)].astype(np.int32)
            t = torch.from_numpy(r).to(self.device)
            return t, t
        if ca.continuous and cb.continuous:
            va, vb = np.asarray(ca.dictionary, dtype=np.float64), np.asarray(cb.dictionary, dtype=np.float64)
            allv = np.unique(np.concatenate([va, vb]))
            ra, rb = np.searchsorted(allv, va), np.searchsorted(allv, vb)
        else:   # strings compare as strings (a numeric side is compared through its CAST(.. AS STRING) form)
            sa, sb = ca.strings(), cb.strings()
            allv = sorted(set(sa) | set(sb))
            pos = {v: i for i, v in enumerate(allv)}
            ra, rb = np.array([pos[v] for v in sa], dtype=np.int64), np.array([pos[v] for v in sb], dtype=np.int64)
        ta = torch.from_numpy(np.r_[-1, ra].astype(np.int32)).to(self.device)
        tb = torch.from_numpy(np.r_[-1, rb].astype(np.int32)).to(self.device)
        return ta, tb

    def _generic_constraint(self, preds, rowmask, attrs, bitmaps, ex_parts, after):
        """Any two-tuple predicate list: `EXISTS t2: AND_p sign_p(t1.left_p, t2.right_p)` only depends on
        a row's projection onto the referenced attributes -> mark the projections that occur (one pass),
        decide every DISTINCT projection against the distinct projections of its equality group
        (dr_dc_exists), flag the rows whose projection violates (one pass)."""
        torch = self.torch
        if len(preds) > 8:
            raise ValueError("a denial constraint with more than 8 predicates")
        ref = DC.references(preds)
        dims = [self.table.by_name[a].dict_size + 1 for a in ref]
        strides, space = [], 1
        for d in dims:
            strides.append(space)
            space *= d
        cols = [self.dt.col(a) for a in ref]
        direct = space <= MAX_PROJECTION_BITS
        if direct:
            bits = torch.zeros((space + 31) // 32, dtype=torch.int32, device=self.device)
            self.ctx.key_presence(cols, strides, self.n_rows, space, bits)
            ex_parts.append((bits, "or"))
            local_keys = None
        else:
            if space >= 2 ** 62:
                raise ValueError("denial constraint projection space {} does not fit a 64-bit key".format(space))
            rk = torch.zeros(self.n_rows, dtype=torch.int64, device=self.device)
            for c, st in zip(cols, strides):
                rk += (c[:self.n_rows].to(torch.int64) + 1) * st
            local_keys = torch.unique(rk)

        def decide():
            if direct:
                w = bits.to(torch.int64) & 0xFFFFFFFF
                nz = torch.nonzero(w).reshape(-1)
                sh = torch.arange(32, device=self.device, dtype=torch.int64)
                hit = ((w[nz][:, None] >> sh[None, :]) & 1).bool()
                keys = (nz[:, None] * 32 + sh[None, :])[hit]
                keys = keys[keys < space]
            else:
                keys = local_keys
                if self.dist is not None:   # union of the shards' distinct projections
                    cnt = torch.tensor([keys.numel()], dtype=torch.int64, device=self.device)
                    sizes = [torch.zeros_like(cnt) for _ in range(self.dist.world)]
                    self.dist.td.all_gather(sizes, cnt, group=self.dist.group)
                    m = int(max(int(x.item()) for x in sizes))
                    pad = torch.full((m,), -1, dtype=torch.int64, device=self.device)
                    pad[:keys.numel()] = keys
                    allk = [torch.empty_like(pad) for _ in range(self.dist.world)]
                    self.dist.td.all_gather(allk, pad, group=self.dist.group)
                    keys = torch.unique(torch.cat(allk))
                    keys = keys[keys >= 0]
            n = int(keys.numel())
            if n == 0:
                return
            codes = {a: ((keys // st) % d - 1) for a, st, d in zip(ref, strides, dims)}     # int64, -1 = NULL
            eq_attrs = list(dict.fromkeys(p.left for p in preds if p.sign == "EQ" and p.left == p.right))
            gkey = torch.zeros(n, dtype=torch.int64, device=self.device)
            for a in eq_attrs:
                gkey = gkey * (self.table.by_name[a].dict_size + 1) + (codes[a] + 1)
            order = torch.argsort(gkey, stable=True)
            gs = gkey[order]
            begin = torch.searchsorted(gs, gs, right=False).to(torch.int32)
            end = torch.searchsorted(gs, gs, right=True).to(torch.int32)
            left, right, signs = [], [], []
            for p in preds:
                la, lb = self._value_ranks(p.left, p.right)
                left.append(la[(codes[p.left][order] + 1)].contiguous())
                right.append(lb[(codes[p.right][order] + 1)].contiguous())
                signs.append(DR_OP[p.sign])
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
            self.ctx.dc_exists(left, right, signs, n, begin, end, out)
            bad = keys[order][out.bool()]
            if bad.numel() == 0:
                return
            if direct:
                acc = torch.zeros((space + 31) // 32, dtype=torch.int64, device=self.device)
                acc.index_put_((bad >> 5,), torch.ones_like(bad) << (bad & 31), accumulate=True)
                viol = acc.to(torch.int32)     # distinct keys: the sum of distinct bits is their OR
                self.ctx.key_flag(cols, strides, self.n_rows, space, viol, rowmask)
            else:
                bad = torch.sort(bad).values
                rk2 = torch.zeros(self.n_rows, dtype=torch.int64, device=self.device)
                for c, st in zip(cols, strides):
                    rk2 += (c[:self.n_rows].to(torch.int64) + 1) * st
                idx = torch.searchsorted(bad, rk2).clamp_(max=bad.numel() - 1)
                flag = (bad[idx] == rk2).to(torch.int32)
                pad = torch.zeros(self.dt.n_pad, dtype=torch.int32, device=self.device)
                pad[:self.n_rows] = flag
                lut = torch.tensor([0, 1], dtype=torch.uint8, device=self.device)
                self.ctx.lut_scan(pad, self.n_rows, lut, 2, rowmask)
            self._or_rows_into(rowmask, attrs, bitmaps)
        after.append(decide)

    def detect_outliers(self, targets, bitmaps, approx_enabled=False):
        """GaussianOutlierErrorDetector (ErrorDetectorApi.scala:249-300).  `approx_enabled` asks Spark for
        percentile_approx; here the EXACT percentile is computed either way (documented deviation)."""
        for a in self.table.continuous_attrs:
            if a not in targets:
                continue
            if self.dist is None:
                q1, q3, n = self.ctx.quartiles(self.dt.val(a), self.n_rows)
            else:
                # sharded: order statistics from the global histogram of the (sorted-dictionary) codes
                col = self.table.by_name[a]
                if col.dict_size > (1 << 24):
                    raise NotImplementedError("sharded exact quartiles of an attribute with more than 2^24 "
                                              "distinct values")
                counts = np.asarray(self.raw_value_counts(a), dtype=np.int64)[1:]
                n = int(counts.sum())
                q1 = q3 = 0.0
                if n:
                    cum = np.cumsum(counts)
                    vals = np.asarray(col.dictionary, dtype=np.float64)
                    qs = []
                    for pct in (0.25, 0.75):
                        pos = (n - 1) * pct
                        lo_r, hi_r = int(np.floor(pos)), int(np.ceil(pos))
                        vlo = vals[int(np.searchsorted(cum, lo_r, side="right"))]
                        vhi = vals[int(np.searchsorted(cum, hi_r, side="right"))]
                        qs.append(vlo if lo_r == hi_r else (hi_r - pos) * vlo + (pos - lo_r) * vhi)
                    q1, q3 = qs
            if n == 0:
                continue
            lower, upper = q1 - 1.5 * (q3 - q1), q3 + 1.5 * (q3 - q1)
            if a not in bitmaps:
                bitmaps[a] = self.new_bitmap()
            self.ctx.range_flag(self.dt.val(a), self.n_rows, lower, upper, bitmaps[a])

    def _global_values(self, a):
        """-> (device float64 values of continuous attribute `a` over the whole table, first global row of this
        shard).  Sharded: one all-gather, rank order."""
        v = self.dt.val(a)[:self.n_rows]
        if self.dist is None:
            return v, 0
        col, counts = self.dist.all_gather_rows(v.contiguous())
        return col, int(sum(counts[:self.dist.rank]))

    def detect_lof(self, targets, bitmaps, k=20):
        """LOFOutlierErrorDetector (errors.py:302-312): exact one-dimensional local outlier factor of every
        continuous target, k = min(20, n - 1) like LocalOutlierFactor's default.  Sharded, every rank scores the
        gathered global column and sets the bits of its own rows only, so the union equals the one-GPU result."""
        ws = None
        for a in self.table.continuous_attrs:
            if a not in targets:
                continue
            col, row_begin = self._global_values(a)
            n = int(col.shape[0])
            if n < 2:
                continue
            if ws is None:
                ws = self.torch.empty(self.ctx.lof_workspace_bytes(n), dtype=self.torch.uint8, device=self.device)
            if a not in bitmaps:
                bitmaps[a] = self.new_bitmap()
            self.ctx.lof_flag(col, n, min(k, n - 1), row_begin, self.n_rows, bitmaps[a], ws)

    def detect_sklearn(self, targets, bitmaps, factory):
        """ScikitLearnBackedErrorDetector (errors.py:219-245): the user's estimator, built by `factory`, runs on
        the host over the global column with NULLs filled by the median (errors.py:237-238); `fit_predict` < 0
        flags a row.  Sharded, only rank 0 fits and one broadcast hands every rank the same answer."""
        import pandas as pd
        torch = self.torch
        for a in self.table.continuous_attrs:
            if a not in targets:
                continue
            col, row_begin = self._global_values(a)
            n = int(col.shape[0])
            flags = torch.zeros(n, dtype=torch.uint8, device=self.device)
            if self.dist is None or self.dist.rank == 0:
                vals = col.cpu().numpy()
                valid = ~np.isnan(vals)
                if n >= 2 and valid.any():
                    pdf = pd.DataFrame({a: vals})
                    pred = np.asarray(factory().fit_predict(pdf[[a]].fillna(np.median(vals[valid]))))
                    flags.copy_(torch.from_numpy((pred < 0).astype(np.uint8)))
            if self.dist is not None:
                td, group = self.dist.td, self.dist.group
                td.broadcast(flags, src=td.get_global_rank(group, 0) if group is not None else 0, group=group)
            mine = flags[row_begin:row_begin + self.n_rows].cpu().numpy()
            if not mine.any():
                continue
            words = np.zeros(self.n_words * 4, dtype=np.uint8)
            packed = np.packbits(mine, bitorder="little")
            words[:len(packed)] = packed
            if a not in bitmaps:
                bitmaps[a] = self.new_bitmap()
            self.ctx.bitmap_or(bitmaps[a], torch.from_numpy(words.view(np.int32)).to(self.device), self.n_rows)

    def bitmaps_from_cells(self, positions, attrs):
        """User-supplied error cells (setErrorCells) -> bitmaps, built on the host."""
        out = {}
        positions = np.asarray(positions, dtype=np.int64)
        attrs = np.asarray(attrs, dtype=object)
        for a in sorted(set(attrs.tolist())):
            pos = positions[attrs == a]
            words = np.zeros(self.n_words, dtype=np.uint32)
            np.bitwise_or.at(words, pos >> 5, (np.uint32(1) << (pos & 31).astype(np.uint32)))
            out[a] = self.torch.from_numpy(words.view(np.int32)).to(self.device)
        return out

    # ---- a8: pair statistics -----------------------------------------------------------------
    def _pair_layout(self, pairs, bits):
        offs = [0]
        for x, y in pairs:
            n = (self.disc_dom[x] + 1) * (self.disc_dom[y] + 1)
            offs.append(offs[-1] + ((n + 31) // 32 if bits else n))
        return offs

    def launch_pair_presence(self, pairs, full=False):
        """Distinct-pair presence bits on a row sample (the whole table when it is small or `full`), not
        waited for.  -> (pairs, word offsets, device bit words, covers_every_row)"""
        attrs = list(dict.fromkeys(a for p in pairs for a in p))
        if len(attrs) > 64:
            raise NotImplementedError("more than 64 discretised attributes")
        idx = {a: i for i, a in enumerate(attrs)}
        offs = self._pair_layout(pairs, bits=True)
        bits = self.torch.zeros(max(offs[-1], 1), dtype=self.torch.int32, device=self.device)
        block_rows = 512
        n_blocks = (self.n_rows + block_rows - 1) // block_rows
        if not full:
            n_blocks = min(n_blocks, PRESENCE_SAMPLE_ROWS // block_rows)
        covers = n_blocks * block_rows >= self.n_rows
        self.ctx.pair_presence([self.disc_cols[a] for a in attrs], [self.disc_dom[a] for a in attrs],
                               [idx[x] for x, _ in pairs], [idx[y] for _, y in pairs], offs, self.n_rows,
                               block_rows, n_blocks, bits)
        return pairs, offs, bits, covers

    def pair_presence_host(self, launched, check_cover=True):
        """-> ({frozenset pair: distinct count seen}, {pair: bool [dom_x+1, dom_y+1]} (decoded on demand), exact)"""
        pairs, offs, bits, covers = launched
        words = bits.cpu().numpy().view(np.uint32)
        exact = covers
        if self.dist is not None and check_cover:   # the sample is exact only if it covered every shard completely
            t = self.torch.tensor([1 if covers else 0], dtype=self.torch.int64, device=self.device)
            self.dist.min_(t)
            exact = bool(int(t.item()))
        # distinct counts of all pairs at once: popcount per word, summed per pair segment (bits past a pair's
        # last entry are never set by the kernel)
        pc = np.unpackbits(words.view(np.uint8)).reshape(-1, 32).sum(axis=1, dtype=np.int64) if len(words) else \
            np.zeros(0, dtype=np.int64)
        cum = np.concatenate([[0], np.cumsum(pc)])
        o = np.asarray(offs, dtype=np.int64)
        counts = cum[np.minimum(o[1:], len(pc))] - cum[np.minimum(o[:-1], len(pc))]
        nnz = {frozenset(p): int(c) for p, c in zip(pairs, counts.tolist())}
        return nnz, _PresenceMap(pairs, offs, words, self.disc_dom), exact

    def pair_nnz_lower_bounds(self, pairs):
        """distinct-pair counts on a row sample (exact when the sample covers the table)."""
        launched = self.launch_pair_presence(pairs)
        self.exchange([(launched[2], "or")])
        nnz, _, exact = self.pair_presence_host(launched)
        return nnz, exact

    def pair_tables(self, pairs, present=None, presence_only=()):
        """Exact co-occurrence tables {(x, y): int64[dom_x+1, dom_y+1]} for `pairs` (over all shards).
        For every x value ONE partner y is left uncounted by the kernel and restored here from the
        column histogram (dr_cooc_skip): the partner that is most frequent overall among those seen
        with x in the presence sample -- on correlated pairs that removes nearly all shared-memory
        atomics, which are what bounds the kernel.  The kernel sees every pair with the LARGER domain as
        x (a determinant has one partner per value; the dependent has several).
        presence_only: pairs for which only the exact distinct-pair count is wanted (full-table
        presence bits, no atomics); both travel in ONE exchange.  -> (tables, {frozenset: nnz})"""
        if not pairs and not presence_only:
            return {}, {}
        attrs = list(dict.fromkeys(a for p in list(pairs) + list(presence_only) for a in p))
        if len(attrs) > 64:
            raise NotImplementedError("more than 64 discretised attributes")
        need = [a for a in attrs if a not in self._hist_cache]
        self.scan_hist(need, {})
        parts, launched_p = [], None
        if presence_only:
            launched_p = self.launch_pair_presence(list(presence_only), full=True)
            parts.append((launched_p[2], "or"))
        kp, offs, skip, skip_off, out = [], [0], [], [0], None
        if pairs:
            for (x, y) in pairs:   # kernel orientation: larger domain first
                kp.append((x, y) if self.disc_dom[x] >= self.disc_dom[y] else (y, x))
            idx = {a: i for i, a in enumerate(attrs)}
            offs = self._pair_layout(kp, bits=False)
            for (x, y) in kp:
                hy = np.asarray(self._hist_cache[y], dtype=np.int64)
                pres = None
                if present is not None:
                    pres = present.get((x, y))
                    if pres is None and (y, x) in present:
                        pres = present[(y, x)].T
                if pres is None:
                    lut = np.full(self.disc_dom[x] + 1, int(np.argmax(hy)), dtype=np.int32)
                else:
                    sc = np.where(pres, hy[None, :] + 1, 0)
                    lut = np.where(sc.max(axis=1) > 0, np.argmax(sc, axis=1), int(np.argmax(hy))).astype(np.int32)
                skip.append(lut)
                skip_off.append(skip_off[-1] + len(lut))
            d_skip = self.torch.from_numpy(np.concatenate(skip)).to(self.device)
            out = self.torch.zeros(offs[-1], dtype=self.torch.int64, device=self.device)
            self.ctx.cooc_skip([self.disc_cols[a] for a in attrs], [self.disc_dom[a] for a in attrs],
                               [idx[x] for x, _ in kp], [idx[y] for _, y in kp], offs, self.n_rows, d_skip,
                               skip_off, out)
            parts.append((out, "sum"))
        self.exchange(parts)
        tables, nnz = {}, {}
        if pairs:
            h = out.cpu().numpy()
            for q, ((x, y), (kx, ky)) in enumerate(zip(pairs, kp)):
                tab = h[offs[q]:offs[q + 1]].reshape(self.disc_dom[kx] + 1, self.disc_dom[ky] + 1).copy()
                rows = np.arange(tab.shape[0])
                tab[rows, skip[q]] = 0
                tab[rows, skip[q]] = np.asarray(self._hist_cache[kx], dtype=np.int64) - tab.sum(axis=1)
                tables[(x, y)] = tab if (kx, ky) == (x, y) else np.ascontiguousarray(tab.T)
                nnz[frozenset((x, y))] = int(np.count_nonzero(tab))
        if launched_p is not None:
            got, _, _ = self.pair_presence_host(launched_p, check_cover=False)
            nnz.update(got)
        return tables, nnz

    def compute_attr_stats(self, targets, domain_stats, attr_freq_thr, pairwise_thr, max_attrs, presence=None):
        """computeAttrStats (RepairApi.scala:396-477) -> (pairwise_stats, tables, having).
        presence: (nnz lower bounds, presence matrices, exact) of a pair sample that was already taken
        (detect() launches it together with the first scan)."""
        disc_attrs = list(self.disc_cols.keys())
        cands = SH.candidate_pairs(targets, disc_attrs)
        scoring = [t for t in targets if len(cands[t]) > max_attrs]

        def uniq(pairs):
            seen, out = set(), []
            for p in pairs:
                k = frozenset(p)
                if k not in seen:
                    seen.add(k)
                    out.append(p)
            return out

        selected = {t: list(cands[t]) for t in targets if t not in scoring}
        tables, present = {}, None
        if scoring:
            all_scored = uniq([p for t in scoring for p in cands[t]])
            if presence is not None and all(frozenset(p) in presence[0] for p in all_scored):
                lower, present, exact = presence
            else:
                launched = self.launch_pair_presence(all_scored)
                self.exchange([(launched[2], "or")])
                lower, present, exact = self.pair_presence_host(launched)
            if exact:
                for t in scoring:
                    selected[t] = SH.select_scored(cands[t], lower, domain_stats, pairwise_thr, max_attrs)
            else:
                und = {t: SH.undecided(cands[t], lower, domain_stats, pairwise_thr) for t in scoring}
                # counted now: per target the `max_attrs` undecided pairs with the smallest lower bounds,
                # unless the bound is already within 5 % of the threshold -- those (typically pairs of
                # independent attributes the sample missed a few rare combinations of) only get their exact
                # distinct count from full-table presence bits; a pair that is selected after all is
                # counted with the `missing` ones below
                count_now, count_set = [p for t in selected for p in selected[t]], set()
                for t in scoring:
                    ranked = sorted(und[t], key=lambda pr: lower[frozenset(pr)] / float(
                        max(domain_stats[pr[0]] * domain_stats[pr[1]], 1)))
                    for pr in ranked[:max_attrs]:
                        den = float(max(domain_stats[pr[0]] * domain_stats[pr[1]], 1))
                        if lower[frozenset(pr)] / den < 0.95 * pairwise_thr:
                            count_now.append(pr)
                count_now = uniq(count_now)
                count_set = {frozenset(p) for p in count_now}
                only_nnz = [p for p in uniq([p for t in scoring for p in und[t]]) if frozenset(p) not in count_set]
                tables, nnz = self.pair_tables(count_now, present, only_nnz)
                for t in scoring:
                    selected[t] = SH.select_scored(und[t], nnz, domain_stats, pairwise_thr, max_attrs)
        pairs = [p for t in targets for p in selected[t]]
        missing = [p for p in uniq(pairs) if p not in tables and (p[1], p[0]) not in tables]
        tables.update(self.pair_tables(missing, present)[0])
        having = SH.having_threshold(self.n_rows_global, attr_freq_thr)
        need_hist = [a for a in disc_attrs if a not in self._hist_cache]
        self.scan_hist(need_hist, {})
        stats = SH.pairwise_entropies(self.n_rows_global, self._hist_cache, tables, pairs, domain_stats, having)
        for t in targets:
            stats.setdefault(t, [])
        return stats, tables, having

    # ---- a9: weak-label domain analysis --------------------------------------------------------
    def prune_weak_labels(self, res, tables, having, continuous, max_attrs_domains, alpha, beta, keep_scores=False):
        """Cells whose current value is the top-1 candidate of the naive-Bayes domain analysis are not
        errors (errors.py:507-530).  All targets in ONE call (dr_domain_prune: top-1 per combination of
        correlated values, then a bitmap-driven look-up): the count tables of every target travel in one
        host->device copy and nothing comes back.  keep_scores (tests) / targets with too many
        combinations take the per-cell kernel (dr_domain_score), one launch per target."""
        torch = self.torch
        work = []
        for t in res.target_columns:
            corr = res.pairwise_stats.get(t, [])[:max_attrs_domains]
            if t in continuous or not corr or t not in res.bitmaps or int(res.n_cells.get(t, 0)) == 0:
                continue
            hist_t = SH.apply_having(self._hist_cache[t], having).astype(np.int64)
            items = []
            for a, _ in corr:
                tab = tables[(t, a)].T if (t, a) in tables else tables[(a, t)]
                tab = SH.apply_having(np.ascontiguousarray(tab), having).astype(np.int64)  # [dom_a+1, dom_t+1]
                items.append((a, np.ascontiguousarray(tab).reshape(-1), self.disc_dom[a],
                              SH.tau_for(alpha, self.n_rows_global, res.domain_stats[a], res.domain_stats[t])))
            work.append((t, hist_t, items))
        removed = torch.zeros(max(len(work), 1), dtype=torch.int64, device=self.device)
        res.weak_removed_dev = removed
        if not work:
            return removed
        combos_ok = all(np.prod([float(d + 1) for _, _, d, _ in items]) <= (1 << 20) and len(items) <= 8
                        for _, _, items in work)
        if combos_ok and not keep_scores and not getattr(self, "domain_per_cell", False):
            parts, offs = [], []
            for t, hist_t, items in work:
                offs.append(sum(len(p) for p in parts))
                parts.append(hist_t)
                for _, tab, _, _ in items:
                    offs.append(sum(len(p) for p in parts))
                    parts.append(tab)
            # (running offsets computed incrementally: the lists are short)
            flat = torch.from_numpy(np.concatenate(parts)).to(self.device)
            base, k, targets = flat.data_ptr(), 0, []
            for t, hist_t, items in work:
                h_ptr = base + 8 * offs[k]
                k += 1
                corr = []
                for a, tab, dom_c, tau in items:
                    corr.append((self.disc_cols[a], base + 8 * offs[k], dom_c, tau))
                    k += 1
                targets.append((self.disc_cols[t], res.bitmaps[t], h_ptr, self.disc_dom[t], corr))
            self.ctx.domain_prune(targets, self.n_rows, self.n_rows_global, beta, removed)
            self._domain_flat = flat   # stays alive until the next pass (the call above synchronised anyway)
            return removed
        for i, (t, hist_t, items) in enumerate(work):
            n = int(res.n_cells.get(t, 0))
            rows = self.bitmap_rows(res.bitmaps[t], count=n)
            cooc = [torch.from_numpy(tab).to(self.device) for _, tab, _, _ in items]
            top1 = torch.empty(n, dtype=torch.int32, device=self.device)
            prob = torch.empty(n, dtype=torch.float64, device=self.device)
            weak = torch.empty(n, dtype=torch.uint8, device=self.device)
            self.ctx.domain_score(rows, n, self.disc_cols[t], self.disc_dom[t], [self.disc_cols[a] for a, _, _, _ in items],
                                  [d for _, _, d, _ in items], cooc, torch.from_numpy(hist_t).to(self.device),
                                  [tau for _, _, _, tau in items], self.n_rows_global, beta, top1, prob, weak)
            self.ctx.bitmap_clear_rows(res.bitmaps[t], rows, weak, n)
            removed[i] += weak.sum()
            res.last_domain = (rows, top1, prob, weak)
        return removed

    # ---- ErrorModel.detect -----------------------------------------------------------------------
    def detect(self, detectors, targets, discrete_thres, opts, given_cells=None):
        """detectors: list of dicts {"type": null|domain|regex|constraint|outlier|lof|sklearn, ...}
        given_cells: optional (positions, attrs) supplied by setErrorCells.

        Pass structure (the same on one GPU and on G shards; exchange() is the only cross-GPU step):
          local 1   fused NULL scan + histograms, constant / LUT detectors, per-key tables and projection
                    bits of the constraints, pair presence on a row sample
          exchange  [histograms | key tables | projection bits | presence bits]
          local 2   constraint flags, detectors that need global counts; cell counts
          exchange  [cell counts]                                   (a few int64)
          local 3   exact tables of the undecided / selected pairs
          exchange  [pair tables]
          local 4   domain scoring, pruning"""
        res = DetectResult()
        continuous = self.table.continuous_attrs
        target_attrs = [a for a in self.table.names if not targets or a in set(targets)]
        res.domain_stats = self.discretize(discrete_thres)
        res.disc_attrs = list(self.disc_cols.keys())
        bitmaps, fused = {}, {}
        ex1, after = [], []
        if given_cells is not None:
            bitmaps = self.bitmaps_from_cells(*given_cells)
        else:
            for det in detectors:
                own = det.get("targets") or []
                tg = [a for a in target_attrs if a in set(own)] if own else target_attrs
                kind = det["type"]
                if kind == "null":
                    self.detect_null(tg, bitmaps, fused)
                elif kind == "regex":
                    self.detect_regex(det["attr"], det["regex"], tg, bitmaps)
                elif kind == "domain":
                    if det["attr"] in tg:
                        if det.get("autofill", False) and det["attr"] in self.table.by_name and \
                                not self.table.by_name[det["attr"]].continuous:
                            if det["attr"] not in bitmaps:
                                bitmaps[det["attr"]] = self.new_bitmap()

                            def autofill(det=det, tg=tg):   # needs the GLOBAL value counts
                                rx = self.domain_values_regex(det["attr"], det.get("values", []), True,
                                                              det.get("min_count_thres", 12))
                                if rx is not None:
                                    self.detect_regex(det["attr"], rx, tg, bitmaps)
                            after.append(autofill)
                        else:
                            rx = self.domain_values_regex(det["attr"], det.get("values", []),
                                                          det.get("autofill", False), det.get("min_count_thres", 12))
                            if rx is not None:
                                self.detect_regex(det["attr"], rx, tg, bitmaps)
                elif kind == "constraint":
                    self.detect_constraints(det.get("path", ""), det.get("constraints", ""), tg, bitmaps, ex1, after)
                elif kind == "outlier":
                    self.detect_outliers(tg, bitmaps, det.get("approx", False))
                elif kind == "lof":
                    self.detect_lof(tg, bitmaps)
                elif kind == "sklearn":
                    self.detect_sklearn(tg, bitmaps, det["factory"])
                else:
                    raise ValueError("unknown detector type: {}".format(kind))
        # local 1 (cont.): one fused pass for the NULL bits of the discretised targets + every histogram,
        # and the presence sample of every pair that may have to be scored
        launched = self.launch_scan_hist([a for a in res.disc_attrs if a not in self._hist_cache], fused)
        max_attrs = opts["error.max_attrs_to_compute_pairwise_stats"]
        potential = [a for a in self.table.names if a in bitmaps and a in self.disc_cols]
        sup = SH.candidate_pairs(potential, res.disc_attrs)
        seen, scored = set(), []
        for t in potential:
            if len(sup[t]) > max_attrs:
                for pr in sup[t]:
                    if frozenset(pr) not in seen:
                        seen.add(frozenset(pr))
                        scored.append(pr)
        pres_launched = self.launch_pair_presence(scored) if scored and len(res.disc_attrs) <= 64 else None
        self.mark("detect:local 1 launched")
        # (sharded: "did the presence sample cover every shard completely" rides in the same collective)
        cover = None
        if pres_launched and self.dist is not None:
            cover = self.torch.tensor([1 if pres_launched[3] else 0], dtype=self.torch.int64, device=self.device)
        self.exchange(ex1 + [(h, "sum") for _, _, h in launched] +
                      ([(pres_launched[2], "or")] if pres_launched else []) +
                      ([(cover, "min")] if cover is not None else []))
        self._absorb_hists(launched)
        presence = self.pair_presence_host(pres_launched, check_cover=False) if pres_launched else None
        if cover is not None:
            presence = (presence[0], presence[1], bool(int(cover.item())))
        self.mark("detect:hists + presence on the host")
        for fn in after:        # local 2: flags that needed the global tables / counts
            fn()
        res.bitmaps = bitmaps
        names_b = list(bitmaps.keys())
        local = self.ctx.bitmap_count_many(list(bitmaps.values()), self.n_rows)
        res.n_cells = dict(zip(names_b, local))
        res.n_cells_detected = dict(res.n_cells)     # before the weak-label pruning of the domain analysis
        glob = local
        if self.dist is not None and names_b:
            t = self.torch.tensor(local, dtype=self.torch.int64, device=self.device)
            self.exchange([(t, "sum")])
            glob = [int(v) for v in t.cpu().numpy()]
        res.n_cells_global = dict(zip(names_b, glob))
        self.mark("detect:flags + cell counts")
        if sum(glob) == 0:
            res.domain_stats = {}
            return res
        res.noisy_columns = [a for a in self.table.names if res.n_cells_global.get(a, 0) > 0]
        if len(res.disc_attrs) == 0:
            res.domain_stats = {}
            return res
        res.target_columns = [a for a in res.noisy_columns if a in self.disc_cols]
        if len(res.target_columns) == 0 or len(res.disc_attrs) <= 1:
            return res
        stats, tables, having = self.compute_attr_stats(
            res.target_columns, res.domain_stats, opts["error.attr_freq_ratio_threshold"],
            opts["error.pairwise_freq_ratio_threshold"], max_attrs, presence)
        res.pairwise_stats = stats
        self.mark("detect:attribute statistics")
        if given_cells is None:
            self.prune_weak_labels(res, tables, having, continuous, opts["error.max_attrs_to_compute_domains"],
                                   opts["error.domain_threshold_alpha"], opts["error.domain_threshold_beta"])
            res.n_cells = dict(zip(res.bitmaps.keys(),
                                   self.ctx.bitmap_count_many(list(res.bitmaps.values()), self.n_rows)))
            self.mark("detect:domain analysis")
        return res

    # ---- cell frames -----------------------------------------------------------------------------
    def cells_of(self, res, attrs=None):
        """-> list of (attr, row positions np.int64, current codes np.int32) for the error cells."""
        out = []
        for a in self.table.names:
            if a not in res.bitmaps or (attrs is not None and a not in attrs):
                continue
            rows = self.bitmap_rows(res.bitmaps[a])
            n = int(rows.numel())
            if n == 0:
                continue
            cur = self.torch.empty(n, dtype=self.torch.int32, device=self.device)
            self.ctx.gather(self.dt.col(a), rows, n, cur)
            out.append((a, rows.cpu().numpy().astype(np.int64), cur.cpu().numpy()))
        return out

    # ---- repair ----------------------------------------------------------------------------------
    def build_dirty_tile(self, res, target_columns):
        """a10: dirty rows (rows with >= 1 error cell in a target column) gathered row-major with the
        error cells masked to NULL.  -> (dirty_rows, tile int32 [D, K], ctile float64 [D, Kc])"""
        rowmask = self.new_bitmap()
        for a in target_columns:
            if a in res.bitmaps:
                self.ctx.bitmap_or(rowmask, res.bitmaps[a], self.n_rows)
        drows = self.bitmap_rows(rowmask)
        D = int(drows.numel())
        K = len(self.table.columns)
        masks = [res.bitmaps.get(c.name) if c.name in target_columns else None for c in self.table.columns]
        tile = self.torch.empty((max(D, 1), K), dtype=self.torch.int32, device=self.device)
        # NULL bitmap of every tile column, taken while gathering (the chain's work lists)
        self.tile_nulls = self.torch.zeros((K, (D + 31) // 32 + 1), dtype=self.torch.int32, device=self.device)
        self.ctx.gather_rows_masked([self.dt.col(c.name) for c in self.table.columns], masks, drows, D, tile,
                                    null_out=self.tile_nulls)
        cont = [c for c in self.table.columns if c.continuous]
        ctile = None
        if cont:
            ctile = self.torch.empty((max(D, 1), len(cont)), dtype=self.torch.float64, device=self.device)
            cmasks = [res.bitmaps.get(c.name) if c.name in target_columns else None for c in cont]
            self.ctx.gather_rows_masked([self.dt.val(c.name) for c in cont], cmasks, drows, D, ctile, f64=True)
        return drows, tile, ctile

    def sample_rows_masked(self, res, target_columns, rows_np):
        """Training sample: the listed LOCAL rows of the repair base (error cells masked), on the host.
        Sharded: every rank contributes its rows and receives the whole sample, in global row order."""
        rows = self.torch.from_numpy(np.ascontiguousarray(rows_np, dtype=np.int32)).to(self.device)
        n = len(rows_np)
        K = len(self.table.columns)
        masks = [res.bitmaps.get(c.name) if c.name in target_columns else None for c in self.table.columns]
        tile = self.torch.empty((max(n, 1), K), dtype=self.torch.int32, device=self.device)
        self.ctx.gather_rows_masked([self.dt.col(c.name) for c in self.table.columns], masks, rows, n, tile)
        tile = tile[:n]
        cont = [c for c in self.table.columns if c.continuous]
        ctile = None
        if cont:
            ctile = self.torch.empty((max(n, 1), len(cont)), dtype=self.torch.float64, device=self.device)
            cmasks = [res.bitmaps.get(c.name) if c.name in target_columns else None for c in cont]
            self.ctx.gather_rows_masked([self.dt.val(c.name) for c in cont], cmasks, rows, n, ctile, f64=True)
            ctile = ctile[:n]
        if self.dist is not None:
            tile, _ = self.dist.all_gather_rows(tile.contiguous())
            if ctile is not None:
                ctile, _ = self.dist.all_gather_rows(ctile.contiguous())
        return tile.cpu().numpy(), (ctile.cpu().numpy() if ctile is not None else None)

    def valid_training_rows(self, res, y, max_rows, seed=42):
        """Rows whose y is non-NULL after masking; at most `max_rows` of the WHOLE table, seeded choice
        without replacement in table order (stand-in for the unseeded df.sample, model.py:755-766).
        -> (local row positions chosen on this shard, global positions of the whole sample, #valid rows
        of the whole table).  A sharded run draws exactly the rows the one-GPU run draws."""
        invalid = self.new_bitmap()
        self.ctx.lut_scan(self.dt.col(y), self.n_rows, None, 0, invalid)  # NULL cells
        if y in res.bitmaps:
            self.ctx.bitmap_or(invalid, res.bitmaps[y], self.n_rows)
        valid = self.torch.bitwise_not(invalid)
        n_local = self.ctx.bitmap_count(valid, self.n_rows)
        before, n_valid = 0, n_local
        if self.dist is not None:
            t = self.torch.tensor([n_local], dtype=self.torch.int64, device=self.device)
            counts = self.torch.empty(self.dist.world, dtype=self.torch.int64, device=self.device)
            self.dist.td.all_gather_into_tensor(counts, t, group=self.dist.group)
            counts = [int(c) for c in counts.cpu()]
            before, n_valid = sum(counts[:self.dist.rank]), sum(counts)
        if n_valid == 0:
            return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 0
        rows = self.bitmap_rows(valid) if n_local else self.torch.zeros(0, dtype=self.torch.int32, device=self.device)
        if n_valid > max_rows:
            rng = np.random.default_rng(seed)
            idx = np.sort(rng.choice(n_valid, size=max_rows, replace=False))
            idx = idx[(idx >= before) & (idx < before + n_local)] - before
            rows = rows[self.torch.from_numpy(idx).to(self.device)]
        local = rows.cpu().numpy().astype(np.int64)
        glob = local + self.table.row_offset
        if self.dist is not None:
            g, _ = self.dist.all_gather_rows(self.torch.from_numpy(glob).to(self.device))
            glob = g.cpu().numpy()
        return local, glob, n_valid

    def reset(self):
        """Forget per-run state so that the same resident table can be processed again."""
        self._hist_cache = {}
        self._raw_cache = {}
        self.disc_cols, self.disc_dom = {}, {}

    @property
    def launches(self):
        """Kernels launched through this engine's context since the engine was created."""
        return self.ctx.launch_count - self._launches0

    def close(self):
        Context.release(self.ctx)
