"""The spec decoder's predicate bits (lz4_decode_spec.cu, BITS != 0) on top of the lane-exact decoder model.

The rule: each 256-word chunk of a block's output gets its bits exactly once, from the step that moves the output position
past the chunk's end -- a batch (at most 33 words, so the chunk is still in the ring: read from there, words before
ring_from from global memory) or a one-sequence step (global memory) --, and the last partial chunk after the block, with
bits at and past the last row zero.

The rule is layered onto the batch rules of models/spec_model.py as they are: its source is taken and the flush is added
at the points where the kernel makes it (every place the output position moves, and the block's end).  Each of those
points must be found exactly once, so a change to the decoder model that moves them fails here loudly instead of leaving a
stale copy of the batch rules behind."""
import inspect

from models import spec_model

_FLUSH = '''
    bits={}
    def flush(w0,w1,rf):
        for g in range(w0,w1,32):
            m=0
            for j in range(32):
                w=g+j
                if w>=w1: continue
                if w>=rf:
                    v=ring[w&(RING-1)]
                    assert v is not None and v==w64(w), ('bits: ring',w)
                else: v=w64(w)
                m|=int(bool(test(v)))<<j
            assert g>>5 not in bits, ('bits: word flushed twice',g>>5)
            bits[g>>5]=m
    def adv_op(adv):
        nonlocal op
        nop=op+adv
        if (nop^op)>>11: flush(((nop>>11)<<8)-256,(nop>>11)<<8,ring_from)
        op=nop
'''

# (anchor in spec_model.py, what it becomes)
_EDITS = [
    ("def decode_block_spec(src, origin):", "def decode_block_spec(src, origin, test):"),
    ("        out[8*w:8*w+8]=v.to_bytes(8,'little'); ring[w&(RING-1)]=v\n",
     "        out[8*w:8*w+8]=v.to_bytes(8,'little'); ring[w&(RING-1)]=v\n" + _FLUSH),
    ("ip=nip; op+=8*33; x=nx;", "ip=nip; adv_op(8*33); x=nx;"),
    ("ip=nip; op+=256; x=nx;", "ip=nip; adv_op(256); x=nx;"),
    ("ip=nip; op+=8*(32 if FB else n+W_s); x=nx;", "ip=nip; adv_op(8*(32 if FB else n+W_s)); x=nx;"),
    ("            stats['one']+=1\n", "            stats['one']+=1\n            op_old=op\n"),
    ("            ring_from=(op+7)>>3\n",
     "            if (op_old^op)>>11: flush((op_old>>11)<<8,(op>>11)<<8,1<<62)\n            ring_from=(op+7)>>3\n"),
    ("    return bytes(out),stats\n",
     "    flush((origin>>11)<<8,origin>>3,1<<62)\n"
     "    nw=((origin>>3)+31)>>5\n"
     "    assert sorted(bits)==list(range(nw)), 'bits: a mask word missing'\n"
     "    return bytes(out),stats,[bits[k] for k in range(nw)]\n"),
]


def _build():
    src = inspect.getsource(spec_model)
    for anchor, repl in _EDITS:
        assert src.count(anchor) == 1, f"spec_model.py changed: {anchor!r} is not there exactly once"
        src = src.replace(anchor, repl)
    ns = {}
    exec(compile(src, "<spec_model with predicate bits>", "exec"), ns)
    return ns["decode_block_spec"]


_decode = _build()


def decode_block_spec_bits(src, origin, test):
    """Decodes like models.spec_model.decode_block_spec and writes the selection bits of `test` (a predicate on the 64-bit
    output words) as the kernel does.  Returns (decoded bytes, batch-shape stats, one 32-bit mask word per 32 rows)."""
    return _decode(src, origin, test)
