"""Recorded answers of the reference's modules, for tests that run this project's Erlang code (erlang/*.erl, tools/*.erl)
under the evaluator: that code calls into erlamsa_main, erlamsa_mutations, erlamsa_cmdparse, ... and the reference's
sources are not part of this repository.

TEST INFRASTRUCTURE (oracle/).  A `Calls` table is attached to a Runtime.  Every call from outside the reference into one
of its modules -- from the project's modules or from the test itself -- is answered from the table:

  record mode  the reference's sources are present (refrun.available()): the call runs there, its answer (or the Erlang
               exception it raised) is stored under a digest of (module, function, arguments); save() writes the table as JSON;
  replay mode  the stored answer is returned; a call that was never recorded (other arguments than the reference was
               asked about) is an error, so the project's side still has to ask exactly what it asked when recorded.

Calls the reference makes inside itself are not intercepted.  Funs in an answer are stored as an atom naming them:
an answer is data for the caller, not code to run."""
import hashlib
import json
import os

from .interp import Bif, Fun
from .terms import NIL, Bits, Cons, ErlError, fmt_term


def encode(x):
    t = type(x)
    if t is int:
        return x
    if t is float:
        return ["f", x]
    if t is str:
        return ["a", x]
    if t is bytes or t is bytearray:
        return ["b", bytes(x).hex()]
    if t is tuple:
        return ["t", [encode(y) for y in x]]
    if x is NIL:
        return ["l", []]
    if t is Cons:
        items = []
        while type(x) is Cons:
            items.append(encode(x.h))
            x = x.t
        return ["l", items] if x is NIL else ["il", items, encode(x)]
    if t is dict:
        return ["m", sorted(([encode(k), encode(v)] for k, v in x.items()), key=lambda kv: json.dumps(kv, sort_keys=True))]
    if t is Bits:
        return ["bits", x.val, x.nbits]
    if t is Fun or t is Bif:
        return ["a", "$fun %s:%s/%d" % (getattr(x, "module", "bif"), x.name, x.arity)]
    raise TypeError("cannot record a %s" % t.__name__)


def decode(x):
    if type(x) is int:
        return x
    tag = x[0]
    if tag == "f":
        return x[1]
    if tag == "a":
        return x[1]
    if tag == "b":
        return bytes.fromhex(x[1])
    if tag == "t":
        return tuple(decode(y) for y in x[1])
    if tag == "l" or tag == "il":
        tail = decode(x[2]) if tag == "il" else NIL
        for y in reversed(x[1]):
            tail = Cons(decode(y), tail)
        return tail
    if tag == "m":
        return {decode(k): decode(v) for k, v in x[1]}
    if tag == "bits":
        return Bits(x[1], x[2])
    raise ValueError("unknown tag %r" % (tag,))


class NotRecorded(RuntimeError):
    """a RuntimeError, so that the evaluator passes it through instead of turning it into an Erlang badarg"""


class Calls(object):
    def __init__(self, path, record):
        self.path = path
        self.record = record
        self.table = {}
        self.modules = set()
        if not record:
            with open(path) as f:
                d = json.load(f)
            self.modules = set(d["modules"])
            self.table = {e["key"]: e for e in d["calls"]}

    def attach(self, rt, ref_src=None):
        """answer rt's calls into the reference's modules from this table (record mode: ref_src is the reference's source dir)"""
        resolve = rt.resolve
        depth = [0]

        def key_of(mod, name, args):
            text = json.dumps([mod, name, [encode(a) for a in args]], sort_keys=True, separators=(",", ":"))
            return "%s:%s/%d %s" % (mod, name, len(args), hashlib.sha256(text.encode()).hexdigest())

        def recorded(mod, name, arity):
            def fn(*args):
                key = key_of(mod, name, args)
                if key not in self.table:
                    raise NotRecorded("call not recorded: %s %s" % (key, [fmt_term(a)[:200] for a in args]))
                e = self.table[key]
                if "raised" in e:
                    raise ErlError(e["raised"][0], decode(e["raised"][1]))
                return decode(e["returned"])
            return Bif(fn, arity, "%s:%s" % (mod, name))

        def recording(mod, name, arity):
            real = resolve(mod, name, arity)

            def fn(*args):
                key = key_of(mod, name, args)
                depth[0] += 1
                try:
                    res = rt.apply_fun(real, list(args))
                except ErlError as ex:
                    self.table[key] = {"key": key, "raised": [ex.cls, encode(ex.reason)]}
                    raise
                finally:
                    depth[0] -= 1
                self.table[key] = {"key": key, "returned": encode(res)}
                return res
            return Bif(fn, arity, "%s:%s" % (mod, name))

        def hooked(modname, name, arity, local=False):
            if local or depth[0]:
                return resolve(modname, name, arity, local)
            if self.record:
                if (modname, name, arity) not in rt.bifs and os.path.exists(os.path.join(ref_src, modname + ".erl")):
                    self.modules.add(modname)
                    return recording(modname, name, arity)
            elif modname in self.modules and (modname, name, arity) not in rt.bifs:
                return recorded(modname, name, arity)
            return resolve(modname, name, arity, local)
        rt.resolve = hooked

    def save(self):
        with open(self.path, "w") as f:
            f.write('{"modules": %s,\n "calls": [\n' % json.dumps(sorted(self.modules)))
            f.write(",\n".join(json.dumps(self.table[k], sort_keys=True, separators=(",", ":")) for k in sorted(self.table)))
            f.write("\n]}\n")
