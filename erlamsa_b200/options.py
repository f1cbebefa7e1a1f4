"""Option handling that mirrors the reference's name surface.

* mutator / pattern codes and default priorities: reference src/erlamsa_mutations.erl:1291-1331,
  src/erlamsa_patterns.erl:395-404 (read back from the native library so there is one table);
* the `-m` / `-p` grammar "code=pri,code,..." of erlamsa_cmdparse:string_to_actions/3
  (reference src/erlamsa_cmdparse.erl:233-257): a bare code takes its priority from the default table;
* the option-map keys read by erlamsa_main:fuzzer/1 (reference src/erlamsa_main.erl:127-163).
"""
import re

from . import _native as N


def mutator_codes():
    L = N.lib()
    return [L.eb200_mutator_code(i).decode() for i in range(N.N_MUTATORS)]


def pattern_codes():
    L = N.lib()
    return [L.eb200_pattern_code(i).decode() for i in range(N.N_PATTERNS)]


def default_mutations():
    """erlamsa_mutations:default/1 -> [{Code, Pri}]"""
    L = N.lib()
    return [(L.eb200_mutator_code(i).decode(), L.eb200_mutator_default_pri(i)) for i in range(N.N_MUTATORS)]


def default_patterns():
    """erlamsa_patterns:default/0"""
    L = N.lib()
    return [(L.eb200_pattern_code(i).decode(), L.eb200_pattern_default_pri(i)) for i in range(N.N_PATTERNS)]


def supported_mutations():
    L = N.lib()
    return [c for i, c in enumerate(mutator_codes()) if L.eb200_mutator_supported(i)]


def supported_patterns():
    L = N.lib()
    return [c for i, c in enumerate(pattern_codes()) if L.eb200_pattern_supported(i)]


def string_to_actions(s, what, defaults):
    """erlamsa_cmdparse:string_to_actions/3 (src/erlamsa_cmdparse.erl:232-257): "bd=2,num,sr=3" -> [("sr",3),("num",DefaultPri),("bd",2)].
    A name without "=N" takes its priority from the DEFAULT table (`-m sgm` means sgm=10, not sgm=1); tokens are cut the way
    string:tokens/2 cuts them (empty pieces vanish, "bd=2=3" has three pieces and falls back to the default priority); the list
    comes back reversed, so that -- turned into a map, as make_mutator/2 and make_pattern/1 do -- the FIRST of two entries for
    one name wins. An unknown name or a priority that is not an integer raises, where the reference fails with
    "No such <what>!" / "Invalid <what> list specification!". Extension: the single word "default" keeps the table."""
    if s == "default":
        return list(defaults)
    known = dict(defaults)
    out = []
    for tok in s.split(","):
        if not tok:
            continue
        parts = [x for x in tok.split("=") if x]
        if not parts:
            raise ValueError("Invalid %s list specification!" % what)
        name = parts[0]
        if name not in known:
            raise ValueError("Unknown %s: %s" % (what, name))
        if len(parts) == 2:
            if not re.fullmatch(r"[+-]?[0-9]+", parts[1]):
                raise ValueError("Invalid %s list specification!" % what)
            out.append((name, int(parts[1])))
        else:
            out.append((name, known[name]))
    out.reverse()
    return out


def make_opts(opts=None):
    """Erlang-style option map (python dict with the reference's keys) -> native eb200_opts."""
    opts = dict(opts or {})
    o = N.Opts()
    N.lib().eb200_default_opts(o)
    if "seed" in opts:
        a, b, c = opts["seed"]
        o.seed[0], o.seed[1], o.seed[2] = int(a), int(b), int(c)
    else:
        # the reference falls back to gen_urandom_seed/0 (src/erlamsa_rnd.erl:50-62)
        import os
        r = os.urandom(6)
        o.seed[0], o.seed[1], o.seed[2] = [int.from_bytes(r[i:i + 2], "big") for i in (0, 2, 4)]
    o.blockscale = float(opts.get("blockscale", 1.0))
    for key, codes, field, what in (("mutations", mutator_codes(), o.muta_pri, "mutation"),
                                    ("patterns", pattern_codes(), o.pat_pri, "pattern")):
        if key in opts:
            sel = opts[key]
            if isinstance(sel, str):
                sel = string_to_actions(sel, what, default_mutations() if key == "mutations" else default_patterns())
            sel = dict(sel)
            for name in sel:
                if name not in codes:
                    raise ValueError("Unknown %s: %s" % (what, name))
            for i, c in enumerate(codes):
                field[i] = int(sel[c]) if c in sel else -1
    if "generators" in opts:
        g = dict(opts["generators"])
        o.gen_direct_pri = int(g.get("direct", -1))
        o.gen_random_pri = int(g.get("random", -1))
        o.gen_file_pri = int(g.get("file", -1))
        o.gen_stdin_pri = int(g.get("stdin", -1))
        o.gen_jump_pri = int(g.get("jump", -1))      # takes part in the parent's draw; a run that lands on it needs jump_on_device
        unknown = set(g) - {"direct", "random", "file", "stdin", "jump"}
        if unknown:
            raise ValueError("generator(s) without a device implementation: %s" % ", ".join(sorted(unknown)))
    # 1: run the jump generator when the parent's draw lands on it; 0 (default): the engine refuses such a run (EB200_ERR_UNSUPPORTED)
    o.jump_on_device = 1 if opts.get("jump_on_device") else 0
    if opts.get("case_stream") is not None:       # (worker seed, number of the worker's first case): one worker of `workers` > 1
        (a, b, c), first = opts["case_stream"]
        o.case_stream_seed[0], o.case_stream_seed[1], o.case_stream_seed[2] = int(a), int(b), int(c)
        o.case_stream_first = int(first)
    o.ssrf_host = str(opts.get("ssrf_host", "localhost")).encode()[:63]
    o.ssrf_port = int(opts.get("ssrf_port", 51234))
    o.rng_mode = {"as183": 0, "philox": 1}[opts.get("rng", "as183")]
    o.first_case = int(opts.get("skip", 0)) + 1
    if "first_case" in opts:
        o.first_case = int(opts["first_case"])
    o.max_case_out = int(opts.get("max_case_out", 0))
    o.scratch_bytes = int(opts.get("scratch_bytes", 0))
    if "donor_pool" in opts:      # (device address of the windows, device address of the lengths, count, stride) -- config C5
        pool, lens, n, stride = opts["donor_pool"]
        o.donor_pool, o.donor_len, o.n_donors, o.donor_stride = int(pool), int(lens), int(n), int(stride)
    return o
