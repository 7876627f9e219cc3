#!/usr/bin/env python3
"""Constant-time audit of the secret-handling kernels, on the SASS that ships (north_star: "secret-scalar paths stay
constant-time per lane: no secret-dependent branches or table indices"; reference discipline: constant_time.h:134-183
masked lookups, goldilocks.c:850-870 comb loop).

What it does
  1. `cuobjdump -sass` of libgoldilocks_b200.so; the listing of every audited kernel (encodings stripped) is written to
     profiles/sass/<kernel>.sass -- the committed SASS the verdicts below refer to.
  2. A forward taint analysis over each kernel's control-flow graph (subroutines called with CALL.REL.NOINC included,
     context-insensitively).  Sources: every load through a kernel-parameter pointer that tools/ct_layout.cpp classes
     `secret` or `out` (scratch of an earlier secret stage), and -- conservatively -- EVERY load from shared or local
     memory (the slot machine's register file lives there).  Loads through `public` pointers (peer points, messages,
     offsets, contexts, fixed tables) and kernel parameters themselves are clean.  Taint flows through every ALU /
     move / shuffle / vote instruction and through the guard predicate of a predicated instruction.
  3. Verdict per kernel.  FAIL on
       * a conditional branch, predicated EXIT/RET or uniform branch whose predicate is tainted,
       * a global, local or constant load/store/atomic whose ADDRESS is tainted (secret table index),
       * a memory instruction executed under a tainted guard predicate.
     Reported but allowed: shared-memory accesses whose address is tainted.  These are the slot machine's handle
     selections (csrc/slots.cuh: a conditional swap picks one of two slot handles per lane instead of moving data).
     Slot s, quad q of lane t lives at ((4s+q)*128 + t)*16 bytes: whatever the secret picks, lane t stays in bank group
     t mod 8 of its own quarter-warp phase, so the selection cannot create a bank conflict -- and shared memory has no
     cache.  The GPU timing test (tests/test_gpu_parity.py::test_secret_paths_time_independent_of_the_scalar) is the
     dynamic check of the same claim.

    python tools/ct_audit.py [--lib path] [--no-write] [--verbose]
Exit status 1 if any kernel fails.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAM_BASE = 0x380            # sm_100: kernel parameters start at c[0x0][0x380]
AUDITED = ["SlotX448", "SlotComb", "SlotCombTable", "SlotX448DerivePk", "SlotEdDerivePk", "SlotEdSignR", "SlotScalarmul", "SlotDoubleScalarmul",
           "SlotDualScalarmul", "SlotDirectScalarmul", "LaneEdSignExpand", "LaneEdSignNonce", "LaneEdSignFinish", "LaneEdSecretScalar", "LaneEdSkToX448"]
# secret-handling kernels of entry points the reference's API does not have (our extensions), reported as their own group,
# one summary line per extension
AUDITED_EXTENSIONS = ["SlotX448Peer", "SlotX448PeerLookup", "SlotDecafPeer"]
EXTENSION_NAMES = {"SlotX448Peer": "X448 peer-set", "SlotX448PeerLookup": "X448 peer-set lookup", "SlotDecafPeer": "decaf peer-set"}

NEGATIVE_CONTROL = "SlotBaseDoubleScalarmul"

NO_DEST = {"STG", "STS", "STL", "ST", "BRA", "BSSY", "BSYNC", "BREAK", "CALL", "EXIT", "RET", "NOP", "BAR", "RED", "WARPSYNC", "MEMBAR", "ERRBAR", "DEPBAR", "YIELD", "BMOV",
           "NANOSLEEP", "CCTL", "UBLKCP", "SYNCS"}
PRED_ONLY_DEST = {"ISETP", "UISETP", "PLOP3", "UPLOP3", "FSETP", "DSETP", "PSETP", "UPSETP"}
KNOWN = NO_DEST | PRED_ONLY_DEST | {"ATOMG", "CS2R", "FLO", "IADD3", "IMAD", "LDC", "LDCU", "LDG", "LDL", "LDS", "LEA", "LOP3", "MOV", "POPC", "PRMT", "S2R", "S2UR", "SEL", "SHF",
                                    "SHFL", "UIADD3", "UIMAD", "ULEA", "UMOV", "VIADD", "VOTEU", "VOTE", "ULOP3", "USHF", "USEL", "IABS", "IMNMX", "VIMNMX", "R2UR", "LD", "UFLO",
                                    "UPOPC", "BREV", "UBREV", "LOP", "ULOP", "I2I", "MATCH", "REDUX", "UVIADD", "UIABS", "UVIMNMX", "P2R", "R2P", "UP2UR", "UR2UP"}


class Ins:
    __slots__ = ("addr", "guard", "gneg", "op", "base", "mods", "operands", "text")


def parse_function(lines):
    out = []
    for line in lines:
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if not m:
            continue
        ins = Ins()
        ins.addr = int(m.group(1), 16)
        text = m.group(2).strip()
        ins.text = text
        g = re.match(r"@(!?U?P\d|!?U?PT)\s+(.*)", text)
        ins.guard, ins.gneg = None, False
        if g:
            ins.guard, ins.gneg, text = g.group(1).lstrip("!"), g.group(1).startswith("!"), g.group(2)
        parts = text.split(None, 1)
        ins.op = parts[0]
        ins.base = ins.op.split(".")[0]
        ins.mods = ins.op.split(".")[1:]
        ins.operands = [o.strip() for o in split_operands(parts[1])] if len(parts) > 1 else []
        out.append(ins)
    return out


def split_operands(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch == "[":
            depth += 1
        elif ch == "]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur)
            cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur)
    return out


REG = re.compile(r"\b(UR\d+|R\d+|UP\d|P\d)\b")
CONST = re.compile(r"c\[0x0\]\[(0x[0-9a-f]+)\]")


def is_pred(o):
    return re.fullmatch(r"!?U?P(\d|T)", o) is not None


def regs_of(o, width):
    """registers named in operand `o`; a general register read as part of a wide operand drags its successors along"""
    out = []
    for m in REG.finditer(o):
        r = m.group(1)
        out.append(r)
        if r[0] == "R" or r.startswith("UR"):
            w = width
            if re.search(re.escape(r) + r"\.64", o):
                w = max(w, 2)
            pre, num = ("UR", int(r[2:])) if r.startswith("UR") else ("R", int(r[1:]))
            for k in range(1, w):
                out.append("%s%d" % (pre, num + k))
    return out


def width_of(ins):
    if "128" in ins.mods:
        return 4
    if "64" in ins.mods or "WIDE" in ins.mods or ins.base == "CS2R" and "32" not in ins.mods:
        return 2
    return 1


def classify(ins):
    """(dest registers incl. predicates, source operand strings)"""
    ops = ins.operands
    if ins.base in NO_DEST:
        return [], ops
    dests, i = [], 0
    while i < len(ops) and is_pred(ops[i]) and not ops[i].startswith("!"):
        dests.append(ops[i]); i += 1
    if ins.base not in PRED_ONLY_DEST and i < len(ops) and re.fullmatch(r"(UR\d+|R\d+|RZ|URZ)", ops[i]):
        d = ops[i]; i += 1
        w = width_of(ins)
        if d not in ("RZ", "URZ"):
            pre, num = ("UR", int(d[2:])) if d.startswith("UR") else ("R", int(d[1:]))
            dests += ["%s%d" % (pre, num + k) for k in range(w)]
        while i < len(ops) and is_pred(ops[i]) and not ops[i].startswith("!") and ins.base in ("IADD3", "UIADD3", "LEA", "ULEA", "IMAD", "VOTEU", "VOTE", "UIMAD", "VIADD", "LOP3", "ULOP3"):
            dests.append(ops[i]); i += 1
    return [d for d in dests if d not in ("PT", "UPT")], ops[i:]


class State:
    """taint and parameter provenance of every register, plus the local-memory frame"""
    __slots__ = ("taint", "prov", "stack", "dyn", "cond")

    def __init__(self):
        self.taint, self.prov, self.stack, self.dyn = set(), {}, {}, (False, frozenset())
        self.cond = {}   # reg -> {(predicate, negated): (taint, prov)}: what the register holds IF that guard held at its last predicated write

    def copy(self):
        s = State()
        s.taint, s.prov, s.stack, s.dyn = set(self.taint), dict(self.prov), dict(self.stack), self.dyn
        s.cond = {r: dict(d) for r, d in self.cond.items()}
        return s

    def join(self, o):
        changed = False
        for r in list(self.cond):
            mine, theirs = self.cond[r], o.cond.get(r, {})
            for g in list(mine):
                if g not in theirs:
                    del mine[g]; changed = True
                else:
                    t, p = mine[g]
                    t2, p2 = theirs[g]
                    if (t2 and not t) or not p2 <= p:
                        mine[g] = (t or t2, p | p2); changed = True
            if not mine:
                del self.cond[r]
        if not o.taint <= self.taint:
            self.taint |= o.taint; changed = True
        for r, p in o.prov.items():
            q = self.prov.get(r, frozenset())
            if not p <= q:
                self.prov[r] = q | p; changed = True
        for k, (t, p) in o.stack.items():
            t0, p0 = self.stack.get(k, (False, frozenset()))
            if (t and not t0) or not p <= p0:
                self.stack[k] = (t0 or t, p0 | p); changed = True
        if (o.dyn[0] and not self.dyn[0]) or not o.dyn[1] <= self.dyn[1]:
            self.dyn = (self.dyn[0] or o.dyn[0], self.dyn[1] | o.dyn[1]); changed = True
        return changed


def audit_kernel(name, functor, ins_list, layout, verbose=False, trace=None):
    fields = layout[functor]["fields"]
    fsize = layout[functor]["size"]

    def param_class(off):
        rel = off - PARAM_BASE
        for f in fields:
            if f["offset"] <= rel < f["offset"] + f["size"]:
                return f["class"], f["name"]
        return ("value", "n/counter") if rel >= fsize else ("value", "pad")

    index = {ins.addr: k for k, ins in enumerate(ins_list)}
    call_targets = sorted({int(i.operands[-1], 16) for i in ins_list if i.base == "CALL"})
    for i in ins_list:
        if i.base not in KNOWN:
            raise SystemExit("ct_audit: unknown opcode %s in %s -- teach tools/ct_audit.py its operand roles" % (i.op, name))

    def sub_of(addr):
        s = None
        for t in call_targets:
            if t <= addr:
                s = t
        return s
    return_sites = {}
    for k, i in enumerate(ins_list):
        if i.base == "CALL":
            return_sites.setdefault(int(i.operands[-1], 16), []).append(k + 1)

    def succ(k):
        i = ins_list[k]
        nxt = [k + 1] if k + 1 < len(ins_list) else []
        if i.base == "BRA":
            tgt = index[int(i.operands[-1], 16)]
            cond = i.guard is not None or (i.op.startswith("BRA.U") and len(i.operands) > 1) or "DIV" in i.mods
            return [tgt] + (nxt if cond else [])
        if i.base == "CALL":
            return [index[int(i.operands[-1], 16)]]
        if i.base == "RET":
            return return_sites.get(sub_of(i.addr), []) + (nxt if i.guard else [])
        if i.base == "EXIT":
            return nxt if i.guard else []
        return nxt

    # what each subroutine may write (registers, predicates, constant-offset stack slots), nested calls included: a value the
    # callee never touches comes back from a call as the CALL SITE left it, not as the join over all call sites
    mods = {t: [set(), set(), False] for t in call_targets}   # regs, stack offsets, writes-dynamic-local
    calls_of = {t: set() for t in call_targets}
    rets_of = {t: [] for t in call_targets}
    for k, i in enumerate(ins_list):
        sub = sub_of(i.addr)
        if sub is None:
            continue
        d, _ = classify(i)
        mods[sub][0].update(d)
        if i.base == "STL":
            aop = next((o for o in i.operands if "[" in o), "")
            m = re.fullmatch(r"\[R1(\+0x[0-9a-f]+)?\]", aop)
            if m:
                base_off = int(m.group(1), 16) if m.group(1) else 0
                mods[sub][1].update(base_off + 4 * b for b in range(width_of(i)))
            else:
                mods[sub][2] = True
        if i.base == "CALL":
            calls_of[sub].add(int(i.operands[-1], 16))
        if i.base == "RET":
            rets_of[sub].append(k)
    changed = True
    while changed:
        changed = False
        for t in call_targets:
            for c in calls_of[t]:
                before = (len(mods[t][0]), len(mods[t][1]), mods[t][2])
                mods[t][0] |= mods[c][0]; mods[t][1] |= mods[c][1]; mods[t][2] = mods[t][2] or mods[c][2]
                if before != (len(mods[t][0]), len(mods[t][1]), mods[t][2]):
                    changed = True

    def merge_return(exit_state, call_state, sub):
        """state after the call: what the callee may have written from its exit state, everything else from the call site"""
        regs, slots, dyn = mods[sub]
        out = call_state.copy()
        for r in regs:
            if r in exit_state.taint:
                out.taint.add(r)
            else:
                out.taint.discard(r)
            if r in exit_state.prov:
                out.prov[r] = exit_state.prov[r]
            else:
                out.prov.pop(r, None)
        for r in list(out.cond):
            if r in regs:
                del out.cond[r]
            else:
                for g in [g for g in out.cond[r] if g[0] in regs]:
                    del out.cond[r][g]
                if not out.cond[r]:
                    del out.cond[r]
        for r in regs:
            if r in exit_state.cond:
                out.cond[r] = dict(exit_state.cond[r])
        for o in slots:
            if o in exit_state.stack:
                out.stack[o] = exit_state.stack[o]
        if dyn:
            out.dyn = exit_state.dyn
        return out

    states = [None] * len(ins_list)
    states[0] = State()
    work = [0]
    findings, info = {}, {"lds_sts_tainted_address": 0, "branches": 0, "memory_ops": 0, "secret_loads": 0, "public_loads": 0}

    def src_taint(st, regs):
        return any(r in st.taint for r in regs)

    def src_prov(st, regs, consts):
        p = frozenset(consts)
        for r in regs:
            p |= st.prov.get(r, frozenset())
        return p

    def transfer(k, st, record):
        i = ins_list[k]
        w = width_of(i)
        dests, srcs = classify(i)
        sregs, consts = [], []
        for pos, o in enumerate(srcs):
            if "[" in o:
                ow = 1                                  # an address: 64-bit pairs carry an explicit .64 suffix (regs_of)
            elif "WIDE" in i.mods:
                ow = 2 if pos == 2 else 1               # a * b + c with a 64-bit addend
            elif i.base in ("STG", "STS", "STL", "ST", "ATOMG", "RED"):
                ow = w                                  # the data operand of a wide store
            else:
                ow = 1
            sregs += regs_of(o, ow)
            consts += [int(c, 16) for c in CONST.findall(o)]
        guard_t = i.guard is not None and i.guard in st.taint
        gkey = (i.guard, i.gneg) if i.guard not in (None, "PT", "UPT") else None

        def rt(r):   # taint of r as this instruction sees it: a value written under the very same guard is the one it reads
            if gkey and gkey in st.cond.get(r, {}):
                return st.cond[r][gkey][0]
            return r in st.taint

        def rp(r):
            if gkey and gkey in st.cond.get(r, {}):
                return st.cond[r][gkey][1]
            return st.prov.get(r, frozenset())
        t = any(rt(r) for r in sregs) or guard_t
        p = frozenset(consts).union(*[rp(r) for r in sregs]) if sregs else frozenset(consts)
        mem = i.base in ("LDG", "STG", "LDL", "STL", "LDS", "STS", "LD", "ST", "ATOMG", "RED", "LDC", "LDCU")
        if mem:
            aop = next((o for o in i.operands if "[" in o), "")
            if i.base in ("LDC", "LDCU"):
                inner = aop[aop.rfind("[") + 1:aop.rfind("]")]
                aregs = regs_of(inner, 1)
            else:
                aregs = regs_of(aop[aop.rfind("["):], 1) if "desc[" in aop else regs_of(aop, 1)
            a_taint = any(rt(r) for r in aregs)
            a_prov = frozenset(int(c, 16) for c in CONST.findall(aop)).union(*[rp(r) for r in aregs]) if aregs else frozenset(int(c, 16) for c in CONST.findall(aop))
            if record:
                info["memory_ops"] += 1
                if guard_t:
                    findings[i.addr] = "memory instruction under a tainted guard predicate: " + i.text
                if a_taint:
                    if i.base in ("LDS", "STS"):
                        info["lds_sts_tainted_address"] += 1
                    else:
                        findings[i.addr] = "tainted ADDRESS (secret-dependent index): " + i.text
            if i.base in ("LDC", "LDCU"):
                m = CONST.search(aop)
                t, p = guard_t or a_taint, (frozenset([int(m.group(1), 16)]) if m else frozenset())
            elif i.base in ("LDS",):
                t, p = True, frozenset()
            elif i.base == "LDL":
                m = re.fullmatch(r"\[R1(\+0x[0-9a-f]+)?\]", aop)
                if m:
                    base_off = int(m.group(1), 16) if m.group(1) else 0
                    t, p = st.dyn
                    for b in range(0, 4 * w, 4):
                        tt, pp = st.stack.get(base_off + b, (False, frozenset()))
                        t, p = t or tt, p | pp
                    t = t or guard_t
                else:
                    t, p = True, frozenset()
            elif i.base in ("LDG", "LD", "ATOMG"):
                classes = {param_class(c)[0] for c in a_prov}
                clean = bool(classes) and classes <= {"public", "value"} and not a_taint
                t, p = (not clean) or guard_t, frozenset()
                if record:
                    info["public_loads" if clean else "secret_loads"] += 1
            elif i.base == "STL":
                data = [o for o in srcs if "[" not in o]
                dregs = []
                for o in data:
                    dregs += regs_of(o, 1)
                m = re.fullmatch(r"\[R1(\+0x[0-9a-f]+)?\]", aop)
                if m and dregs:
                    base_off = int(m.group(1), 16) if m.group(1) else 0
                    num = int(dregs[0][1:]) if dregs[0].startswith("R") and dregs[0] != "RZ" else None
                    for b in range(w):
                        r = "R%d" % (num + b) if num is not None else None
                        st.stack[base_off + 4 * b] = ((r in st.taint) or guard_t, st.prov.get(r, frozenset())) if r else (guard_t, frozenset())
                else:
                    tt = any(r in st.taint for r in dregs) or guard_t
                    pp = frozenset().union(*[st.prov.get(r, frozenset()) for r in dregs]) if dregs else frozenset()
                    st.dyn = (st.dyn[0] or tt, st.dyn[1] | pp)
        elif i.base in ("S2R", "S2UR", "CS2R"):
            t, p = guard_t, frozenset()
        # BREAK: a predicated exit from a convergence region (BSSY ... BSYNC) -- control flow like a branch
        if record and (i.base in ("BRA", "BREAK", "EXIT", "RET") or i.base == "CALL"):
            preds = [o.lstrip("!") for o in i.operands if is_pred(o)] + ([i.guard] if i.guard else [])
            preds = [q for q in preds if q not in ("PT", "UPT")]
            if preds:
                info["branches"] += 1
            if any(q in st.taint for q in preds):
                findings[i.addr] = "control flow on a tainted predicate: " + i.text
        if record and i.base == "RET" and any(r in st.taint for r in regs_of(i.operands[0], 2)):
            findings[i.addr] = "indirect return through a tainted register: " + i.text
        for d in dests:
            if d[0] == "P" or d.startswith("UP"):          # a rewritten predicate invalidates every record made under it
                for r in list(st.cond):
                    for g in [g for g in st.cond[r] if g[0] == d]:
                        del st.cond[r][g]
                    if not st.cond[r]:
                        del st.cond[r]
            if gkey is None:
                st.cond.pop(d, None)
                if t:
                    st.taint.add(d)
                else:
                    st.taint.discard(d)
                if p:
                    st.prov[d] = p
                else:
                    st.prov.pop(d, None)
                continue
            rec = st.cond.setdefault(d, {})
            rec[gkey] = (t, p)
            other = rec.get((gkey[0], not gkey[1]))
            if other is not None:                          # written under P and under !P: fully defined by the two
                tt, pp = t or other[0], p | other[1]
                if tt:
                    st.taint.add(d)
                else:
                    st.taint.discard(d)
                if pp:
                    st.prov[d] = pp
                else:
                    st.prov.pop(d, None)
            else:
                if t:
                    st.taint.add(d)
                if p:
                    st.prov[d] = st.prov.get(d, frozenset()) | p
        return st

    rounds = 0
    while work:
        k = work.pop()
        rounds += 1
        out = transfer(k, states[k].copy(), False)
        ik = ins_list[k]
        if ik.base == "CALL":                      # the callee's returns have to be re-merged with this call site's new state
            work.extend(r for r in rets_of[int(ik.operands[-1], 16)] if states[r] is not None)
        for s in succ(k):
            o = out
            if ik.base == "RET" and s > 0 and ins_list[s - 1].base == "CALL" and not (ik.guard and s == k + 1):
                if states[s - 1] is None:
                    continue
                o = merge_return(out, states[s - 1], sub_of(ik.addr))
            if states[s] is None:
                states[s] = o.copy()
                work.append(s)
            elif states[s].join(o):
                work.append(s)
    for k in range(len(ins_list)):
        if states[k] is not None:
            if trace is not None and ins_list[k].addr in trace:
                st = states[k]
                regs = sorted(set(REG.findall(ins_list[k].text)))
                print("  trace %04x  %s" % (ins_list[k].addr, ins_list[k].text))
                for r in regs:
                    print("        %-5s taint=%s prov=%s cond=%s" % (r, r in st.taint, sorted(hex(x) for x in st.prov.get(r, [])), st.cond.get(r)))
                print("        stack tainted: %s  dyn=%s" % (sorted(hex(o) for o, (t, _) in st.stack.items() if t), st.dyn[0]))
            transfer(k, states[k].copy(), True)
    unreachable = sum(1 for s in states if s is None)
    return {"kernel": name, "instructions": len(ins_list), "unreachable": unreachable, "subroutines": len(call_targets),
            "conditional_control_flow_checked": info["branches"], "memory_instructions_checked": info["memory_ops"],
            "loads_through_secret_or_scratch_pointers": info["secret_loads"], "loads_through_public_pointers": info["public_loads"],
            "shared_memory_handle_selected_accesses": info["lds_sts_tainted_address"],
            "violations": [{"addr": "0x%04x" % a, "what": w} for a, w in sorted(findings.items())], "verdict": "PASS" if not findings else "FAIL"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "libgoldilocks_b200", "libgoldilocks_b200.so"))
    ap.add_argument("--no-write", action="store_true", help="do not rewrite profiles/sass and profiles/ct_audit.json")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--only", default=None, help="comma-separated functor names")
    ap.add_argument("--trace", default=None, help="comma-separated hex addresses whose entry state is printed (use with --only)")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "ct_layout")
        subprocess.run(["g++", "-std=c++17", "-O0", "-w", "-o", exe, os.path.join(ROOT, "tools", "ct_layout.cpp")], check=True)
        layout = json.loads(subprocess.run([exe], capture_output=True, text=True, check=True).stdout)
    sass = subprocess.run(["cuobjdump", "-sass", args.lib], capture_output=True, text=True, check=True).stdout.splitlines()
    funcs, cur = {}, None
    for line in sass:
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur:
            funcs[cur].append(line)
    results = []
    outdir = os.path.join(ROOT, "profiles", "sass")
    if not args.no_write:
        os.makedirs(outdir, exist_ok=True)
    trace = {int(a, 16) for a in args.trace.split(",")} if args.trace else None
    for functor in (args.only.split(",") if args.only else AUDITED + AUDITED_EXTENSIONS):
        mangled = [f for f in funcs if re.search(r"I\d+%sE" % functor, f)]
        if len(mangled) != 1:
            raise SystemExit("ct_audit: expected one kernel for %s, found %s" % (functor, mangled))
        ins = parse_function(funcs[mangled[0]])
        if not args.no_write:
            with open(os.path.join(outdir, functor + ".sass"), "w") as f:
                f.write("// %s  (cuobjdump -sass of libgoldilocks_b200.so, encodings stripped; tools/ct_audit.py)\n" % mangled[0])
                for i in ins:
                    f.write("/*%04x*/  %s ;\n" % (i.addr, i.text))
        r = audit_kernel(mangled[0], functor, ins, layout, args.verbose, trace)
        r["functor"] = functor
        results.append(r)
        print("%-22s %-4s  %5d instr, %3d conditional branches, %4d memory ops (%d secret / %d public loads), %d handle-selected LDS/STS%s"
              % (functor, r["verdict"], r["instructions"], r["conditional_control_flow_checked"], r["memory_instructions_checked"],
                 r["loads_through_secret_or_scratch_pointers"], r["loads_through_public_pointers"], r["shared_memory_handle_selected_accesses"],
                 "" if not r["violations"] else "  <-- %d violations" % len(r["violations"])))
        if r["violations"] and (args.verbose or True):
            for v in r["violations"][:12]:
                print("      %s  %s" % (v["addr"], v["what"]))
    # negative control: a kernel that IS variable-time in its scalars (goldilocks_448_base_double_scalarmul_non_secret indexes
    # its tables with scalar digits, as the reference's wNAF does) must be caught when those scalars are labelled secret
    control = None
    if not args.only:
        mangled = [f for f in funcs if re.search(r"I\d+%sE" % NEGATIVE_CONTROL, f)]
        r = audit_kernel(mangled[0], NEGATIVE_CONTROL, parse_function(funcs[mangled[0]]), layout)
        kinds = sorted({v["what"].split(":")[0] for v in r["violations"]})
        print("%-22s %-4s  negative control (public scalars labelled secret): %d violations %s" % (NEGATIVE_CONTROL, r["verdict"], len(r["violations"]), kinds))
        control = {"functor": NEGATIVE_CONTROL, "verdict": r["verdict"], "violations": len(r["violations"]), "kinds": kinds}
        if r["verdict"] != "FAIL" or not any("ADDRESS" in k for k in kinds):
            print("FAIL: the negative control was not caught -- the audit is not looking")
            return 1
    if not args.no_write:
        with open(os.path.join(ROOT, "profiles", "ct_audit.json"), "w") as f:
            json.dump({"param_base": PARAM_BASE, "kernels": results, "negative_control": control}, f, indent=1)
    bad = [r["functor"] for r in results if r["verdict"] != "PASS"]
    if bad:
        print("FAIL: " + ", ".join(bad))
        return 1
    groups = [("reference API", [r for r in results if r["functor"] not in AUDITED_EXTENSIONS])]
    groups += [("%s extensions" % EXTENSION_NAMES[f], [r for r in results if r["functor"] == f]) for f in AUDITED_EXTENSIONS]
    for label, group in groups:
        if group:
            print("%s: all %d secret-handling kernels PASS" % (label, len(group)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
