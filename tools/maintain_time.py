"""Times bm25x_index_maintain (bm25::maintain on the device) against the path a caller has without it: bm25x_index_create
of the maintained corpus from host memory (the host-side re-sort that path would also need is not included).

Workloads: the C3 shape (10 M docs, vocab 100 k, 128 terms per doc, uniform) and the C4 shape (the same with Zipf(1)
tokens).  1 % of the sealed documents are deleted, and 100 k growing documents (same shape, ordinals up to 1 % past the
sealed vocabulary) are added with every 5th one deleted.  Per workload the JSON gives the call's total and device time,
the device time of the compaction pass alone (k_mt_compact, from a torch.profiler run of its own), its algorithmic bytes
and its rate as a fraction of a device-to-device copy timed in the same run, the PCIe bytes, the create() time, and the
card's name and power limit.  The maintained handle must be byte-identical to the created one, so a fast and wrong
maintain cannot pass.

    python tools/maintain_time.py OUT_DIR [--workloads c3,c4] [--docs N] [--growing G]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import _pkg  # noqa: E402

WORKLOADS = {"c3": dict(seed=0xB25C0DE0 + 3, zipf=0.0), "c4": dict(seed=0xB25C0DE0 + 4, zipf=1.0)}
NONE = 0xFFFFFFFF


def card(device):
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?", "?"])[:2]
    return {"gpu": name, "power_limit": power}


def growing_docs(m, seed, n, vocab, doclen, zipf):
    """Growing documents as a term-major corpus (the generator's form) and as the doc-major chain maintain takes."""
    gc = m.synth_corpus(seed, n, vocab, doclen, doclen, zipf)
    df = np.diff(gc.post_off.astype(np.int64))
    term = np.repeat(np.arange(gc.n_terms, dtype=np.uint32), df)
    order = np.lexsort((term, gc.post_doc))
    off = np.concatenate([[0], np.cumsum(np.bincount(gc.post_doc, minlength=n))]).astype(np.uint64)
    return gc, off, term[order].copy(), gc.post_tf[order].copy()


def expected_corpus(c, sdel, gc, gdel):
    """The maintained corpus (keyless) without a global sort: every sealed list is filtered and relabelled in place, the
    growing postings follow it (tests/maintain_oracle.py states the same on small inputs)."""
    N, T, G = c.n_docs, c.n_terms, gc.n_docs
    alive, galive = ~sdel.astype(bool), ~gdel.astype(bool)
    ns = int(alive.sum())
    relabel = np.full(N, NONE, np.uint32)
    relabel[alive] = np.arange(ns, dtype=np.uint32)
    grow_new = np.full(G, NONE, np.uint32)
    grow_new[galive] = ns + np.arange(int(galive.sum()), dtype=np.uint32)
    s_len = np.bincount(c.post_doc, minlength=N)[alive]                    # distinct tokens (maintain.rs:337,356-360)
    keep = alive[c.post_doc]
    dead = np.nonzero(~keep)[0]
    s_cnt = np.diff(c.post_off.astype(np.int64)) - np.bincount(
        np.searchsorted(c.post_off, dead, side="right") - 1, minlength=T)
    s_doc = relabel[c.post_doc[keep]]
    s_tf = c.post_tf[keep]
    del keep, dead
    gkeep = galive[gc.post_doc]
    g_term = np.repeat(np.arange(gc.n_terms, dtype=np.int64), np.diff(gc.post_off.astype(np.int64)))[gkeep]
    g_doc, g_tf = grow_new[gc.post_doc[gkeep]], gc.post_tf[gkeep]
    g_len = np.minimum(np.bincount(gc.post_doc, weights=gc.post_tf.astype(np.float64), minlength=G)[galive], NONE)
    T_new = max(T, gc.n_terms if len(g_term) == 0 else int(g_term.max()) + 1)
    s_cnt = np.concatenate([s_cnt, np.zeros(T_new - T, np.int64)])
    g_cnt = np.bincount(g_term, minlength=T_new)
    off = np.concatenate([[0], np.cumsum(s_cnt + g_cnt)]).astype(np.uint64)
    s_off = np.concatenate([[0], np.cumsum(s_cnt)])
    g_off = np.concatenate([[0], np.cumsum(g_cnt)])
    doc = np.empty(int(off[-1]), np.uint32)
    tf = np.empty(int(off[-1]), np.uint32)
    for t in range(T_new):
        a, sa, sb, ga, gb = int(off[t]), int(s_off[t]), int(s_off[t + 1]), int(g_off[t]), int(g_off[t + 1])
        doc[a:a + sb - sa], tf[a:a + sb - sa] = s_doc[sa:sb], s_tf[sa:sb]
        doc[a + sb - sa:a + sb - sa + gb - ga], tf[a + sb - sa:a + sb - sa + gb - ga] = g_doc[ga:gb], g_tf[ga:gb]
    doc_len = np.concatenate([s_len, g_len]).astype(np.uint32)
    return dict(n_docs=len(doc_len), doc_len=doc_len, n_terms=T_new, post_off=off, post_doc=doc, post_tf=tf)


def device_equal(torch, a, b):
    la, lb = a.layout(), b.layout()
    if list(la.bytes) != list(lb.bytes):
        return False

    def view(lay, i):
        n = int(lay.bytes[i])
        obj = type("DevArray", (), {"__cuda_array_interface__": {
            "shape": (n,), "typestr": "|u1", "data": (int(lay.dev_ptr[i]), False), "version": 3}})()
        return torch.as_tensor(obj, device=f"cuda:{lay.device}")
    return all(int(la.bytes[i]) == 0 or torch.equal(view(la, i), view(lb, i)) for i in range(len(la.bytes)))


def copy_rate(torch, device, nbytes, reps=5):
    """Device-to-device copy, bytes read + written per second."""
    src = torch.empty(nbytes, dtype=torch.uint8, device=device)
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del src, dst
    torch.cuda.empty_cache()
    return 2 * nbytes / (ms * 1e-3), ms


def run(m, torch, name, a, out_dir):
    wl = WORKLOADS[name]
    t0 = time.time()
    c = m.synth_corpus(wl["seed"], a.docs, a.vocab, a.doclen, a.doclen, wl["zipf"])
    rng = np.random.default_rng(wl["seed"])
    sdel = (rng.random(c.n_docs) < 0.01).astype(np.uint8)
    gc, g_off, g_term, g_tf = growing_docs(m, wl["seed"] + 1, a.growing, a.vocab + a.vocab // 100, a.doclen, wl["zipf"])
    gdel = (np.arange(a.growing) % 5 == 2).astype(np.uint8)
    ix = m.Index.from_corpus(c, device=a.device)
    gen_s = time.time() - t0
    kw = dict(deleted=sdel, elem_off=g_off, elem_term=g_term, elem_tf=g_tf, growing_deleted=gdel)

    new, relabel, st = ix.maintain(**kw)                                   # timed run (kernels are loaded by warm_up)
    res = {"workload": name, "docs": c.n_docs, "vocab": a.vocab, "postings_sealed": int(c.n_postings),
           "growing_docs": a.growing, "growing_elements": int(len(g_tf)), "sealed_deleted": int(sdel.sum()),
           "growing_deleted": int(gdel.sum()), "setup_s": round(gen_s, 1),
           "total_ms": st.total_ms, "device_ms": st.device_ms, "h2d_bytes": st.h2d_bytes, "d2h_bytes": st.d2h_bytes,
           "postings_in": st.postings_in, "postings_out": st.postings_out,
           "pcie_bytes_per_posting_in": (st.h2d_bytes + st.d2h_bytes) / st.postings_in}
    lay_old = ix.layout()
    n_pad = int(lay_old.n_postings_padded)
    new.close()

    # the compaction pass alone: a profiled run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        new, _, _ = ix.maintain(**kw)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        if "k_mt_" in ev.key:
            dev_us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            kern[ev.key] = round(dev_us / 1000.0, 3)
    res["kernels_ms"] = kern
    compact_ms = sum(v for k, v in kern.items() if "k_mt_compact" in k)
    # algorithmic bytes of k_mt_compact: every padded slot of the old lists read (8 B), every sealed survivor written
    # (8 B); the relabel / fieldnorm / delete-mark lookups (9 B per posting) hit tables that sit in L2
    g_written = int(np.count_nonzero(gdel[np.repeat(np.arange(a.growing), np.diff(g_off.astype(np.int64)))] == 0))
    sealed_out = int(st.postings_out) - g_written
    bytes_compact = 8 * n_pad + 8 * sealed_out
    rate, copy_ms = copy_rate(torch, f"cuda:{a.device}", 4 << 30)
    res.update({"compact_ms": compact_ms, "compact_bytes_algo": bytes_compact,
                "compact_bytes_per_s": bytes_compact / (compact_ms * 1e-3) if compact_ms else None,
                "copy_bytes_per_s": rate, "copy_ms_4GiB": copy_ms,
                "compact_fraction_of_copy": (bytes_compact / (compact_ms * 1e-3)) / rate if compact_ms else None})
    prof.export_chrome_trace(os.path.join(out_dir, f"maintain_{name}.pt.trace.json"))

    # the path without maintain: create() of the maintained corpus from host memory
    exp = expected_corpus(c, sdel, gc, gdel)
    del c
    t1 = time.perf_counter()
    ref = m.Index(exp["n_docs"], exp["doc_len"], exp["n_terms"], exp["post_off"], exp["post_doc"], exp["post_tf"],
                  device=a.device, payload=_payload(sdel, gdel))
    res["create_ms"] = (time.perf_counter() - t1) * 1e3
    res["byte_identical"] = bool(device_equal(torch, new, ref))
    res["speedup_vs_create"] = res["create_ms"] / res["total_ms"]
    for x in (ref, new, ix):
        x.close()
    return res


def _payload(sdel, gdel):
    """Payloads of the maintained documents: the sealed ones' synthetic ctids, then the growing ordinals' ones."""
    def ctid(i):
        blk = i // 291
        return np.stack([blk >> 16, blk & 0xFFFF, i % 291 + 1], axis=-1).astype(np.uint16)
    return np.concatenate([ctid(np.nonzero(sdel == 0)[0]), ctid(np.nonzero(gdel == 0)[0])])


def warm_up(m, device):
    c = m.synth_corpus(1, 2000, 100, 8)
    ix = m.Index.from_corpus(c, device=device)
    new, _, _ = ix.maintain(deleted=(np.arange(2000) % 3 == 0).astype(np.uint8))
    new.close()
    ix.close()


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("out_dir")
    p.add_argument("--workloads", default="c3,c4")
    p.add_argument("--docs", type=int, default=10_000_000)
    p.add_argument("--vocab", type=int, default=100_000)
    p.add_argument("--doclen", type=int, default=128)
    p.add_argument("--growing", type=int, default=100_000)
    p.add_argument("--device", type=int, default=0)
    a = p.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    import torch
    m = _pkg.load()
    m.load_library()
    if m.device_count() < 1:
        raise SystemExit("no CUDA device: maintain runs on the GPU only")
    torch.cuda.set_device(a.device)
    warm_up(m, a.device)
    out = {"card": card(a.device), "results": []}
    for name in a.workloads.split(","):
        r = run(m, torch, name, a, a.out_dir)
        print(json.dumps(r), flush=True)
        out["results"].append(r)
    with open(os.path.join(a.out_dir, "maintain_time.json"), "w") as f:
        json.dump(out, f, indent=1)
    if not all(r["byte_identical"] for r in out["results"]):
        raise SystemExit("maintained index differs from create() of the maintained corpus")


if __name__ == "__main__":
    main()
