#!/usr/bin/env python3
"""CLI of the B200 chunk path: `compress` / `decompress` with the flags the reference documents
(README.md:75-102: --chunk-size, --methods, --disable-methods, --show-progress).  `analyze` and
`gui` are out of scope (plotting / UI)."""
import argparse
import json
import os
import sys
import time

METHOD_TOKENS = {"rle": 1, "dictionary": 2, "dict": 2, "huffman": 3, "delta": 4, "deflate": 5, "bzip2": 6, "lzma": 7,
                 "zstandard": 8, "zstd": 8, "lz4": 9, "brotli": 10, "lzham": 11, "none": 255, "raw": 255}
METHOD_LABELS = {1: "Run-Length Encoding (RLE)", 2: "Dictionary-Based", 3: "Huffman Coding", 4: "Delta Encoding",
                 5: "DEFLATE", 6: "BZIP2", 7: "LZMA", 255: "No Compression"}


def parse_methods(text):
    ids = []
    for tok in (text or "").split(","):
        tok = tok.strip().lower()
        if not tok:
            continue
        if tok.isdigit():
            ids.append(int(tok))
        elif tok in METHOD_TOKENS:
            ids.append(METHOD_TOKENS[tok])
        else:
            raise ValueError("unknown compression method %r" % tok)
    return ids


def _format_file_size(size_bytes):
    """compression_analyzer.py:857-876"""
    if size_bytes == 0:
        return "0 B"
    names = ["B", "KB", "MB", "GB", "TB"]
    i = 0
    while size_bytes >= 1024 and i < len(names) - 1:
        size_bytes /= 1024.0
        i += 1
    return f"{size_bytes:.1f} {names[i]}"


def _append_history(input_path, stats, results_dir="compression_results"):
    """the record the reference appends (main.py:184-194 -> CompressionAnalyzer.load_results / add_result /
    save_results, compression_analyzer.py:30-72, 74-138), json only: the history is loaded keeping the most
    recent record per file name (in first-occurrence order), a record with the same file name is replaced in
    place, a new one is appended"""
    os.makedirs(results_dir, exist_ok=True)
    path = os.path.join(results_dir, "compression_history.json")
    results = []
    if os.path.exists(path):
        try:
            with open(path) as f:
                loaded = json.load(f)
            latest = {}
            for r in loaded:  # (:95-101)
                name = r.get("filename", "unknown")
                if name not in latest or r.get("timestamp", 0) > latest[name].get("timestamp", 0):
                    latest[name] = r
            results = list(latest.values())
        except Exception as e:  # noqa: BLE001 (main.py:189-192)
            print(f"Error loading results: {e}")
    base = os.path.basename(input_path)
    rec = dict(stats)
    rec["chunk_stats"] = dict(stats["chunk_stats"])
    # (json.dump turns the reference's int method ids into strings as well)
    rec["chunk_stats"]["method_usage"] = {str(k): v for k, v in stats["chunk_stats"].get("method_usage", {}).items()}
    rec.update(filename=base, extension=os.path.splitext(base)[1].lower() or "unknown",
               filename_no_ext=os.path.splitext(base)[0], timestamp=time.time(),
               size_label=_format_file_size(stats.get("original_size", 0)))
    for i, r in enumerate(results):
        if r.get("filename") == base:
            if rec["timestamp"] > r.get("timestamp", 0):
                print(f"Replacing previous result for '{base}'")
                results[i] = rec
            break
    else:
        results.append(rec)
    with open(path, "w") as f:
        json.dump(results, f, indent=2)
    return path


def compress_file(args):
    from adaptive_compression_b200 import AdaptiveCompressor
    print(f"Compressing {args.input} to {args.output}...")
    try:
        methods = parse_methods(args.methods) if args.methods else None
        disabled = parse_methods(args.disable_methods) if args.disable_methods else None
        c = AdaptiveCompressor(chunk_size=args.chunk_size, methods=methods, disable_methods=disabled,
                               per_chunk_raw=args.per_chunk_raw, use_marker_search=args.marker_search)
        stats = c.compress(args.input, args.output)
        print("\nCompression Statistics:")
        print(f"  Original size: {stats['original_size']} bytes")
        print(f"  Compressed size: {stats['compressed_size']} bytes")
        print(f"  Compression ratio: {stats['ratio']:.4f}")
        print(f"  Space saving: {stats['percent_reduction']:.2f}%")
        print(f"  Elapsed time: {stats['elapsed_time']:.4f} seconds")
        print(f"  Throughput: {stats['throughput_mb_per_sec']:.2f} MB/s")
        print("\nChunk Statistics:")
        print(f"  Total chunks: {stats['chunk_stats']['total_chunks']}")
        for mid, count in stats["chunk_stats"]["method_usage"].items():
            if count > 0:
                print(f"    {METHOD_LABELS.get(int(mid), 'Method %s' % mid)}: {count} chunks")
        if not args.no_history:
            _append_history(args.input, stats)
        print("\nCompression completed successfully.")
        return stats
    except Exception as e:  # noqa: BLE001 - the reference prints and exits 1 (main.py:197-199)
        print(f"Error during compression: {e}")
        sys.exit(1)


def decompress_file(args):
    from adaptive_compression_b200 import AdaptiveCompressor
    print(f"Decompressing {args.input} to {args.output}...")
    try:
        methods = parse_methods(args.methods) if args.methods else None
        stats = AdaptiveCompressor(methods=methods).decompress(args.input, args.output)
        print("\nDecompression Statistics:")
        print(f"  Compressed size: {stats['compressed_size']} bytes")
        print(f"  Decompressed size: {stats['decompressed_size']} bytes")
        print(f"  Elapsed time: {stats['elapsed_time']:.4f} seconds")
        print(f"  Throughput: {stats['throughput_mb_per_sec']:.2f} MB/s")
        print("\nDecompression completed successfully.")
        return stats
    except Exception as e:  # noqa: BLE001 (main.py:214-216)
        print(f"Error during decompression: {e}")
        sys.exit(1)


def parse_chunk_size(text):
    """--chunk-size N | dynamic | N1,N2,..."""
    t = text.strip().lower()
    if t in ("dynamic", "auto", "default"):
        from adaptive_compression_b200.adaptive_compressor import REFERENCE_CANDIDATES
        return list(REFERENCE_CANDIDATES)
    if "," in t:
        return [int(x) for x in t.split(",") if x.strip()]
    return int(t)


def build_parser():
    p = argparse.ArgumentParser(description="Adaptive Marker-Based Compression (B200 chunk path)")
    sub = p.add_subparsers(dest="command", help="Command to execute")
    c = sub.add_parser("compress", help="Compress a file")
    c.add_argument("input")
    c.add_argument("output")
    c.add_argument("--chunk-size", type=parse_chunk_size, default="dynamic",
                   help="'dynamic' (default) = the reference's candidate list 131072..1024 (adaptive_compressor.py:61-62: "
                        "what the reference's own CLI always does); N = one chunk size, the fast fixed grid (4096 in the "
                        "benchmarked configurations); or a comma-separated candidate list")
    c.add_argument("--methods", default=None, help="Comma-separated list of compression methods to use")
    c.add_argument("--disable-methods", default=None, help="Comma-separated list of compression methods to disable")
    c.add_argument("--show-progress", action="store_true", help="accepted for compatibility; the GPU path has no per-chunk progress")
    c.add_argument("--per-chunk-raw", action="store_true", help="extension: a chunk without a winner is its own raw package")
    c.add_argument("--marker-search", action="store_true", help="extension: put the found marker in the header")
    c.add_argument("--no-history", action="store_true", help="do not append to compression_results/compression_history.json")
    d = sub.add_parser("decompress", help="Decompress a file")
    d.add_argument("input")
    d.add_argument("output")
    d.add_argument("--show-progress", action="store_true")
    d.add_argument("--methods", default=None,
                   help="Comma-separated list of the methods the file's packages may use (same tokens as compress; "
                        "default: the native methods 1-4); e.g. rle,dictionary,huffman,delta,deflate,bzip2,lzma")
    sub.add_parser("analyze", help="(out of scope in this build: plotting)")
    sub.add_parser("gui", help="(out of scope in this build: UI)")
    return p


def main(argv=None):
    p = build_parser()
    args = p.parse_args(argv)
    if args.command == "compress":
        return compress_file(args)
    if args.command == "decompress":
        return decompress_file(args)
    if args.command in ("analyze", "gui"):
        print("`%s` is not part of the B200 chunk path (see DESIGN.md, out of scope)." % args.command)
        sys.exit(1)
    p.print_help()


if __name__ == "__main__":
    main()
