"""B200-native hybrid retrieval for Legal-RAG-engine (sm_100a CUDA behind a C ABI).

Layout
  csrc/       hand-written CUDA kernels + the C ABI of include/lrx.h
  _lib.py     ctypes binding (fails loudly when the CUDA library is missing)
  engine.py   host-side mirror of the reference's RetrievalEngine / search
  store.py    on-disk vector store (fp16 matrix, CSR postings, metadata.json)
  bm25_index.py  BM25Okapi statistics + CSR postings builder
  sharding.py multi-GPU: aligned row shards + in-kernel peer exchange of candidate records
  synth.py    seeded synthetic corpora of the benchmark shapes
"""
__version__ = "0.1.0"
