// TEST INFRASTRUCTURE ONLY — pass 1 of the single-stream route (emu_stream.cpp: the block finder,
// the counting jobs, the chain, the writing jobs, on 32 host threads) stopped before pass 2, in a
// library of its own (libemu_route*.so), with the chain of block jobs chosen by the caller:
// chain_kernel (the sequential walk) or a function given by address, such as emu_block.cpp's
// emu_chain_parallel_args (chain_parallel_kernel on a block of host threads).  What it leaves — the
// in-place token layout and the match-head bitmap — is the input of pass 2 (emu_block.cpp:
// emu_jump_resolve).
#include "emu_stream.cpp"

static void (*emu_chain_fn)(const sfb::FindArgs*) = nullptr;
extern "C" void emu_set_chain(void (*fn)(const sfb::FindArgs*)) { emu_chain_fn = fn; }

// One stream into dst_base + dst_off (dst_base 128-byte aligned), match heads into match_bits.
// n_cand < 0: the candidate block starts are the finder's (as the library runs the route), else
// cand[0 .. n_cand) (true, wrong and duplicate starts alike).  The steps are emu_huff_stream_jobs'
// with the chain from emu_set_chain.  stats[0] = jobs on the chain, stats[1] = tail job.
extern "C" void emu_stream_pass1(const uint8_t* src, uint64_t src_len, uint8_t* dst_base, uint64_t dst_off,
                                 uint64_t dst_cap, uint32_t* match_bits, uint8_t* status, uint64_t* written,
                                 const uint64_t* cand, int64_t n_cand, uint32_t* stats)
{
  std::vector<uint8_t> sbuf(src_len + 64, 0xEE);
  if (src_len) std::memcpy(sbuf.data() + 16, src, src_len);
  const uint8_t* const s = sbuf.data() + 16;
  std::vector<uint64_t> found;
  if (n_cand < 0) {
    found.resize(8 * src_len / 64 + 64);
    n_cand = emu_find_blocks(s, src_len, found.data(), static_cast<uint32_t>(found.size()));
    cand = found.data();
  }
  const uint32_t nc = static_cast<uint32_t>(n_cand);
  EmuWarp warp;
  emu_warp = &warp;
  std::vector<uint16_t> smem(StreamCfg::SMEM_BYTES / 2 + 64, 0xDEAD);
  std::vector<uint32_t> lens(sfb::SCRATCH_WORDS * 32, 0xDEADBEEFu);
  emu_stream_smem = smem.data();
  const uint64_t zero = 0;
  uint32_t tab_size = 64;
  while (tab_size < 2 * (nc + 1)) tab_size *= 2;
  std::vector<uint32_t> job_tab(tab_size, 0u);
  std::vector<sfb::BlockJob> jobs(nc + 1);
  for (uint32_t k = 0; k <= nc; ++k) {
    sfb::BlockJob jb{};
    jb.start_bit = k ? cand[k - 1] : 0;
    jb.end_bit = jb.start_bit;
    jb.base = sfb::JOB_NONE;
    jb.flags = sfb::JOB_ENDS;
    jobs[k] = jb;
    if (k) {
      uint32_t slot = sfb::job_slot(jb.start_bit, tab_size - 1);
      while (job_tab[slot]) slot = (slot + 1) & (tab_size - 1);
      job_tab[slot] = k;
    }
  }
  uint32_t job_count = nc + 1, tail_job = 0, rec_count = 0;
  std::vector<sfb::WinRec> recs(emu_rec_cap + 1);
  sfb::StreamArgs a{};
  a.src_base = s;
  a.src_off = &zero;
  a.src_len = &src_len;
  a.dst_base = dst_base;
  a.dst_delta = 0;
  a.dst_off = &dst_off;
  a.dst_cap = &dst_cap;
  a.status = status;
  a.written = written;
  a.list = nullptr;
  a.idx_base = 0;
  a.n = 1;
  a.lens_scratch = lens.data();
  a.match_bits = match_bits;
  a.jobs = jobs.data();
  a.job_count = &job_count;
  a.job_cap = nc + 1;
  a.job_tab = job_tab.data();
  a.tab_mask = tab_size - 1;
  a.tail_job = &tail_job;
  a.recs = recs.data();
  a.rec_count = &rec_count;
  a.rec_cap = emu_rec_cap;
  unsigned long long counter = 0;
  a.stream_counter = &counter;
  a.mode = 1;
  run_warp(a);
  sfb::FindArgs f{};
  f.idx = 0;
  f.jobs = jobs.data();
  f.job_count = &job_count;
  f.job_cap = nc + 1;
  f.tail_job = &tail_job;
  f.dst_cap = &dst_cap;
  threadIdx.x = 0;
  blockIdx.x = 0;
  if (emu_chain_fn) emu_chain_fn(&f);
  else sfb::chain_kernel(f);
  counter = 0;
  a.mode = 2;
  run_warp(a);
  if (stats) {
    uint32_t on = 0;
    for (auto& jb : jobs) on += jb.base != sfb::JOB_NONE;
    stats[0] = on;
    stats[1] = tail_job;
  }
  emu_warp = nullptr;
  emu_stream_smem = nullptr;
}
