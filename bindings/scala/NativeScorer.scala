// NativeScorer.scala — JNA binding of libmrscore.so (include/mrscore.h) plus the glue that turns the reference's string maps
// into the int-id CSR the library takes.  Not compiled in this repository's image (no JDK); see INTEGRATION.md.
package music_recommandation

import com.sun.jna.{Library, Native, Pointer}
import com.sun.jna.ptr.{IntByReference, LongByReference, PointerByReference}

trait MrScore extends Library {
  def mr_create(out: PointerByReference, deviceIds: Array[Int], nDevices: Int, flags: Int): Int
  def mr_destroy(h: Pointer): Unit
  def mr_last_error(h: Pointer): String
  def mr_load(h: Pointer, nTrain: Int, nTest: Int, nSongs: Int, trRowPtr: Array[Long], trCol: Array[Int],
              teRowPtr: Array[Long], teCol: Array[Int], degTrain: Array[Int], degTest: Array[Int], degSongAll: Array[Int]): Int
  def mr_set_test_users(h: Pointer, nTest: Int, teRowPtr: Array[Long], teCol: Array[Int], degTest: Array[Int],
                        pairIndexBase: Long, nPairsTotal: Long): Int
  def mr_score_dense(h: Pointer, model: Int, outUxS: Array[Double]): Int
  def mr_blend_dense(h: Pointer, kind: Int, param: Double, seed: Long, ubm: Array[Double], ibm: Array[Double],
                     out: Array[Double], nPairs: Long, firstIndex: Long, nTotal: Long): Int
  def mr_topk(h: Pointer, model: Int, param: Double, seed: Long, k: Int, outSong: Array[Int], outScore: Array[Double],
              outLen: Array[Int]): Int
  def mr_evaluate_dense(h: Pointer, scoresUxS: Array[Double], nUsers: Int, nSongs: Int, labRowPtr: Array[Long], labCol: Array[Int],
                        nThresholds: Int, outMap: Array[Double]): Int
  // TSV -> int-id data model on the GPU (MusicRecommender.scala:26-91); the result object is read with mr_ingest_get(which = MR_ING_*)
  def mr_score_users(h: Pointer, model: Int, userIdx: Array[Int], n: Int, outNxS: Array[Double]): Int   // DIST getRanks1 (distributed.scala:198-205, 269-276)
  def mr_score_songs(h: Pointer, model: Int, songIds: Array[Int], n: Int, outNxU: Array[Double]): Int   // DIST getRanks2 (distributed.scala:214-221, 285-292)
  def mr_map_at_k(h: Pointer, k: Int, topSong: Array[Int], topLen: Array[Int], nUsers: Int, labRowPtr: Array[Long], labCol: Array[Int],
                  outMap: com.sun.jna.ptr.DoubleByReference, outAp: Array[Double]): Int
  def mr_write_model(path: String, scoresUxS: Array[Double], nUsers: Int, nSongs: Int, userChars: Array[Byte], userOff: Array[Long],
                     songChars: Array[Byte], songOff: Array[Long], append: Int, rowsWritten: LongByReference): Int   // writeModelOnFile MR:489-496
  def mr_prepare_async(h: Pointer): Int   // head-row build on its own stream; the next scoring call completes it
  def mr_set_option(h: Pointer, option: Int, value: Long): Int   // MR_OPT_SONG_WINDOW_LO = 3 / _HI = 4: one song partition of distributed.scala:459-461 per handle
  // join of the partitions' ranked lists (device pointers; the driver-side collect + ranking of distributed.scala:461, 479)
  def mr_topk_merge(h: Pointer, k: Int, nParts: Int, nUsers: Int, partSong: Array[Pointer], partScore: Array[Pointer], partLen: Array[Pointer],
                    outSong: Pointer, outScore: Pointer, outLen: Pointer): Int
  // songs like each query song: the k co-listened songs of highest item-item cosine (MusicRecommender.scala:230-239), [n][k] / [n]
  def mr_similar_songs(h: Pointer, songIds: Array[Int], n: Int, k: Int, outSong: Array[Int], outScore: Array[Double], outLen: Array[Int]): Int
  // listeners like each query test user (indices into the current shard): the k train users of highest user-user cosine (MR:140-149)
  def mr_similar_users(h: Pointer, userIdx: Array[Int], n: Int, k: Int, outUser: Array[Int], outScore: Array[Double], outLen: Array[Int]): Int
  // why song songIds(r) scores what it does for test user userIdx(r) under MR_UBM / MR_IBM: the m largest contributors ([n][m] ids, cosine
  // terms, fixed-point terms), their number, the exact numerator and the library's score per pair (DESIGN.md §4.9)
  def mr_explain(h: Pointer, model: Int, userIdx: Array[Int], songIds: Array[Int], n: Int, m: Int, outId: Array[Int], outTerm: Array[Double],
                 outNum: Array[Long], outLen: Array[Int], outCount: Array[Int], outTotal: Array[Long], outScore: Array[Double]): Int
  // who scores each query song highest under a model (any MR_*, as mr_topk): the k test users of the current shard, score descending then
  // user index ascending, [n][k] / [n] (DESIGN.md §4.10)
  def mr_song_audience(h: Pointer, model: Int, param: Double, seed: Long, songIds: Array[Int], n: Int, k: Int, outUser: Array[Int],
                       outScore: Array[Double], outLen: Array[Int]): Int
  // filtered top-k (DESIGN.md §4.11): an allowed song set (n = -1: every song) and per-user exclusion rows of the current shard (null: none);
  // then per model-set entry each user's ranking without the filtered songs, truncated to k (outputs as mr_topk's, one array per entry)
  def mr_set_topk_filter(h: Pointer, allowSongs: Array[Int], nAllow: Int, exRowptr: Array[Long], exCol: Array[Int]): Int
  def mr_topk_filtered(h: Pointer, nModels: Int, models: Array[Int], params: Array[Double], seeds: Array[Long], k: Int,
                       outSong: Array[Pointer], outScore: Array[Pointer], outLen: Array[Pointer]): Int
  def mr_topk_filtered_device(h: Pointer, nModels: Int, models: Array[Int], params: Array[Double], seeds: Array[Long], k: Int): Int
  def mr_ingest_tsv(device: Int, train: Array[Byte], trainLen: Long, test: Array[Byte], testLen: Long, labels: Array[Byte],
                    labelsLen: Long, out: PointerByReference): Int
  def mr_ingest_error(g: Pointer): String
  def mr_ingest_dims(g: Pointer, nTrain: IntByReference, nTest: IntByReference, nSongs: IntByReference, nLabelOnly: IntByReference): Int
  def mr_ingest_get(g: Pointer, which: Int, ptr: PointerByReference, nElems: LongByReference): Int
  def mr_ingest_free(g: Pointer): Unit
}

object NativeScorer {
  val UBM = 0; val IBM = 1; val LC = 2; val AGG = 3; val STOCH = 4
  lazy val lib: MrScore = Native.load("mrscore", classOf[MrScore])

  /** CSR of a user -> songs map over sorted user and song arrays; column ids ascending and unique within a row. */
  def csr(users: Array[String], songIndex: Map[String, Int], m: Map[String, Array[String]]): (Array[Long], Array[Int], Array[Int]) = {
    val rows = users.map(u => m(u).map(songIndex).distinct.sorted)
    val ptr = rows.scanLeft(0L)(_ + _.length)
    (ptr, rows.flatten, users.map(u => m(u).length))          // third: `.length` incl. duplicates (MusicRecommender.scala:147)
  }
}

/** Owns one handle = one GPU.  `check` maps the error codes back to the reference's exits. */
class NativeScorer(trainUsers: Array[String], testUsers: Array[String], songs: Array[String],
                   trainMap: Map[String, Array[String]], testMap: Map[String, Array[String]],
                   songsToUsers: Map[String, Array[String]], device: Int = 0) {
  import NativeScorer._
  private val sortedTrain = trainUsers.sorted
  val sortedTest: Array[String] = testUsers.sorted
  val sortedSongs: Array[String] = songs.sorted
  private val songIndex = sortedSongs.zipWithIndex.toMap
  private val ref = new PointerByReference()
  check(lib.mr_create(ref, Array(device), 1, 0))
  private val h = ref.getValue
  private val (trPtr, trCol, degTr) = csr(sortedTrain, songIndex, trainMap)
  private val (tePtr, teCol, degTe) = csr(sortedTest, songIndex, testMap)
  check(lib.mr_load(h, sortedTrain.length, sortedTest.length, sortedSongs.length, trPtr, trCol, tePtr, teCol, degTr, degTe,
                    sortedSongs.map(s => songsToUsers(s).length)))        // train + test-visible listeners (MusicRecommender.scala:237)

  private def check(rc: Int): Unit = rc match {
    case 0 =>
    case 1 => System.err.println(lib.mr_last_error(h) + "\n"); System.exit(-1)   // MusicRecommender.scala:366-369
    case 2 => System.exit(2)                                                     // MusicRecommender.scala:326
    case _ => throw new RuntimeException(s"libmrscore error $rc: ${lib.mr_last_error(h)}")
  }

  /** getUserBasedModel / getItemBasedModel: already in the order of main.scala:57-59. */
  def model(kind: Int): Array[(String, (String, Double))] = {
    val (u, s) = (sortedTest.length, sortedSongs.length)
    val buf = new Array[Double](u * s)
    check(lib.mr_score_dense(h, kind, buf))
    for { i <- (0 until u).toArray; j <- 0 until s; x = buf(i * s + j) if !x.isNaN } yield sortedTest(i) -> (sortedSongs(j), x)
  }

  def blend(kind: Int, ubm: Array[(String, (String, Double))], ibm: Array[(String, (String, Double))], param: Double,
            seed: Long = 0L): Array[(String, (String, Double))] = {
    val n = math.min(ubm.length, ibm.length)
    val out = new Array[Double](n)
    check(lib.mr_blend_dense(h, kind, param, seed, ubm.map(_._2._2), ibm.map(_._2._2), out, n, 0L, ubm.length))
    for (i <- (0 until n).toArray) yield {
      if (ubm(i)._1 != ibm(i)._1 || ubm(i)._2._1 != ibm(i)._2._1) System.exit(2)
      ubm(i)._1 -> (ubm(i)._2._1, out(i))
    }
  }

  def topK(kind: Int, k: Int = 500, param: Double = 0.5, seed: Long = 0L): Array[(String, Array[(String, Double)])] = {
    val u = sortedTest.length
    val (song, score, len) = (new Array[Int](u * k), new Array[Double](u * k), new Array[Int](u))
    check(lib.mr_topk(h, kind, param, seed, k, song, score, len))
    for (i <- (0 until u).toArray) yield sortedTest(i) -> (0 until len(i)).map(r => sortedSongs(song(i * k + r)) -> score(i * k + r)).toArray
  }

  def close(): Unit = lib.mr_destroy(h)
}
