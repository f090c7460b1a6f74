// callsite_compile.cpp -- the CALL EXPRESSIONS of the reference, pasted from
//   src/VectorIndex/Common/VIWithDataPart.cpp:416-430 (createVectorIndex), :461-478 (serialize), :688-700 (load),
//   :851-853 (computeTopDistanceSubset), :921-936 (search), VIWithDataPart.h:332-337 (build),
//   src/VectorIndex/Common/BruteForceSearch.h:77-105, src/VectorIndex/Common/VectorIndexIO.h (stream classes),
//   src/VectorIndex/Common/VIPartReader.h (reader), src/Storages/MergeTree/TantivyIndexStore.cpp:654, :713, :742, :824,
//   :908-917, :939-948, :962, :974, :986, :998
// and compiled with -Wall -Wextra -Werror against shim/b200_search_shim.hpp, with stand-ins only for ClickHouse's own types
// (disk streams, the part reader's column access).  Then it RUNS on the GPU (tests/test_gpu_shim.py): builds an index
// through the reader, searches it with a filter bitmap, serialises it through the stream classes, loads it back, and
// drives the BM25 entry points.  Prints "CALLSITES OK".
#include <b200_search_shim.hpp>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <filesystem>
#include <variant>

using String = std::string;
using UInt64 = uint64_t;

// ---- VectorIndex/Common/VICommon.h:120-170: the aliases src/VectorIndex builds on --------------------------------
namespace VectorIndex {
using VectorIndexIStream = Search::AbstractIStream;
using VectorIndexOStream = Search::AbstractOStream;
using VIBitmap = Search::DenseBitmap;
using VIBitmapPtr = std::shared_ptr<Search::DenseBitmap>;
using SearchResult = Search::SearchResult;
using SearchResultPtr = std::shared_ptr<SearchResult>;
using VIParameter = Search::Parameters;
using VIType = Search::IndexType;
using VIMetric = Search::Metric;
using VIDataType = Search::DataType;
using FloatVI = Search::VectorIndex<VectorIndexIStream, VectorIndexOStream, VIBitmap, VIDataType::FloatVector>;
using FloatVIPtr = std::shared_ptr<FloatVI>;
using BinaryVI = Search::VectorIndex<VectorIndexIStream, VectorIndexOStream, VIBitmap, VIDataType::BinaryVector>;
using BinaryVIPtr = std::shared_ptr<BinaryVI>;
using VIVariantPtr = std::variant<FloatVIPtr, BinaryVIPtr>;
template <Search::DataType> struct SearchIndexDataTypeMap;
template <> struct SearchIndexDataTypeMap<Search::DataType::FloatVector> { using VectorDatasetType = float; using IndexDatasetType = float; };
template <> struct SearchIndexDataTypeMap<Search::DataType::BinaryVector> { using VectorDatasetType = uint8_t; using IndexDatasetType = bool; };
template <Search::DataType T> using VISourcePartReader = Search::IndexSourceDataReader<typename SearchIndexDataTypeMap<T>::IndexDatasetType>;

// ---- VectorIndexIO.h:33-164 with the ClickHouse disk replaced by an in-memory "disk" -----------------------------
using Disk = std::map<std::string, std::string>;
class VectorIndexReader : public Search::AbstractIStream {
public:
    explicit VectorIndexReader(Disk * disk, const String & file) { auto it = disk->find(file); if (it != disk->end()) in = &it->second; }
    Search::AbstractIStream & read(char * s, std::streamsize count) override {
        last_read_bytes = 0;
        if (in) { last_read_bytes = std::min<size_t>(size_t(count), in->size() - pos); memcpy(s, in->data() + pos, last_read_bytes); pos += last_read_bytes; }
        return *this;
    }
    bool is_open() const override { return in != nullptr; }
    bool fail() const override { return in ? !(operator bool()) : true; }
    bool eof() const override { return in ? pos >= in->size() : true; }
    std::streamsize gcount() const override { return std::streamsize(last_read_bytes); }
    explicit operator bool() const override { return in != nullptr; }
    Search::AbstractIStream & seekg(std::streampos offset, std::ios_base::seekdir) override { pos = size_t(offset); return *this; }
private:
    const std::string * in = nullptr;
    size_t pos = 0, last_read_bytes = 0;
};
class VectorIndexWriter : public Search::AbstractOStream {
public:
    explicit VectorIndexWriter(Disk * disk, const String & file) : out(&(*disk)[file]) {}
    Search::AbstractOStream & write(const char * s, std::streamsize count) override { out->append(s, size_t(count)); return *this; }
    bool good() override { return true; }
    void close() override {}
    Search::AbstractOStream & seekp(std::streampos, std::ios_base::seekdir) override { return *this; }
private:
    std::string * out;
};

// ---- VIPartReader.h:38-306 with the MergeTree column replaced by a float array ------------------------------------
template <Search::DataType T>
class VIPartReader : public VISourcePartReader<T> {
public:
    using DataChunk = typename VISourcePartReader<T>::DataChunk;
    VIPartReader(const float * rows_, size_t n_, size_t dimension_) : rows(rows_), total(n_), dimension(dimension_) {}
    size_t numDataRead() const override { return num_rows_read; }
    size_t dataDimension() const override { return dimension; }
    bool eof() override { return num_rows_read == total; }
    void seekg(std::streamsize, std::ios::seekdir) override { throw std::runtime_error("seekg() is not implemented in VIPartReader"); }
    std::shared_ptr<DataChunk> sampleData(size_t n) override {
        std::vector<std::shared_ptr<DataChunk>> chunks;
        size_t num_rows = 0;
        while (num_rows < n) {
            auto chunk = readDataImpl(n - num_rows);
            if (chunk == nullptr) break;
            num_rows += chunk->numData();
            chunks.push_back(chunk);
        }
        reset();
        if (chunks.empty()) return nullptr;
        size_t tot = 0;
        for (auto & c : chunks) tot += c->numData();
        float * data = new float[dimension * tot]();
        Search::idx_t * ids = new Search::idx_t[tot]();
        size_t at = 0;
        for (auto & c : chunks) { memcpy(data + at * dimension, c->getData(), c->numData() * dimension * sizeof(float)); memcpy(ids + at, c->getDataID(), c->numData() * sizeof(Search::idx_t)); at += c->numData(); }
        auto merged_chunk = std::make_shared<DataChunk>(data, tot, dimension, [=]() { delete[] data; });
        merged_chunk->setDataID(ids, [=]() { delete[] ids; });
        return merged_chunk;
    }
protected:
    std::shared_ptr<DataChunk> readDataImpl(size_t n) override {
        if (n == 0 || num_rows_read == total) return nullptr;
        const size_t total_rows = std::min(n, total - num_rows_read), current_round_start_row = num_rows_read;
        float * vector_raw_data = new float[dimension * total_rows];
        Search::idx_t * ids = new Search::idx_t[total_rows]();
        memcpy(vector_raw_data, rows + current_round_start_row * dimension, total_rows * dimension * sizeof(float));
        for (size_t row = 0; row < total_rows; row++) ids[row] = Search::idx_t(current_round_start_row + row);
        num_rows_read += total_rows;
        std::shared_ptr<DataChunk> chunk = std::make_shared<DataChunk>(vector_raw_data, total_rows, dimension, [=]() { delete[] vector_raw_data; });
        chunk->setDataID(ids, [=]() { delete[] ids; });
        return chunk;
    }
    void reset() { num_rows_read = 0; }
private:
    const float * rows;
    size_t total, dimension, num_rows_read = 0;
};
}  // namespace VectorIndex

using namespace VectorIndex;

#define REQUIRE(cond) do { if (!(cond)) { std::printf("FAILED line %d: %s\n", __LINE__, #cond); return 1; } } while (0)

// BruteForceSearch.h:63-111, verbatim body
template <Search::DataType T>
void tryBruteForceSearch(const typename SearchIndexDataTypeMap<T>::VectorDatasetType * x, const typename SearchIndexDataTypeMap<T>::VectorDatasetType * y,
                         size_t d, size_t k, size_t nx, size_t ny, int64_t * result_id, float * distance, const VIMetric & metric_type) {
    if constexpr (T == Search::DataType::FloatVector) {
        if (metric_type == VIMetric::IP) {
            faiss::float_minheap_array_t res = {size_t(nx), size_t(k), result_id, distance};
            faiss::knn_inner_product(x, y, d, nx, ny, &res, nullptr);
        } else if (metric_type == VIMetric::L2) {
            faiss::float_maxheap_array_t res = {size_t(nx), size_t(k), result_id, distance};
            faiss::knn_L2sqr(x, y, d, nx, ny, &res, nullptr);
        } else {
            throw std::runtime_error("Metric not implemented in brute force search for Float32 Vector");
        }
    } else if constexpr (T == Search::DataType::BinaryVector) {
        if (metric_type == VIMetric::Hamming) {
            faiss::hammings_knn_mc(x, y, nx, ny, k, d / 8, reinterpret_cast<int32_t *>(distance), result_id, nullptr);
        } else if (metric_type == VIMetric::Jaccard) {
            jaccard_knn(x, y, nx, ny, k, d / 8, distance, result_id, nullptr);
        } else {
            throw std::runtime_error("Metric not implemented in brute force search for Binary Vector");
        }
    }
}

int main() {
    try {
        // ---------------- brute force (golden 00001: rows [n,n,n], query [0.1]*3)
        const size_t dimension = 3, total_vec = 3000;
        std::vector<float> y(dimension * total_vec), q = {0.1f, 0.1f, 0.1f};
        for (size_t n = 0; n < total_vec; ++n) y[3 * n] = y[3 * n + 1] = y[3 * n + 2] = float(n);
        std::vector<int64_t> ids(10); std::vector<float> dis(10);
        tryBruteForceSearch<Search::DataType::FloatVector>(q.data(), y.data(), dimension, 10, 1, total_vec, ids.data(), dis.data(), VIMetric::L2);
        for (int i = 0; i < 10; ++i) REQUIRE(ids[size_t(i)] == i);
        REQUIRE(std::fabs(dis[0] - 0.030000001f) < 1e-7f && std::fabs(dis[9] - 237.62997f) < 1e-3f);
        std::vector<uint8_t> by = {0x0f, 0xff, 0x00, 0xf0}, bq = {0x0f};
        std::vector<int64_t> bid(2); std::vector<float> bdis(2);
        tryBruteForceSearch<Search::DataType::BinaryVector>(bq.data(), by.data(), 8, 2, 1, 4, bid.data(), bdis.data(), VIMetric::Hamming);
        REQUIRE(bid[0] == 0 && reinterpret_cast<int32_t *>(bdis.data())[0] == 0 && reinterpret_cast<int32_t *>(bdis.data())[1] == 4);

        // ---------------- createVectorIndex (VIWithDataPart.cpp:416-430)
        const String index_name = "v1", metric_str = "L2";
        const Search::DataType vector_search_type = Search::DataType::FloatVector;
        VIParameter index_des;
        index_des.setParam("ncentroids", 16);
        index_des.setParam("metric_type", metric_str);
        std::erase_if(index_des, [](const auto & item) { auto const & [key, value] = item; (void)value; return key == "metric_type"; });   // :402-408
        auto index_type = Search::getVectorIndexType("IVFFLAT", vector_search_type);
        auto metric = Search::getMetricType(metric_str, vector_search_type);
        const size_t max_threads = 8;
        String vector_index_cache_prefix = "store/all_1_1_0/v1/";
        VIVariantPtr index_variant;
        if (vector_search_type == Search::DataType::FloatVector)
            index_variant = Search::createVectorIndex<VectorIndexIStream, VectorIndexOStream, VIBitmap, VIDataType::FloatVector>(
                index_name, index_type, metric, dimension, total_vec, index_des, max_threads, vector_index_cache_prefix,
                []() { return false; });
        else if (vector_search_type == Search::DataType::BinaryVector)
            index_variant = Search::createVectorIndex<VectorIndexIStream, VectorIndexOStream, VIBitmap, VIDataType::BinaryVector>(
                index_name, index_type, metric, dimension, total_vec, index_des, max_threads, vector_index_cache_prefix,
                []() { return false; });

        // ---------------- build (VIWithDataPart.h:325-339)
        {
            VIPartReader<Search::DataType::FloatVector> reader(y.data(), total_vec, dimension);
            VISourcePartReader<Search::DataType::FloatVector> * part_reader = &reader;
            FloatVIPtr index_ptr = std::get<FloatVIPtr>(index_variant);
            const size_t max_build_index_train_block_size = 100u << 20, max_build_index_add_block_size = 12000;   // small add block: several chunks
            const int num_threads = 4;
            auto cancel_build_callback = []() { return false; };
            index_ptr->setTrainDataChunkSize(max_build_index_train_block_size);
            index_ptr->setAddDataChunkSize(max_build_index_add_block_size);
            REQUIRE(index_ptr->getResourceUsage().build_memory_usage_bytes > 0);
            index_ptr->build(part_reader, num_threads, cancel_build_callback);
            REQUIRE(index_ptr->numData() == total_vec && index_ptr->ready());
        }

        // ---------------- search with a filter (VIWithDataPart.cpp:905-936) + transferToNewRowIds' accessors (:61-65)
        SearchResultPtr ret;
        {
            VIBitmapPtr filter = std::make_shared<VIBitmap>(total_vec, true), delete_bitmap = std::make_shared<VIBitmap>(total_vec, true);
            delete_bitmap->unset(0);
            VIBitmapPtr merged_filter = Search::intersectDenseBitmaps(filter, delete_bitmap);
            VIParameter parameters;
            parameters.setParam("nprobe", 16);
            const int32_t k = 5;
            const bool first_stage_only = false;
            auto search_queries = std::make_shared<Search::DataSet<SearchIndexDataTypeMap<Search::DataType::FloatVector>::IndexDatasetType>>(q.data(), 1, int64_t(dimension));
            const FloatVIPtr & float_index = std::get<FloatVIPtr>(index_variant);
            ret = float_index->search(search_queries, k, parameters, first_stage_only, merged_filter.get());
            REQUIRE(ret->numQueries() == 1 && ret->getNumCandidates() >= k);
            for (size_t kk = 0; kk < ret->numQueries(); kk++)
                for (auto & label : ret->getResultIndices(kk)) REQUIRE(label >= 1 && label <= 5);
            auto per_id = ret->getResultIndices();
            auto per_distance = ret->getResultDistances();
            REQUIRE(per_id[0] == 1 && std::fabs(per_distance[0] - 2.4299998f) < 1e-5f);
            // computeTopDistanceSubset (:851-853)
            if (float_index->supportTwoStageSearch() || true) {
                auto first_stage_result = ret;
                const int32_t top_k = 3;
                auto re = float_index->computeTopDistanceSubset(search_queries, first_stage_result, top_k);
                REQUIRE(re->getResultIndices()[0] == 1 && re->getResultIndices()[2] == 3);
            }
        }

        // ---------------- serialize (VIWithDataPart.cpp:451-500) and load (:688-704) through the stream classes
        Disk disk_store;
        Disk * disk = &disk_store;
        {
            auto index_serialize_folder = String("tmp/") + std::string(index_name + "-");
            auto file_writer = Search::IndexDataFileWriter<VectorIndexOStream>(
                index_serialize_folder, [&](const std::string & name, std::ios::openmode /*mode*/) { return std::make_shared<VectorIndexWriter>(disk, name); });
            String version, memory_usage, disk_usage;
            std::visit(
                [&](auto && index_ptr) {
                    index_ptr->serialize(&file_writer);
                    index_ptr->saveDataID(&file_writer);
                    version = index_ptr->getVersion().toString();
                    auto usage = index_ptr->getResourceUsage();
                    memory_usage = std::to_string(usage.memory_usage_bytes);
                    disk_usage = std::to_string(usage.disk_usage_bytes);
                },
                index_variant);
            REQUIRE(!version.empty() && std::stoull(memory_usage) > 0 && std::stoull(disk_usage) > 0);
            REQUIRE(disk->count("tmp/v1-data_bin") == 1);
        }
        {
            VIParameter index_params;
            index_params.setParam("load_index_version", String("1"));
            VIVariantPtr loaded = Search::createVectorIndex<VectorIndexIStream, VectorIndexOStream, VIBitmap, VIDataType::FloatVector>(
                index_name, index_type, metric, dimension, total_vec, index_params, max_threads, vector_index_cache_prefix, []() { return false; });
            auto file_reader = Search::IndexDataFileReader<VectorIndexIStream>(
                String("tmp/v1-"), [disk](const std::string & name, std::ios::openmode /*mode*/) { return std::make_shared<VectorIndexReader>(disk, name); });
            auto check_index_expired = []() { return false; };
            UInt64 index_total_vec = 0;
            std::visit(
                [&](auto && index_ptr) {
                    index_ptr->load(&file_reader, check_index_expired);
                    index_ptr->loadDataID(&file_reader);
                    index_total_vec = index_ptr->numData();
                },
                loaded);
            REQUIRE(index_total_vec == total_vec);
            VIParameter parameters;
            auto search_queries = std::make_shared<Search::DataSet<float>>(q.data(), 1, int64_t(dimension));
            auto again = std::get<FloatVIPtr>(loaded)->search(search_queries, 5, parameters, false, nullptr);
            REQUIRE(again->getResultIndices()[0] == 0 && again->getResultIndices()[1] == 1);
        }
        REQUIRE(String(Search::enumToString(index_type)) == "IVFFLAT");
        Search::IndexType parsed;
        REQUIRE(Search::findEnumByName("mstg", parsed) && parsed == Search::IndexType::MSTG);
        REQUIRE(Search::getDefaultIndexType(Search::DataType::FloatVector) == "SCANN" && String(Search::MYSCALE_VALID_INDEX_PARAMETER).find("ncentroids") != String::npos);

        // ---------------- TantivyIndexStore.cpp call sites
        {
            // the part's FTS cache directory (index_files_manager): a fresh one per run, so concurrent runs never share it
            String fts_dir_template = (std::filesystem::temp_directory_path() / "b200_callsite_fts_XXXXXX").string();
            REQUIRE(mkdtemp(fts_dir_template.data()) != nullptr);
            const String index_files_cache_path = fts_dir_template;
            std::vector<String> indexed_columns = {"doc", "title"};
            const String index_json_parameter = "{}";
            TANTIVY::FFIBoolResult create_status = TANTIVY::ffi_create_index_with_parameter(index_files_cache_path, indexed_columns, index_json_parameter);   // :713
            REQUIRE(!create_status.error.is_error && create_status.result);
            const char * texts[3] = {"Ancient empires rise and fall", "Artistic expressions reflect heritages", "Ancient philosophies provide wisdom"};
            for (uint64_t row_id = 0; row_id < 3; ++row_id) {
                std::vector<String> column_names = {"doc", "title"}, docs = {texts[row_id], row_id == 1 ? "ancient title" : "other"};
                TANTIVY::FFIBoolResult index_status = TANTIVY::ffi_index_multi_column_docs(index_files_cache_path, row_id, column_names, docs);   // :742
                REQUIRE(!index_status.error.is_error && index_status.result);
            }
            TANTIVY::FFIBoolResult commit_result = TANTIVY::ffi_index_writer_commit(index_files_cache_path);   // :824
            REQUIRE(!commit_result.error.is_error);
            TANTIVY::FFIBoolResult load_status = TANTIVY::ffi_load_index_reader(index_files_cache_path);        // :654
            REQUIRE(!load_status.error.is_error && load_status.result);
            String sentence = "Ancient";
            bool enable_nlq = true, operator_or = true;
            TANTIVY::Statistics statistics;
            size_t topk = 5;
            std::vector<String> column_names = {"doc"};
            std::vector<uint8_t> u8_alived_bitmap;
            TANTIVY::FFIVecRowIdWithScoreResult result = TANTIVY::ffi_bm25_search(                                // :908-917
                index_files_cache_path, sentence, column_names, static_cast<uint32_t>(topk), u8_alived_bitmap, false, enable_nlq, operator_or, statistics);
            REQUIRE(!result.error.is_error && result.result.size() == 2 && result.result[0].row_id == 2 && result.result[1].row_id == 0);   // the shorter document scores higher
            u8_alived_bitmap = {0x06};   // row 0 deleted
            result = TANTIVY::ffi_bm25_search(index_files_cache_path, sentence, column_names, static_cast<uint32_t>(topk), u8_alived_bitmap, true,   // :939-948
                                              enable_nlq, operator_or, statistics);
            REQUIRE(!result.error.is_error && result.result.size() == 1 && result.result[0].row_id == 2);
            column_names = {"doc", "title"};
            result = TANTIVY::ffi_bm25_search(index_files_cache_path, sentence, column_names, static_cast<uint32_t>(topk), {}, false, enable_nlq, operator_or, statistics);
            REQUIRE(result.result.size() == 3);
            TANTIVY::FFIVecDocWithFreqResult df = TANTIVY::ffi_get_doc_freq(index_files_cache_path, sentence);   // :962
            REQUIRE(!df.error.is_error && df.result.size() == 2 && df.result[0].doc_freq == 2 && df.result[1].doc_freq == 1);
            TANTIVY::FFIU64Result nd = TANTIVY::ffi_get_total_num_docs(index_files_cache_path);                   // :974
            REQUIRE(nd.result == 3);
            TANTIVY::FFIFieldTokenNumsResult tk = TANTIVY::ffi_get_total_num_tokens(index_files_cache_path);      // :986
            REQUIRE(tk.result.size() == 2 && tk.result[0].field_total_tokens == 13);
            REQUIRE(TANTIVY::ffi_get_indexed_doc_counts(index_files_cache_path).result == 3);                     // :998
            TANTIVY::FFIBoolResult free_status = TANTIVY::ffi_free_index_reader(index_files_cache_path);          // :769
            REQUIRE(free_status.result);
            free_status = TANTIVY::ffi_free_index_writer(index_files_cache_path);                                 // :792
            REQUIRE(TANTIVY::ffi_get_total_num_docs(index_files_cache_path).error.is_error);                      // store gone: an FFI error, never a crash
            // a later query re-opens the part's index from its cache directory (getTantivyIndexReader, :646-686)
            load_status = TANTIVY::ffi_load_index_reader(index_files_cache_path);
            REQUIRE(!load_status.error.is_error && load_status.result);
            result = TANTIVY::ffi_bm25_search(index_files_cache_path, sentence, column_names, static_cast<uint32_t>(topk), {}, false, enable_nlq, operator_or, statistics);
            REQUIRE(!result.error.is_error && result.result.size() == 3);
            TANTIVY::ffi_free_index_reader(index_files_cache_path);
            REQUIRE(TANTIVY::ffi_load_index_reader(index_files_cache_path + "/no_such_dir").error.is_error);
            std::filesystem::remove_all(index_files_cache_path);
        }
        std::printf("CALLSITES OK\n");
        return 0;
    } catch (const SearchIndexException & e) {
        std::printf("SearchIndexException %d: %s\n", e.getCode(), e.what());
        return 2;
    } catch (const std::exception & e) {
        std::printf("exception: %s\n", e.what());
        return 3;
    }
}
